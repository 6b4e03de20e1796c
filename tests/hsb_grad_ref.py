"""Reference for HSBGrad, the gradient of HSB (include/polee_b200.h, DESIGN.md K4), for the tests.

A serial restatement of the definition in Float64: nodes one at a time in array order (parents before children, as
the tree arrays require), rows vectorised with numpy, every product and sum in the association the definition gives
(numpy does not contract to FMA).  y uses the C library's exp, as the reference op does; the device's exp differs from
it in rare last bits, which is the only source of difference from the device."""
import math

import numpy as np


def _trees(left, right, leaf, B):
    N = np.shape(left)[-1]
    L, R, F = (np.broadcast_to(np.asarray(a, np.int64).reshape(-1, N), (B, N)) for a in (left, right, leaf))
    return L, R, F, np.cumsum(F < 0, axis=1) - 1


def sigmoid(y_logit):
    """y = 1 / (1 + exp(-y_logit)) in Float64 with the C library's exp"""
    yl = np.asarray(y_logit, np.float64)
    e = np.array([math.exp(-v) for v in yl.ravel()], np.float64).reshape(yl.shape)
    return 1.0 / (1.0 + e)


def forward(y_logit, left, right, leaf):
    """(x [B][n], u [B][2n-1], y [B][n-1]) in Float64: u_root = 1, u_left = y u_j, u_right = (1 - y) u_j, x = u at leaves"""
    y = sigmoid(y_logit)
    B, nm1 = y.shape
    L, R, F, K = _trees(left, right, leaf, B)
    N = L.shape[1]
    rows = np.arange(B)
    u = np.zeros((B, N))
    u[:, 0] = 1.0
    x = np.zeros((B, nm1 + 1))
    for j in range(N):
        lf = F[:, j] >= 0
        if lf.any():
            x[rows[lf], F[lf, j]] = u[lf, j]
        r = rows[~lf]
        if r.size:
            yk = y[r, K[r, j]]
            u[r, L[r, j]] = yk * u[r, j]
            u[r, R[r, j]] = (1.0 - yk) * u[r, j]
    return x, u, y


def hsb_grad(x_grad, y_logit, left, right, leaf):
    """y_logit_grad [B][n-1] in Float64 (the device rounds it to Float32): G = x_grad at a leaf,
    G_j = y G_l + (1 - y) G_r, y_logit_grad_k = ((y (1 - y)) u_j) (G_l - G_r)"""
    _, u, y = forward(y_logit, left, right, leaf)
    B, nm1 = y.shape
    L, R, F, K = _trees(left, right, leaf, B)
    N = L.shape[1]
    xg = np.asarray(x_grad, np.float64).reshape(B, nm1 + 1)
    rows = np.arange(B)
    G = np.zeros((B, N))
    out = np.zeros((B, nm1))
    for j in range(N - 1, -1, -1):
        lf = F[:, j] >= 0
        if lf.any():
            G[lf, j] = xg[rows[lf], F[lf, j]]
        r = rows[~lf]
        if r.size:
            k = K[r, j]
            yk = y[r, k]
            gl, gr = G[r, L[r, j]], G[r, R[r, j]]
            G[r, j] = yk * gl + (1.0 - yk) * gr
            out[r, k] = ((yk * (1.0 - yk)) * u[r, j]) * (gl - gr)
    return out
