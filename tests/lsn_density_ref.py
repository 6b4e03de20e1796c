"""Reference for the log density of the LogitSkewNormalPTT approximation (DESIGN.md K5), for the tests.

A serial restatement of the definition: y from the oracle's InvHSB (the same IEEE adds and divides as k4_inv_hsb), the
subtree sums u_j by the same bottom-up walk in Python floats, sigma from the C library's expf, the node terms in numpy
Float64, and the gradient through the oracle's InvHSBGrad with ladj_grad = 1."""
import ctypes as C

import numpy as np

_libm = C.CDLL("libm.so.6")
_libm.expf.restype = C.c_float
_libm.expf.argtypes = [C.c_float]


def sigma_of(omega):
    """Float64(expf(omega)) with the C library's expf, as the fit forms sigma"""
    return np.array([_libm.expf(float(o)) for o in np.ravel(omega)], np.float64).reshape(np.shape(omega))


def _log_u(x, L, R, F):
    """log u_j of one row, indexed by k (the j-th internal node in array order)"""
    N = len(F)
    n = (N + 1) // 2
    u = [0.0] * N
    out = np.zeros(max(n - 1, 0))
    k = n - 2
    for j in range(N - 1, -1, -1):
        if F[j] >= 0:
            u[j] = float(x[F[j]])
        else:
            u[j] = u[L[j]] + u[R[j]]
            out[k] = np.log(u[j])
            k -= 1
    return out


def approx_log_prob(oracle, x, mu, omega, alpha, left, right, leaf, want_grad=True):
    """log q(x) -> lp [B], or (lp, x_grad [B][n] Float32); mu / omega / alpha [param_batch][n-1], param_batch 1 or B"""
    x = np.atleast_2d(np.ascontiguousarray(x, np.float32))
    B, n = x.shape
    N = 2 * n - 1
    mu, omega, alpha = (np.asarray(a, np.float32).reshape(-1, n - 1) if n > 1 else np.zeros((1, 0), np.float32)
                        for a in (mu, omega, alpha))
    L, R, F = (np.ascontiguousarray(np.broadcast_to(np.asarray(a, np.int32).reshape(-1, N), (B, N)))
               for a in (left, right, leaf))
    y, _ = oracle.inv_hsb(x, L, R, F)
    logu = np.stack([_log_u(x[b], L[b].tolist(), R[b].tolist(), F[b].tolist()) for b in range(B)])
    sigma = sigma_of(omega)
    if mu.shape[0] == 1:
        mu, sigma, alpha = (np.broadcast_to(a, (B, n - 1)) for a in (mu, sigma, alpha))
    with np.errstate(all="ignore"):
        ly, l1my = np.log(y), np.log1p(-y)
        s = (ly - l1my - mu) / sigma
        w = np.arcsinh(s) - alpha
        z0, r, aw = np.sinh(w), np.hypot(1.0, s), np.abs(w)
        log_cosh_w = aw + np.log1p(np.exp(-2.0 * aw)) - np.log(2.0)
        term = (-0.5 * z0 * z0 - 0.5 * np.log(2 * np.pi) + log_cosh_w - 0.5 * np.log1p(s * s) - np.log(sigma) - ly - l1my
                - logu)
        term = np.where((y > 0.0) & (y < 1.0), term, -np.inf)
        g_s = (np.tanh(w) - z0 * np.cosh(w)) / r - s / (r * r)
        y_grad = g_s / (sigma * y * (1.0 - y)) + 1.0 / (1.0 - y) - 1.0 / y
    lp = np.array([sum(row.tolist()) for row in term]) if n > 1 else np.zeros(B)   # serial sums
    if not want_grad:
        return lp
    x_grad = oracle.inv_hsb_grad(y_grad, np.ones(B, np.float32), y, np.zeros(B, np.float32), L, R, F)
    return lp, x_grad
