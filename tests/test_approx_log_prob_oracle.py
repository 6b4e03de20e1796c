"""The reference log density of the LogitSkewNormalPTT approximation (DESIGN.md K5, tests/lsn_density_ref.py) against
the fit's forward path and against finite differences of itself (CPU only)."""
import numpy as np
import pytest

import lsn_density_ref as ref
from conftest import relerr


def _params(rng, nm1):
    mu = rng.uniform(-2, 2, nm1).astype(np.float32)
    omega = np.log(rng.uniform(0.1, 1.0, nm1)).astype(np.float32)
    alpha = rng.uniform(-0.5, 0.5, nm1).astype(np.float32)
    return mu, omega, alpha


def _forward(l, r, f, n, y):
    """x = T(y) and sum_j log u_j (hsb_ladj) in Float64: u_root = 1, u_left = y u, u_right = (1 - y) u"""
    N = 2 * n - 1
    u = np.zeros(N)
    u[0] = 1.0
    x = np.zeros(n)
    hsb_ladj, k = 0.0, 0
    for j in range(N):
        if f[j] >= 0:
            x[f[j]] = u[j]
        else:
            u[l[j]], u[r[j]] = y[k] * u[j], (1.0 - y[k]) * u[j]
            hsb_ladj += np.log(u[j])
            k += 1
    return x, hsb_ladj


@pytest.mark.parametrize("tree", ["fixture", "balanced1000"])
def test_log_density_is_the_change_of_variables_of_the_forward_path(oracle, fx, tree):
    from polee_b200 import synth
    pi, js = (fx.parent_idxs, fx.js) if tree == "fixture" else synth.balanced_tree(1000)
    n = (len(js) + 1) // 2
    l, r, f = oracle.make_inverse_ptt_params(pi, js)
    rng = np.random.default_rng(7)
    mu, omega, alpha = _params(rng, n - 1)
    sigma = ref.sigma_of(omega)
    for _ in range(3):
        z0 = rng.normal(size=n - 1)
        c = alpha.astype(np.float64) + np.arcsinh(z0)
        zs = np.sinh(c)
        y = 1.0 / (1.0 + np.exp(-(mu.astype(np.float64) + sigma * zs)))
        x, hsb_ladj = _forward(l, r, f, n, y)
        skew_ladj = np.sum(np.log(np.cosh(c)) - 0.5 * np.log1p(z0 * z0))
        ln_ladj = np.sum(np.log(sigma * y * (1.0 - y)))
        expected = np.sum(-0.5 * z0 * z0 - 0.5 * np.log(2 * np.pi)) - (skew_ladj + ln_ladj + hsb_ladj)
        lp = ref.approx_log_prob(oracle, x.astype(np.float32), mu, omega, alpha, l, r, f, want_grad=False)
        assert relerr(lp[0], expected) <= 1e-6, (lp[0], expected)


def test_gradient_matches_central_differences(oracle):
    from polee_b200 import synth
    n = 64
    l, r, f = oracle.make_inverse_ptt_params(*synth.random_tree(n, seed=3))
    rng = np.random.default_rng(5)
    mu, omega, alpha = _params(rng, n - 1)
    x = rng.dirichlet(np.ones(n) * 2.0).astype(np.float32)
    lp, g = ref.approx_log_prob(oracle, x, mu, omega, alpha, l, r, f)
    assert np.isfinite(lp).all() and np.isfinite(g).all()
    fd = np.zeros(n)
    for i in range(n):
        xp, xm = x.copy(), x.copy()
        h = np.float32(1e-3) * x[i]
        xp[i] += h
        xm[i] -= h
        step = float(xp[i]) - float(xm[i])                 # the step the Float32 values actually took
        fd[i] = (ref.approx_log_prob(oracle, xp, mu, omega, alpha, l, r, f, want_grad=False)[0] -
                 ref.approx_log_prob(oracle, xm, mu, omega, alpha, l, r, f, want_grad=False)[0]) / step
    assert relerr(g[0], fd) <= 1e-4, (g[0], fd)


def test_boundary_row_is_minus_inf_and_single_leaf_is_zero(oracle):
    from polee_b200 import synth
    n = 16
    l, r, f = oracle.make_inverse_ptt_params(*synth.balanced_tree(n))
    rng = np.random.default_rng(1)
    mu, omega, alpha = _params(rng, n - 1)
    x = rng.dirichlet(np.ones(n), 2).astype(np.float32)
    x[1, 3] = 0.0                                           # its sibling leaf is non-zero: y = 0 or 1 at the parent
    lp = ref.approx_log_prob(oracle, x, mu, omega, alpha, l, r, f, want_grad=False)
    assert np.isfinite(lp[0]) and lp[1] == -np.inf
    assert lp[0] == ref.approx_log_prob(oracle, x[:1], mu, omega, alpha, l, r, f, want_grad=False)[0]
    e = np.zeros(0, np.float32)
    lp1, g1 = ref.approx_log_prob(oracle, np.ones((1, 1), np.float32), e, e, e, [-1], [-1], [0])
    assert lp1[0] == 0.0 and g1[0, 0] == 0.0
