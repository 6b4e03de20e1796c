"""Device log density of the LogitSkewNormalPTT approximation (polee_approx_log_prob_*, DESIGN.md K5) against the
reference restatement (tests/lsn_density_ref.py), the fit's own forward pass, its host form and torch autograd."""
import ctypes as C

import numpy as np
import pytest

import lsn_density_ref as ref
from conftest import relerr

pytestmark = pytest.mark.gpu


def _compare(lp, g, lp_o, g_o):
    """lp within 1e-10 relative; each finite row's x_grad within 1e-6 of that row's largest |x_grad|"""
    inf, inf_o = np.isneginf(lp), np.isneginf(lp_o)
    assert np.array_equal(inf, inf_o)
    fin = ~inf
    assert relerr(lp[fin], lp_o[fin]) <= 1e-10
    for b in np.nonzero(fin)[0]:
        assert np.abs(g[b] - g_o[b]).max() <= 1e-6 * np.abs(g_o[b]).max(), b


def _lsn_x(rng, B, l, r, f, mu, omega, alpha):
    """x = HSB(y) for y drawn from the approximation (parameters [1 or B][n-1])"""
    import polee_b200 as pb
    z0 = rng.normal(size=(B, mu.shape[-1]))
    zs = np.sinh(alpha.astype(np.float64) + np.arcsinh(z0))
    return pb.hsb((mu + np.exp(omega.astype(np.float64)) * zs).astype(np.float32), l, r, f)


def test_sampler_draws_match_reference(fx, oracle):
    import polee_b200 as pb
    s = pb.ApproxLikelihoodSampler()
    s.set_transform((fx.parent_idxs, fx.js), fx.mu, np.exp(fx.omega), fx.alpha)
    xs = s.rand(16, seed=3)
    lp, g = s.log_prob(xs, want_grad=True)
    assert np.array_equal(s.log_prob(xs), lp)
    mu, omega, alpha = s.params
    lp_o, g_o = ref.approx_log_prob(oracle, xs, mu, omega, alpha, *oracle.make_inverse_ptt_params(fx.parent_idxs, fx.js))
    assert np.isfinite(lp).all()
    _compare(lp, g, lp_o, g_o)


@pytest.mark.parametrize("trees", ["shared", "per_row"])
@pytest.mark.parametrize("param_batch", ["one", "per_row"])
def test_20000_leaves_match_reference(oracle, trees, param_batch):
    import polee_b200 as pb
    from polee_b200 import synth
    n, B = 20000, 6
    if trees == "shared":
        l, r, f = (a[None] for a in pb.make_inverse_ptt_params(*synth.balanced_tree(n)))
    else:
        l, r, f = (np.stack(a) for a in zip(*[pb.make_inverse_ptt_params(*synth.random_tree(n, seed=b)) for b in range(B)]))
    rng = np.random.default_rng(11)
    P = 1 if param_batch == "one" else B
    mu = rng.uniform(-2, 2, (P, n - 1)).astype(np.float32)
    omega = np.log(rng.uniform(0.1, 1.0, (P, n - 1))).astype(np.float32)
    alpha = rng.uniform(-0.5, 0.5, (P, n - 1)).astype(np.float32)
    x = _lsn_x(rng, B, l, r, f, mu, omega, alpha)
    lp, g = pb.approx_log_prob(x, mu, omega, alpha, l, r, f)
    lp_o, g_o = ref.approx_log_prob(oracle, x, mu, omega, alpha, l, r, f)
    _compare(lp, g, lp_o, g_o)


def test_log_density_of_the_fits_own_draws(fx, oracle):
    """log q(xs) = sum log phi(zs0) - ladj for the draws lsn_draws makes (the ELBO's forward Jacobian terms, from the
    oracle): the density inverts the fit's forward path."""
    import polee_b200 as pb
    K = 8
    h = pb.Handle(num_mc_samples=K, noise_mode=1)
    h.set_sample(pb.RNASeqSample(fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval, fx.efflens))
    h.set_tree(fx.parent_idxs, fx.js)
    h.set_params(fx.mu, fx.omega, fx.alpha)
    zs0 = np.random.default_rng(4).normal(size=(K, fx.n - 1)).astype(np.float32)
    d = h.lsn_draws(zs0)
    h.close()
    lp = pb.approx_log_prob(d["xs"], fx.mu, fx.omega, fx.alpha, *pb.make_inverse_ptt_params(fx.parent_idxs, fx.js),
                            want_grad=False)
    model = oracle.Model(fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval)
    kept = 0
    for k in range(K):
        # the 1e-16 leaf floor, the 1e-10 clamp of xs and the clamp of y are not invertible
        if (d["xs"][k] <= 1e-10).any() or ((d["ys"][k] <= 1e-10) | (d["ys"][k] >= 1 - 1e-10)).any():
            continue
        o = oracle.lsn_draw(fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval, fx.efflens, fx.parent_idxs, fx.js, fx.mu,
                            fx.omega, fx.alpha, zs0[k], gradonly=False)
        ladj = o["elbo"] - model.log_likelihood(o["xs"], gradonly=False)[0]
        z = zs0[k].astype(np.float64)
        expected = np.sum(-0.5 * z * z - 0.5 * np.log(2 * np.pi)) - ladj
        assert relerr(lp[k], expected) <= 1e-4, (k, lp[k], expected)
        kept += 1
    assert kept >= 6


def _device_case(B=5, n=3001, seed=2):
    import polee_b200 as pb
    from polee_b200 import synth
    l, r, f = pb.make_inverse_ptt_params(*synth.random_tree(n, seed=seed))
    rng = np.random.default_rng(seed)
    mu = rng.uniform(-2, 2, (B, n - 1)).astype(np.float32)
    omega = np.log(rng.uniform(0.1, 1.0, (B, n - 1))).astype(np.float32)
    alpha = rng.uniform(-0.5, 0.5, (B, n - 1)).astype(np.float32)
    return (l, r, f), _lsn_x(rng, B, l, r, f, mu, omega, alpha), mu, omega, alpha


def test_device_form_equals_host_form_bit_for_bit():
    import torch
    import polee_b200 as pb
    idx, x, mu, omega, alpha = _device_case()
    B, n = x.shape
    plan = pb.HsbPlan(n, *idx)
    lp_h, g_h = plan.approx_log_prob(x, mu, omega, alpha)
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        d = [torch.from_numpy(a).cuda() for a in (x, mu, omega, alpha)]
        out = []
        for want_grad in (True, True, False):
            lp = torch.empty(B, dtype=torch.float64, device="cuda")
            g = torch.empty((B, n), dtype=torch.float32, device="cuda") if want_grad else None
            plan.approx_log_prob_device(B, B, *(t.data_ptr() for t in d), lp.data_ptr(), g.data_ptr() if want_grad else 0,
                                        st.cuda_stream)
            out.append((lp, g))
    st.synchronize()
    (lp1, g1), (lp2, g2), (lp3, _) = [(lp.cpu().numpy(), None if g is None else g.cpu().numpy()) for lp, g in out]
    assert np.array_equal(lp1, lp_h) and np.array_equal(g1, g_h)
    assert np.array_equal(lp1, lp2) and np.array_equal(g1, g2)
    assert np.array_equal(lp3, lp1)
    assert np.array_equal(plan.approx_log_prob(x, mu, omega, alpha, want_grad=False), lp_h)
    plan.close()


def test_torch_autograd():
    import torch
    import polee_b200 as pb
    idx, x, mu, omega, alpha = _device_case()
    B, n = x.shape
    plan = pb.HsbPlan(n, *idx)
    lp_h, g_h = plan.approx_log_prob(x, mu, omega, alpha)
    xt = torch.from_numpy(x).cuda().requires_grad_(True)
    lp = pb.approx_log_prob_torch(plan, xt, *(torch.from_numpy(a).cuda() for a in (mu, omega, alpha)))
    w = torch.from_numpy(np.random.default_rng(0).normal(size=B)).cuda()
    (gx,) = torch.autograd.grad((w * lp).sum(), xt)
    assert np.array_equal(lp.detach().cpu().numpy(), lp_h)
    expected = (w[:, None].cpu() * torch.from_numpy(g_h)).to(torch.float32).numpy()
    assert np.array_equal(gx.cpu().numpy(), expected)
    plan.close()


def test_edge_cases():
    import polee_b200 as pb
    from polee_b200 import _lib as L
    idx, x, mu, omega, alpha = _device_case()
    B, n = x.shape
    lp, g = pb.approx_log_prob(x, mu, omega, alpha, *idx)
    assert np.isfinite(lp).all()
    # a zero leaf whose sibling subtree is not zero: y = 0 or 1 at their parent
    l, r, f = idx
    p = next(j for j in range(2 * n - 1) if f[j] < 0 and f[r[j]] >= 0 and f[l[j]] < 0)
    x2 = x.copy()
    x2[2, f[r[p]]] = 0.0
    lp2, g2 = pb.approx_log_prob(x2, mu, omega, alpha, *idx)
    assert lp2[2] == -np.inf
    keep = np.arange(B) != 2
    assert np.array_equal(lp2[keep], lp[keep]) and np.array_equal(g2[keep], g[keep])

    plan = pb.HsbPlan(n, *idx)
    with pytest.raises(pb.PoleeError) as e:
        plan.approx_log_prob(x, mu[:2], omega[:2], alpha[:2])
    assert e.value.code == L.POLEE_EINVAL
    lib, P = plan.lib, C.c_void_p
    buf = [np.ascontiguousarray(a) for a in (x, mu, omega, alpha)]
    lpb = np.zeros(B)
    ptrs = [a.ctypes.data_as(P) for a in buf]
    for miss in range(5):
        args = ptrs + [lpb.ctypes.data_as(P)]
        args[miss] = None
        assert lib.polee_approx_log_prob_with_plan(plan.p, C.c_int64(B), C.c_int64(B), *args, None) == L.POLEE_EINVAL
        assert lib.polee_approx_log_prob_device(plan.p, C.c_int64(B), C.c_int64(B), *args, None, None) == L.POLEE_EINVAL
    assert lib.polee_approx_log_prob_with_plan(plan.p, C.c_int64(0), C.c_int64(1), *ptrs, lpb.ctypes.data_as(P),
                                               None) == L.POLEE_EINVAL
    plan.close()

    with pytest.raises(pb.PoleeError) as e:
        pb.approx_log_prob(np.full((1, 3), 1 / 3, np.float32), [0, 0], [0, 0], [0, 0], [1, 3, -1, -1, -1],
                           [2, 4, -1, -1, -1], [-1, -1, 0, 0, 1])
    assert e.value.code == L.POLEE_EBADTREE

    lp1, g1 = pb.approx_log_prob(np.ones((3, 1), np.float32), [], [], [], [-1], [-1], [0])   # n = 1
    assert np.array_equal(lp1, np.zeros(3)) and np.array_equal(g1, np.zeros((3, 1), np.float32))
