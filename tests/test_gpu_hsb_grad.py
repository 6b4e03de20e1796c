"""HSBGrad on the device (polee_hsb_grad*, DESIGN.md K4) against the Float64 restatement (tests/hsb_grad_ref.py), the
fit's own tree backward, its host and plan-less forms, torch autograd and the TF plugin's registrations."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import hsb_grad_ref as ref
from conftest import GOLDEN
from test_hsb_grad_oracle import hsb_grad_shim_cmd

pytestmark = pytest.mark.gpu

P = C.c_void_p


def _p(a):
    return a.ctypes.data_as(P)


def _check(dev, want):
    """each row within 1e-6 of that row's largest |value|, and >= 98 % of all elements bit-identical to the Float32
    rounding of the reference: y's exp (the device's against the C library's) is the only source of difference"""
    assert dev.dtype == np.float32 and dev.shape == want.shape
    for b in range(want.shape[0]):
        assert np.abs(dev[b] - want[b]).max() <= 1e-6 * np.abs(want[b]).max(), b
    assert (dev == want.astype(np.float32)).mean() >= 0.98


def _idx(parent_js_list):
    import polee_b200 as pb
    return [np.stack(a) for a in zip(*[pb.make_inverse_ptt_params(*t) for t in parent_js_list])]


def _inputs(B, n, seed):
    rng = np.random.default_rng(seed)
    return rng.normal(size=(B, n)).astype(np.float32), rng.uniform(-3, 3, (B, n - 1)).astype(np.float32)


@pytest.mark.parametrize("case", ["fixture_shared", "random97_shared", "per_row"])
def test_reference_vector_trees(case):
    import polee_b200 as pb
    v = np.load(os.path.join(GOLDEN, "hsb_reference_vectors.npz"))
    g = lambda k: v["%s__%s" % (case, k)]  # noqa: E731
    yl = g("y_logit")
    xg = np.random.default_rng(7).normal(size=(yl.shape[0], yl.shape[1] + 1)).astype(np.float32)
    idx = [g("left"), g("right"), g("leaf")]
    want = ref.hsb_grad(xg, yl, *idx)
    _check(pb.hsb_grad(xg, yl, *idx), want)
    if case != "per_row":
        assert np.array_equal(pb.hsb_grad(xg, yl, *[a[:1] for a in idx]), pb.hsb_grad(xg, yl, *idx))


@pytest.mark.parametrize("shape", ["balanced", "random"])
@pytest.mark.parametrize("trees", ["shared", "per_row"])
def test_20000_leaves(shape, trees):
    import polee_b200 as pb
    from polee_b200 import synth
    n = 20000
    B = 64 if trees == "shared" else 32
    make = (lambda s: synth.balanced_tree(n)) if shape == "balanced" else (lambda s: synth.random_tree(n, seed=s))
    if trees == "shared":
        idx = _idx([make(0)])
    elif shape == "balanced":  # the balanced tree with its leaves permuted differently in every row
        pi, js = make(0)
        rng = np.random.default_rng(5)
        perm = lambda: np.concatenate([[0], rng.permutation(n) + 1]).astype(np.int32)  # noqa: E731
        idx = _idx([(pi, np.where(js > 0, perm()[js], 0).astype(np.int32)) for _ in range(B)])
    else:
        idx = _idx([make(s) for s in range(B)])
    xg, yl = _inputs(B, n, 3)
    dev = pb.hsb_grad(xg, yl, *idx)
    _check(dev, ref.hsb_grad(xg, yl, *idx))
    assert np.array_equal(pb.hsb_grad(xg, yl, *idx), dev)  # reruns give the same bits
    if trees == "shared":
        assert np.array_equal(pb.hsb_grad(xg, yl, *[np.repeat(a, B, 0) for a in idx]), dev)


def test_constant_x_grad_gives_zero(fx):
    """sum(x) = 1 whatever y_logit: x_grad = c 1 on a row has a zero gradient"""
    import polee_b200 as pb
    from polee_b200 import synth
    for pi, js in ((fx.parent_idxs, fx.js), synth.random_tree(6000, seed=2)):
        l, r, f = pb.make_inverse_ptt_params(pi, js)
        n = (len(js) + 1) // 2
        c = np.array([1.0, -3.5, 1e3], np.float32)
        yl = np.random.default_rng(1).uniform(-4, 4, (3, n - 1)).astype(np.float32)
        g = pb.hsb_grad(np.repeat(c[:, None], n, 1), yl, l, r, f)
        assert (np.abs(g) <= 1e-12 * np.abs(c)[:, None]).all()


def test_device_host_and_planless_forms_agree():
    import torch
    import polee_b200 as pb
    from polee_b200 import _lib as L
    from polee_b200 import synth
    lib = L.load_library()
    for trees in ("shared", "per_row"):
        n, B = 5000, 8
        idx = _idx([synth.random_tree(n, seed=s) for s in range(1 if trees == "shared" else B)])
        xg, yl = _inputs(B, n, 9)
        plan = pb.HsbPlan(n, *idx)
        host = np.zeros((B, n - 1), np.float32)
        assert lib.polee_hsb_grad_with_plan(plan.p, C.c_int64(B), _p(xg), _p(yl), _p(host)) == 0
        st = torch.cuda.Stream()
        with torch.cuda.stream(st):
            d_xg, d_yl = torch.from_numpy(xg).cuda(), torch.from_numpy(yl).cuda()
            d_out = torch.full((B, n - 1), float("nan"), device="cuda")
            for _ in range(2):  # the second call reuses the plan's scratch
                plan.hsb_grad_device(B, d_xg.data_ptr(), d_yl.data_ptr(), d_out.data_ptr(), st.cuda_stream)
        st.synchronize()
        assert np.array_equal(d_out.cpu().numpy(), host)
        assert np.array_equal(pb.hsb_grad(xg, yl, *idx), host)
        plan.close()


@pytest.mark.parametrize("tree", ["fixture", "random6000"])
def test_matches_the_fits_tree_backward(fx, tree):
    """y (1 - y) transform_gradients_no_ladj(y, x_grad): the fit's k3s_tree_bwd keeps the reference's Float32 G (one
    Float32 rounding per level, ~40 levels on these trees, each <= 6e-8 relative), so the two agree to about 1e-5 of a
    row's largest value, not bit for bit"""
    import polee_b200 as pb
    from polee_b200 import synth
    pi, js = (fx.parent_idxs, fx.js) if tree == "fixture" else synth.random_tree(6000, seed=4)
    n = (len(js) + 1) // 2
    B = 4
    xg, yl = _inputs(B, n, 13)
    y = ref.sigmoid(yl)
    t = pb.PolyaTreeTransform(pi, js)
    fit = y * (1 - y) * t.transform_gradients_no_ladj(y, xg.astype(np.float64)).astype(np.float64)
    dev = pb.hsb_grad(xg, yl, *pb.make_inverse_ptt_params(pi, js))
    for b in range(B):
        assert np.abs(dev[b] - fit[b]).max() <= 5e-5 * np.abs(fit[b]).max(), b


def test_torch_hsb_backward_is_hsb_grad(fx):
    import torch
    import polee_b200 as pb
    idx = pb.make_inverse_ptt_params(fx.parent_idxs, fx.js)
    plan = pb.HsbPlan(fx.n, *idx)
    w_np, yl_np = _inputs(6, fx.n, 17)
    yl = torch.from_numpy(yl_np).cuda().requires_grad_()
    x = pb.hsb_torch(plan, yl)
    assert np.array_equal(x.detach().cpu().numpy(), pb.hsb(yl_np, *idx))
    (g,) = torch.autograd.grad((torch.from_numpy(w_np).cuda() * x).sum(), yl)
    assert np.array_equal(g.cpu().numpy(), pb.hsb_grad(w_np, yl_np, *idx))
    plan.close()


def test_torch_inv_hsb_backward_is_inv_hsb_grad(fx):
    import torch
    import polee_b200 as pb
    idx = pb.make_inverse_ptt_params(fx.parent_idxs, fx.js)
    plan = pb.HsbPlan(fx.n, *idx)
    B = 5
    rng = np.random.default_rng(19)
    x_np = rng.dirichlet(np.ones(fx.n), B).astype(np.float32)
    gy, gl = rng.normal(size=(B, fx.n - 1)), rng.normal(size=(B, 1)).astype(np.float32)
    y_np, ladj_np = pb.inv_hsb(x_np, *idx)
    for use in ("both", "y", "ladj"):
        x = torch.from_numpy(x_np).cuda().requires_grad_()
        y, ladj = pb.inv_hsb_torch(plan, x)
        assert np.array_equal(y.detach().cpu().numpy(), y_np) and np.array_equal(ladj.detach().cpu().numpy(), ladj_np)
        loss = 0
        if use != "ladj":
            loss = loss + (torch.from_numpy(gy).cuda() * y).sum()
        if use != "y":
            loss = loss + (torch.from_numpy(gl).cuda() * ladj).sum()
        (g,) = torch.autograd.grad(loss, x)
        want = pb.inv_hsb_grad(gy if use != "ladj" else np.zeros_like(gy), gl if use != "y" else np.zeros_like(gl), y_np,
                               ladj_np, *idx)
        assert np.array_equal(g.cpu().numpy(), want), use
    plan.close()


def test_torch_reparameterised_draw_matches_finite_differences(fx):
    """x = hsb_torch(mu + e^omega sinh(asinh eps + alpha)): d(sum w x)/d(mu, omega, alpha) through autograd against
    central differences of the Float64 restatement.  The device forms y_logit in Float32 and returns a Float32
    gradient, so agreement is to ~1e-4 of the largest entry, not to the bits."""
    import torch
    import polee_b200 as pb
    idx = pb.make_inverse_ptt_params(fx.parent_idxs, fx.js)
    plan = pb.HsbPlan(fx.n, *idx)
    nm1, B = fx.n - 1, 3
    rng = np.random.default_rng(23)
    eps = rng.normal(size=(B, nm1))
    w = rng.normal(size=(B, fx.n))
    prm = [fx.mu.astype(np.float64), fx.omega.astype(np.float64), fx.alpha.astype(np.float64)]
    t = [torch.tensor(a, dtype=torch.float32, device="cuda", requires_grad=True) for a in prm]
    e = torch.tensor(eps, dtype=torch.float32, device="cuda")
    x = pb.hsb_torch(plan, t[0] + torch.exp(t[1]) * torch.sinh(torch.asinh(e) + t[2]))
    grads = torch.autograd.grad((torch.tensor(w, dtype=torch.float32, device="cuda") * x).sum(), t)
    ks = rng.choice(nm1, 24, replace=False)
    h = 1e-6

    def loss(mu, om, al):  # rows: the B draws of every perturbed parameter set, stacked
        yl = mu[:, None] + np.exp(om)[:, None] * np.sinh(np.arcsinh(eps)[None] + al[:, None])
        xs = ref.forward(yl.reshape(-1, nm1), *idx)[0].reshape(mu.shape[0], B, fx.n)
        return (xs * w[None]).sum((1, 2))

    for which in range(3):
        g = grads[which].cpu().numpy().astype(np.float64)
        assert np.isfinite(g).all()
        stack = [np.repeat(a[None], 2 * len(ks), 0) for a in prm]
        stack[which][np.arange(0, 2 * len(ks), 2), ks] += h
        stack[which][np.arange(1, 2 * len(ks), 2), ks] -= h
        L = loss(*stack)
        fd = (L[0::2] - L[1::2]) / (2 * h)
        assert np.abs(g[ks] - fd).max() <= 1e-4 * np.abs(fd).max() + 1e-6, (which, g[ks], fd)
    plan.close()


def test_tf_shim_hsb_grad_registrations(tmp_path):
    """The plugin's HSBGrad DEVICE_CPU and DEVICE_GPU kernels, driven through the stub TF API, give the C ABI's bits"""
    import torch
    import polee_b200 as pb
    out = str(tmp_path / "libhsb_grad_shim.so")
    subprocess.check_call(hsb_grad_shim_cmd(out))
    shim = C.CDLL(out)
    v = np.load(os.path.join(GOLDEN, "hsb_reference_vectors.npz"))
    st = torch.cuda.Stream()
    for case in ("fixture_shared", "per_row"):
        g = lambda k: np.ascontiguousarray(v["%s__%s" % (case, k)])  # noqa: E731
        L, R, F, yl = g("left"), g("right"), g("leaf"), g("y_logit")
        B, n = yl.shape[0], yl.shape[1] + 1
        xg = np.random.default_rng(29).normal(size=(B, n)).astype(np.float32)
        want = pb.hsb_grad(xg, yl, L, R, F)
        host = np.zeros((B, n - 1), np.float32)
        assert shim.shim_hsb_grad(C.c_int64(B), C.c_int64(n), _p(xg), _p(yl), _p(L), _p(R), _p(F), _p(host)) == 0
        assert np.array_equal(host, want)
        with torch.cuda.stream(st):
            t_xg, t_yl = torch.from_numpy(xg).cuda(), torch.from_numpy(yl).cuda()
            t_out = torch.zeros((B, n - 1), dtype=torch.float32, device="cuda")
            assert shim.shim_hsb_grad_gpu(C.c_int64(B), C.c_int64(n), P(t_xg.data_ptr()), P(t_yl.data_ptr()), _p(L), _p(R),
                                          _p(F), P(t_out.data_ptr()), P(st.cuda_stream)) == 0
        st.synchronize()
        assert np.array_equal(t_out.cpu().numpy(), want)


def test_errors_and_n1(fx):
    import torch
    import polee_b200 as pb
    from polee_b200 import _lib as L
    lib = L.load_library()
    with pytest.raises(pb.PoleeError) as e:
        pb.hsb_grad(np.zeros((1, 3), np.float32), np.zeros((1, 2), np.float32), [1, 3, -1, -1, -1], [2, 4, -1, -1, -1],
                    [-1, -1, 0, 0, 1])
    assert e.value.code == L.POLEE_EBADTREE
    l, r, f = pb.make_inverse_ptt_params(fx.parent_idxs, fx.js)
    n, B = fx.n, 2
    xg, yl = _inputs(B, n, 31)
    out = np.zeros((B, n - 1), np.float32)
    args = [_p(xg), _p(yl), _p(l), _p(r), _p(f), _p(out)]
    call = lambda a, b=B, ib=1: lib.polee_hsb_grad(C.c_int32(0), C.c_int64(b), C.c_int64(n), a[0], a[1], a[2], a[3], a[4],  # noqa: E731
                                                   C.c_int64(ib), a[5])
    assert call(args) == L.POLEE_OK
    for i in range(len(args)):
        assert call(args[:i] + [None] + args[i + 1:]) == L.POLEE_EINVAL, i
    assert call(args, b=0) == L.POLEE_EINVAL
    assert call(args, ib=3) == L.POLEE_EINVAL
    plan = pb.HsbPlan(n, l, r, f)
    hp = [_p(xg), _p(yl), _p(out)]
    for i in range(3):
        a = hp[:i] + [None] + hp[i + 1:]
        assert lib.polee_hsb_grad_with_plan(plan.p, C.c_int64(B), *a) == L.POLEE_EINVAL, i
        assert lib.polee_hsb_grad_device(plan.p, C.c_int64(B), *a, None) == L.POLEE_EINVAL, i
    assert lib.polee_hsb_grad_with_plan(plan.p, C.c_int64(0), *hp) == L.POLEE_EINVAL
    assert lib.polee_hsb_grad_with_plan(None, C.c_int64(B), *hp) == L.POLEE_EINVAL
    plan.close()
    per_row = pb.HsbPlan(n, np.stack([l] * 3), np.stack([r] * 3), np.stack([f] * 3))  # idx_batch 3, B 2
    assert lib.polee_hsb_grad_with_plan(per_row.p, C.c_int64(B), *hp) == L.POLEE_EINVAL
    per_row.close()
    # n = 1: no internal node, an empty output and POLEE_OK
    g1 = pb.hsb_grad(np.ones((3, 1), np.float32), np.zeros((3, 0), np.float32), [-1], [-1], [0])
    assert g1.shape == (3, 0)
    plan1 = pb.HsbPlan(1, [-1], [-1], [0])
    d = torch.ones((3, 1), device="cuda")
    plan1.hsb_grad_device(3, d.data_ptr(), d.data_ptr(), d.data_ptr())
    torch.cuda.synchronize()
    assert (d == 1).all()
    plan1.close()
