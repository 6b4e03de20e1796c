"""The HSBGrad reference (tests/hsb_grad_ref.py) on the CPU: its forward is the reference's HSB, and its gradient is
the derivative of that forward."""
import os
import subprocess

import numpy as np
import pytest

import hsb_grad_ref as ref
from conftest import GOLDEN, ROOT


def _fd_check(oracle, parent_idxs, js, seed):
    l, r, f = oracle.make_inverse_ptt_params(parent_idxs, js)
    n = (len(js) + 1) // 2
    rng = np.random.default_rng(seed)
    yl = rng.uniform(-2, 2, n - 1)
    w = rng.normal(size=n)
    g = ref.hsb_grad(w[None], yl[None], l, r, f)[0]
    h = 1e-5
    rows = np.repeat(yl[None], 2 * (n - 1), axis=0)  # row 2k: y_logit_k + h, row 2k + 1: y_logit_k - h
    k = np.arange(n - 1)
    rows[2 * k, k] += h
    rows[2 * k + 1, k] -= h
    loss = ref.forward(rows, l, r, f)[0] @ w
    fd = (loss[0::2] - loss[1::2]) / (2 * h)
    scale = np.abs(g).max()
    assert scale > 0
    assert np.abs(g - fd).max() <= 1e-6 * scale
    big = np.abs(g) > 1e-3 * scale
    assert (np.abs(g - fd)[big] <= 1e-6 * np.abs(g)[big] + 1e-9 * scale).all()


def test_forward_matches_reference_hsb(oracle):
    v = np.load(os.path.join(GOLDEN, "hsb_reference_vectors.npz"))
    for case in ("fixture_shared", "random97_shared", "per_row"):
        g = lambda k: v["%s__%s" % (case, k)]  # noqa: E731
        x = ref.forward(g("y_logit"), g("left"), g("right"), g("leaf"))[0]
        xo = oracle.hsb(g("y_logit"), g("left"), g("right"), g("leaf"))
        assert np.array_equal(x.astype(np.float32), xo), case
        np.testing.assert_allclose(x.sum(1), 1.0, rtol=1e-12)


def test_gradient_matches_finite_differences_random_64(oracle):
    from polee_b200 import synth
    _fd_check(oracle, *synth.random_tree(64, seed=5), seed=1)


def test_gradient_matches_finite_differences_fixture(oracle, fx):
    _fd_check(oracle, fx.parent_idxs, fx.js, seed=2)


def test_gradient_of_constant_x_grad_is_zero(oracle, fx):
    """sum(x) is 1 whatever y_logit, so x_grad = c 1 has a zero gradient"""
    l, r, f = oracle.make_inverse_ptt_params(fx.parent_idxs, fx.js)
    yl = np.random.default_rng(3).uniform(-3, 3, (2, fx.n - 1))
    g = ref.hsb_grad(np.full((2, fx.n), 2.5), yl, l, r, f)
    assert np.abs(g).max() <= 1e-12 * 2.5


def test_hsb_grad_tf_harness_compiles(tmp_path):
    """The HSBGrad registrations of the TF plugin and their stub-TF harness compile and link (the GPU tests drive them)"""
    lib = os.path.join(ROOT, "polee_b200", "libpolee_b200.so")
    if not os.path.exists(lib):
        pytest.skip("libpolee_b200.so is not built")
    out = str(tmp_path / "libhsb_grad_shim.so")
    subprocess.check_call(hsb_grad_shim_cmd(out))
    assert os.path.getsize(out) > 0


def hsb_grad_shim_cmd(out):
    """g++ command that links polee_b200/tf/hsb_ops_b200.cpp with tests/tf_shim/hsb_grad_harness.cpp against the stub
    TF API (as tests/tf_shim/Makefile builds the shim of the other three ops)"""
    return ["g++", "-std=c++14", "-shared", "-fPIC", "-O2", "-Wall", "-I" + os.path.join(ROOT, "oracle", "tf_stub"),
            "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "polee_b200", "tf", "hsb_ops_b200.cpp"),
            os.path.join(ROOT, "tests", "tf_shim", "hsb_grad_harness.cpp"), "-o", out,
            "-L" + os.path.join(ROOT, "polee_b200"), "-lpolee_b200", "-Wl,-rpath," + os.path.join(ROOT, "polee_b200"),
            "-lpthread"]
