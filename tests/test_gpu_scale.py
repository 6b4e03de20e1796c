"""GPU tests at BASELINE.json sizes: the likelihood and its gradient against the oracle, elementwise, for every device
layout and arithmetic (equivalence classes in Float32 = the default and in Float64, fused row tiles, split,
reference-order accumulation), plus size-independent
properties: identity sum_j x_j g_j = m, determinism, agreement between K-batched and one-at-a-time evaluation."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _device_sample(m, n, seed, **kw):
    import torch
    from polee_b200 import synth
    s = synth.make_sample(m, n, seed=seed, device="cuda", **kw)
    colptr = s["colptr"].to(torch.int32)
    rowval = s["rowval"].to(torch.int32)
    return s, colptr, rowval


LAYOUTS = {"ec": {}, "ec64": {}, "fused": {"POLEE_LAYOUT": "fused"}, "split": {"POLEE_LAYOUT": "split"}, "exact": {}}
EXACT_MODE = {"exact": 1, "ec64": 2}   # opts.exact_accumulation (include/polee_b200.h)


def _layout_handle(pb, layout, monkeypatch, K, m, n, colptr, rowval, nzval):
    monkeypatch.delenv("POLEE_LAYOUT", raising=False)
    for k, v in LAYOUTS[layout].items():
        monkeypatch.setenv(k, v)
    h = pb.Handle(num_mc_samples=K, num_steps=3, exact_accumulation=EXACT_MODE.get(layout, 0))
    h.set_matrix_device(m, n, colptr.data_ptr(), rowval.data_ptr(), nzval.data_ptr())
    return h


def test_config2_shape_vs_oracle(oracle):
    """C2: m = 1 048 576, n = 20 000, K = 1 -- the oracle still finishes in seconds here."""
    import torch
    import polee_b200 as pb
    from polee_b200 import synth
    s, colptr, rowval = _device_sample(1 << 20, 20000, 20260002)
    ns = synth.to_numpy_sample(s)
    tree = synth.balanced_tree(20000, s["gene_sizes"].cpu().numpy())
    h = pb.Handle(num_mc_samples=1, num_steps=4, noise_mode=1)
    h.set_matrix_device(s["m"], s["n"], colptr.data_ptr(), rowval.data_ptr(), s["nzval"].data_ptr())
    h.set_efflens(ns["efflens"])
    h.set_tree(*tree)
    xs = np.random.default_rng(0).dirichlet(np.ones(20000)).astype(np.float32).clip(1e-10)
    lp, g = h.loglik_grad(xs, gradonly=False)
    lp_o, g_o = oracle.Model(ns["m"], ns["n"], ns["colptr"], ns["rowval"], ns["nzval"]).log_likelihood(xs, gradonly=False)
    assert abs(lp[0] - lp_o) <= 1e-8 * abs(lp_o)
    nz = g_o != 0
    assert np.max(np.abs(g[0][nz] - g_o[nz]) / g_o[nz]) <= 1e-5
    noise = np.random.default_rng(1).normal(size=(4, 1, 19999)).astype(np.float32)
    dev = h.fit(noise=noise)
    ora = oracle.fit_lsn_ptt(ns["m"], ns["n"], ns["colptr"], ns["rowval"], ns["nzval"], ns["efflens"], *tree,
                             num_steps=4, num_mc_samples=1, noise=noise)
    for key in ("mu", "omega", "alpha"):
        assert np.abs(dev[key] - ora[key]).max() <= 2e-4, key
    h.close()
    del s, colptr, rowval
    torch.cuda.empty_cache()


@pytest.fixture(scope="module")
def c3_sample():
    import torch
    from polee_b200 import synth
    m, n = 30_000_000, 200_000
    s, colptr, rowval = _device_sample(m, n, 20260003)
    ns = synth.to_numpy_sample(s)
    tree = synth.balanced_tree(n, s["gene_sizes"].cpu().numpy())
    yield s, colptr, rowval, ns, tree
    del s, colptr, rowval
    torch.cuda.empty_cache()


def test_config3_vs_oracle_all_layouts(oracle, c3_sample, monkeypatch):
    """C3 (the headline config: m = 30 M, n = 200 k, K = 8): ONE loglik_grad per device layout, lp and x_grad of two of
    the eight draws against the oracle elementwise (north_star: 1e-5 relative; the oracle needs < 1 s per draw)."""
    import polee_b200 as pb
    s, colptr, rowval, ns, tree = c3_sample
    m, n, K = s["m"], s["n"], 8
    xs = np.random.default_rng(0).dirichlet(np.ones(n), K).astype(np.float32).clip(1e-10)
    M = oracle.Model(m, n, ns["colptr"], ns["rowval"], ns["nzval"])
    ref = {k: M.log_likelihood(xs[k], gradonly=False) for k in (0, 5)}
    got = {}
    for layout in ("ec", "ec64", "fused", "split", "exact"):
        h = _layout_handle(pb, layout, monkeypatch, K, m, n, colptr, rowval, s["nzval"])
        h.set_tree(*tree)
        info = h.layout_info()
        if layout in ("ec", "ec64"):
            assert info["ec_rows"] > 0.9 * m, info             # the class layout takes nearly every row of C3
        else:
            assert info["ec_rows"] == 0 and info["general_kind"] == ("fused" if layout == "fused" else "split"), info
        lp, g = h.loglik_grad(xs, gradonly=False)
        h.close()
        for k, (lp_o, g_o) in ref.items():
            assert abs(lp[k] - lp_o) <= 1e-8 * abs(lp_o), (layout, k)
            nz = g_o != 0
            assert np.array_equal(g[k][~nz], g_o[~nz]), layout
            err = float(np.max(np.abs(g[k][nz] - g_o[nz]) / g_o[nz]))
            assert err <= 1e-5, (layout, k, err)
        got[layout] = g
    assert np.max(np.abs(got["ec"] - got["exact"]) / np.maximum(got["exact"], 1e-300)) <= 2e-6
    assert np.max(np.abs(got["ec64"] - got["exact"]) / np.maximum(got["exact"], 1e-300)) <= 2e-7


def test_config3_shape_properties(c3_sample):
    """C3 on one B200, default layout: gradient identity, determinism, batched == single, a finite fit."""
    import polee_b200 as pb
    s, colptr, rowval, ns, tree = c3_sample
    m, n, K = s["m"], s["n"], 8
    h = pb.Handle(num_mc_samples=K, num_steps=3)
    h.set_matrix_device(m, n, colptr.data_ptr(), rowval.data_ptr(), s["nzval"].data_ptr())
    nnz = s["nnz"]
    h.set_efflens(ns["efflens"])
    h.set_tree(*tree)
    rng = np.random.default_rng(0)
    xs = rng.dirichlet(np.ones(n), K).astype(np.float32).clip(1e-10)
    lp, g = h.loglik_grad(xs, gradonly=False)
    assert np.all(np.isfinite(lp)) and np.all(np.isfinite(g))
    ident = (xs.astype(np.float64) * g).sum(1)
    assert np.max(np.abs(ident - m)) <= 1e-5 * m                   # sum_j x_j g_j = m for every draw
    lp2, g2 = h.loglik_grad(xs, gradonly=False)
    assert np.array_equal(g, g2) and np.array_equal(lp, lp2)        # deterministic: no atomics
    lp1, g1 = h.loglik_grad(xs[3], gradonly=False)                  # K = 1 kernels on the same data
    assert abs(lp1[0] - lp[3]) <= 1e-10 * abs(lp[3])
    assert np.max(np.abs(g1[0] - g[3]) / np.maximum(g[3], 1e-300)) <= 1e-9
    out = h.fit()
    assert all(np.all(np.isfinite(out[k])) for k in ("mu", "omega", "alpha"))
    assert nnz > 100_000_000
    h.close()


def test_config5_many_samples_replicas():
    """C5 shape in miniature: whole samples handed to per-device workers (no collective); concurrent handles on
    one GPU give exactly the sequential results."""
    import polee_b200 as pb
    from polee_b200 import synth
    samples, trees = [], []
    for i in range(5):
        s = synth.make_sample(40000 + 7000 * i, 2500, seed=300 + i)
        ns = synth.to_numpy_sample(s)
        samples.append(pb.RNASeqSample(ns["m"], ns["n"], ns["colptr"], ns["rowval"], ns["nzval"], ns["efflens"]))
        trees.append(synth.balanced_tree(2500, s["gene_sizes"].numpy()))
    seq = [pb.approximate_likelihood(pb.LogitSkewNormalPTTApprox(), s, tree_topology=t, num_steps=30, num_mc_samples=8)
           for s, t in zip(samples, trees)]
    par = pb.prep_many(samples, trees, devices=(0, 0, 0), num_steps=30, num_mc_samples=8)
    for a, b in zip(seq, par):
        assert all(np.array_equal(a[k], b[k]) for k in ("mu", "omega", "alpha"))


def test_config4_shape_long_rows_vs_oracle(oracle, monkeypatch):
    """C4 shape (heavy multi-mapping: 10 % of the rows span 64-512 transcripts), one rank's share of the 8-GPU config:
    m = 4 M, n = 250 k, nnz ~ 120 M.  Every layout that accepts long rows against the oracle elementwise, then the
    gradient identity, determinism and a finite fit on the default layout."""
    import torch
    import polee_b200 as pb
    from polee_b200 import synth
    m, n, K = 4_000_000, 250_000, 8
    s, colptr, rowval = _device_sample(m, n, 20260004, long_rows=True)
    assert s["nnz"] > 100_000_000
    ns = synth.to_numpy_sample(s)
    tree = synth.balanced_tree(n, s["gene_sizes"].cpu().numpy())
    xs = np.random.default_rng(0).dirichlet(np.ones(n), K).astype(np.float32).clip(1e-10)
    M = oracle.Model(m, n, ns["colptr"], ns["rowval"], ns["nzval"])
    ref = {k: M.log_likelihood(xs[k], gradonly=False) for k in (2,)}
    for layout in ("ec", "ec64", "split", "exact"):
        h = _layout_handle(pb, layout, monkeypatch, K, m, n, colptr, rowval, s["nzval"])
        h.set_tree(*tree)
        lp, g = h.loglik_grad(xs, gradonly=False)
        h.close()
        for k, (lp_o, g_o) in ref.items():
            assert abs(lp[k] - lp_o) <= 1e-8 * abs(lp_o), (layout, k)
            nz = g_o != 0
            err = float(np.max(np.abs(g[k][nz] - g_o[nz]) / g_o[nz]))
            assert err <= 1e-5, (layout, k, err)
    monkeypatch.delenv("POLEE_LAYOUT", raising=False)
    h = pb.Handle(num_mc_samples=K, num_steps=3)
    h.set_matrix_device(m, n, colptr.data_ptr(), rowval.data_ptr(), s["nzval"].data_ptr())
    del s, colptr, rowval
    torch.cuda.empty_cache()
    h.set_efflens(ns["efflens"])
    h.set_tree(*tree)
    lp, g = h.loglik_grad(xs, gradonly=False)
    ident = (xs.astype(np.float64) * g).sum(1)
    assert np.max(np.abs(ident - m)) <= 1e-5 * m
    lp2, g2 = h.loglik_grad(xs, gradonly=False)
    assert np.array_equal(g, g2) and np.array_equal(lp, lp2)
    out = h.fit()
    assert all(np.all(np.isfinite(out[k])) for k in ("mu", "omega", "alpha"))
    h.close()
