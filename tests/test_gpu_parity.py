"""GPU parity tests: the CUDA path (through the C ABI) against the oracle on the same seeded inputs.

Tolerances (north_star): integer / index work bit-exact; log-likelihood and gradient within 1e-5 relative;
tree forward/backward bit-exact given identical inputs (same IEEE ops per node, level-synchronous order is
irrelevant); reparameterised quantities within Float32 libm differences (stated per assert)."""
import numpy as np
import pytest

from conftest import relerr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pb():
    import polee_b200
    return polee_b200


def _sample(pb, fx):
    return pb.RNASeqSample(fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval, fx.efflens)


def _synth_sample(pb, s):
    return pb.RNASeqSample(s["m"], s["n"], s["colptr"], s["rowval"], s["nzval"], s["efflens"])


@pytest.mark.parametrize("exact", [False, True])
@pytest.mark.parametrize("K", [1, 2, 3, 5, 6, 7, 8, 12, 16])
def test_loglik_and_gradient_fixture(pb, fx, oracle, K, exact):
    """K1 + K2 vs sparse.jl restated: lp and x_grad <= 1e-5 relative, identity sum_j x_j g_j = m.
    exact=True: reference-order all-Float64 sums (p bit-identical); exact=False: the default fast kernels."""
    rng = np.random.default_rng(K)
    xs = rng.dirichlet(np.ones(fx.n), K).astype(np.float32).clip(1e-10)
    xs[0] = np.float32(1) / np.float32(fx.n)
    h = pb.Handle(num_mc_samples=K, exact_accumulation=exact)
    h.set_sample(_sample(pb, fx))
    h.set_tree(fx.parent_idxs, fx.js)
    lp, g = h.loglik_grad(xs, gradonly=False)
    M = oracle.Model(fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval)
    for k in range(K):
        lp_o, g_o = M.log_likelihood(xs[k], gradonly=False)
        assert abs(lp[k] - lp_o) <= 1e-5 * abs(lp_o)
        assert abs(lp[k] - lp_o) <= (1e-12 if exact else 1e-9) * abs(lp_o)   # exact: p is bit-identical, only the sum order differs
        assert relerr(g[k], g_o) <= 1e-5
        assert abs(xs[k].astype(np.float64) @ g[k] - fx.m) <= 1e-5 * fx.m
    assert abs(lp[0] - (-364724.375767)) < 1e-4                  # SURVEY 8c known answer
    lp0, g0 = h.loglik_grad(xs, gradonly=True)
    assert np.all(lp0 == 0.0) and np.array_equal(g0, g)          # gradonly: same gradient, lp = 0; deterministic
    h.close()


def test_frag_probs_bitwise(pb, fx, oracle):
    """1/frag_probs: frag_probs is accumulated exactly as pAt_mul_B! does, then rounded once to Float32."""
    xs = np.random.default_rng(0).dirichlet(np.ones(fx.n)).astype(np.float32).clip(1e-10)
    h = pb.Handle(num_mc_samples=1, exact_accumulation=True)
    h.set_sample(_sample(pb, fx))
    h.set_tree(fx.parent_idxs, fx.js)
    w = h.frag_prob_recip(xs)
    M = oracle.Model(fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval)
    M.log_likelihood(xs)
    expect = (np.float32(1) / M.frag_probs.astype(np.float32)).astype(np.float32)
    assert np.array_equal(w, expect)
    h.close()
    h = pb.Handle(num_mc_samples=1)                                 # default fast kernels: same to ~1 ulp of Float32
    h.set_sample(_sample(pb, fx))
    h.set_tree(fx.parent_idxs, fx.js)
    assert relerr(h.frag_prob_recip(xs), expect) <= 3e-7
    h.close()


def test_factored_likelihood(pb, fx, oracle):
    ks = np.random.default_rng(2).integers(1, 9, fx.m)
    xs = np.random.default_rng(3).dirichlet(np.ones(fx.n)).astype(np.float32).clip(1e-10)
    lp, g = pb.log_likelihood(_sample(pb, fx), xs, gradonly=False, ks=ks, tree=(fx.parent_idxs, fx.js))
    lp_o, g_o = oracle.Model(fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval).log_likelihood(xs, gradonly=False, ks=ks)
    assert abs(lp - lp_o) <= 1e-8 * abs(lp_o) and relerr(g, g_o) <= 1e-5


def _trees(fx):
    from polee_b200 import synth
    from polee_b200.api import sequential_tree
    return {"fixture": (fx.parent_idxs, fx.js), "sequential": sequential_tree(fx.n),
            "random": synth.random_tree(fx.n, 3), "balanced": synth.balanced_tree(fx.n),
            # large trees: several bottom bins and a top part
            "balanced_20001": synth.balanced_tree(20001), "random_6000": synth.random_tree(6000, 9),
            "random_6000_K16": synth.random_tree(6000, 9),
            "spine_1225": synth.spine_tree(1200, 100), "sequential_6000": sequential_tree(6000)}


# the kernels each tree of test_tree_forward_backward_bit_exact takes (Handle.layout_info()["tree_route"]);
# sequential_6000 runs with POLEE_CHAIN_MIN_NODES raised, so that it does not take the chain scans
_TREE_ROUTES = {"fixture": "dfs", "sequential": "path", "random": "dfs", "balanced": "dfs", "balanced_20001": "dfs",
                "random_6000": "dfs", "random_6000_K16": "dfs", "spine_1225": "levels_smem",
                "sequential_6000": "levels_global"}


@pytest.mark.parametrize("tree", list(_TREE_ROUTES))
def test_tree_forward_backward_bit_exact(pb, fx, oracle, tree, monkeypatch):
    """transform!, both transform_gradients and inverse_transform! bit for bit against the oracle, on every route but
    the chain scans (test_large_sequential_tree_scan_path); random_6000_K16 runs 16 draws, where the DFS-run kernel
    needs 4 times the shared memory of K = 4."""
    pi, js = _trees(fx)[tree]
    n = (len(pi) + 1) // 2
    K = 16 if tree.endswith("_K16") else 4
    rng = np.random.default_rng(1)
    to = oracle.PTT(pi, js)
    if tree in ("spine_1225", "sequential_6000"):
        # ys of a near-uniform composition: u stays O(1/n) along paths of 1200 or 6000 nodes
        x0 = rng.dirichlet(np.ones(n) * 5.0, K).astype(np.float32)
        ys = np.stack([to.inverse_transform(x0[k])[0] for k in range(K)])
    else:
        lo = 0.3 if tree == "sequential" else 0.01   # keep a depth-312 product inside the Float32 range
        ys = rng.uniform(lo, 0.99, (K, n - 1))
    x_grad = rng.normal(size=(K, n)) * 1000
    if tree == "sequential_6000":
        monkeypatch.setenv("POLEE_CHAIN_MIN_NODES", str(10 ** 9))
    t = pb.PolyaTreeTransform(pi, js)
    xs, ladj = t.transform(ys, compute_ladj=True)
    assert t.handle.layout_info()["tree_route"] == _TREE_ROUTES[tree]
    yg = t.transform_gradients(ys, x_grad)
    yg0 = t.transform_gradients_no_ladj(ys, x_grad)
    for k in range(K):
        xo, ladj_o = to.transform(ys[k], True)
        assert np.array_equal(xs[k], xo)
        assert abs(ladj[k] - ladj_o) <= 1e-12 * abs(ladj_o)
        assert np.array_equal(yg[k], to.transform_gradients(ys[k], x_grad[k]), equal_nan=True)
        assert np.array_equal(yg0[k], to.transform_gradients_no_ladj(ys[k], x_grad[k]).astype(np.float32), equal_nan=True)
    # transform!(inverse_transform!(x)) = x   (KAT 1 of SURVEY 8c)
    x = rng.dirichlet(np.ones(n)).astype(np.float32)
    y_inv, ladj_inv = t.inverse_transform(x)
    yo, lo_ = to.inverse_transform(x)
    # y: one Float64 add and one divide per node in the reference's association -> the same bits; ladj: the device's logf
    # (<= 1 ulp) feeds a Float64 accumulator in the reference's order
    assert np.array_equal(y_inv, yo) and abs(ladj_inv - lo_) <= 1e-6 * abs(lo_)
    np.testing.assert_allclose(t.transform(y_inv)[0], x, rtol=3e-6)


@pytest.mark.parametrize("tree", ["fixture", "balanced", "sequential", "sequential_scan"])
def test_inverse_transform_on_device(pb, fx, oracle, tree):
    """inverse_transform! (ptt.jl:257-285) is a device kernel (level-synchronous sums; a serial per-draw sweep for deep
    caterpillar trees): y bit-identical to the oracle for several draws at once (K = 3 is padded to 4 lanes), and the
    fit's starting point mu = Float32(logit(inverse_transform!(fill(1f0/n)))) (l-a.jl:451-453) equals the oracle's."""
    from polee_b200 import synth
    if tree == "fixture":
        n, (pi, js) = fx.n, (fx.parent_idxs, fx.js)
    elif tree == "balanced":
        n = 5000
        pi, js = synth.balanced_tree(n)
    else:
        n = 700 if tree == "sequential" else 3000          # >= 4096 nodes: the chain path
        pi, js = pb.api.sequential_tree(n)
    rng = np.random.default_rng(len(tree))
    K = 3
    xs = rng.dirichlet(np.ones(n) * 2.0, K).astype(np.float32)
    h = pb.Handle(num_mc_samples=K)
    h.n = n
    h.set_tree(pi, js)
    ys, ladj = h.ptt_inverse_transform(xs)
    to = oracle.PTT(pi, js)
    for k in range(K):
        yo, lo_ = to.inverse_transform(xs[k])
        assert np.array_equal(ys[k], yo), (tree, k)
        assert abs(ladj[k] - lo_) <= 1e-6 * abs(lo_)
    mu, omega, alpha = h.get_params()
    y0, _ = to.inverse_transform(np.full(n, np.float32(1) / np.float32(n), np.float32))
    mu_o = np.log(y0 / (1.0 - y0)).astype(np.float32)
    assert np.abs(mu - mu_o).max() <= 2e-7 * max(1.0, np.abs(mu_o).max()) and (mu != mu_o).mean() <= 1e-3
    assert np.all(omega == np.log(np.float32(0.1))) and np.all(alpha == 0)
    h.close()


def test_bad_trees_are_rejected(pb, fx):
    import polee_b200._lib as L
    h = pb.Handle(num_mc_samples=1)
    bad = fx.parent_idxs.copy()
    bad[5] = 600                                       # parent index after the child
    with pytest.raises(pb.PoleeError) as e:
        h.set_tree(bad, fx.js)
    assert e.value.code == L.POLEE_EBADTREE
    js = fx.js.copy()
    js[np.nonzero(js)[0][0]] = js[np.nonzero(js)[0][1]]  # duplicate leaf id
    with pytest.raises(pb.PoleeError):
        h.set_tree(fx.parent_idxs, js)
    with pytest.raises(pb.PoleeError):                 # fit without inputs: EINVAL, not a crash
        h.run_steps(1)
    h.close()


@pytest.mark.parametrize("K,gradonly", [(6, False), (8, True), (1, False)])
def test_one_step_of_draws_matches_oracle(pb, fx, oracle, K, gradonly):
    """likelihood-approximation.jl:511-559 for K draws with injected noise, at non-trivial parameters."""
    rng = np.random.default_rng(10 + K)
    h = pb.Handle(num_mc_samples=K, gradonly=gradonly, noise_mode=1, num_steps=2)
    h.set_sample(_sample(pb, fx))
    h.set_tree(fx.parent_idxs, fx.js)
    mu, om, al = h.get_params()
    al = (rng.normal(size=fx.n - 1) * 0.1).astype(np.float32)
    om = (om + rng.normal(size=fx.n - 1) * 0.3).astype(np.float32)
    h.set_params(mu, om, al)
    zs0 = rng.normal(size=(K, fx.n - 1)).astype(np.float32)
    d = h.lsn_draws(zs0)
    acc = {k: np.zeros(fx.n - 1, np.float32) for k in ("mu_grad", "omega_grad", "alpha_grad")}
    elbo = 0.0
    for k in range(K):
        o = oracle.lsn_draw(fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval, fx.efflens, fx.parent_idxs, fx.js, mu, om, al,
                            zs0[k], gradonly=gradonly)
        assert relerr(d["ys"][k], o["ys"]) <= 2e-6           # Float32 expf / sinhf / asinhf: CUDA vs glibc, few ulp
        assert relerr(d["xs"][k], o["xs"]) <= 2e-5           # product of <= 18 such factors
        scale = np.abs(o["x_grad"]).max()
        assert np.abs(d["x_grad"][k] - o["x_grad"]).max() <= 1e-5 * scale
        assert np.abs(d["y_grad"][k] - o["y_grad"]).max() <= 1e-5 * np.abs(o["y_grad"]).max()
        for key in acc:
            acc[key] += o[key]
        elbo += o["elbo"]
    for key in acc:
        ref = acc[key] / np.float32(K)
        assert np.abs(d[key] - ref).max() <= 1e-5 * np.abs(ref).max(), key
    if not gradonly:
        assert abs(d["elbo"] - elbo / K) <= 1e-7 * abs(elbo / K)
    h.close()


@pytest.mark.parametrize("K,steps", [(6, 80), (8, 40)])
def test_fit_trajectory_matches_oracle_with_injected_noise(pb, fx, oracle, K, steps):
    """End to end: same noise -> the fitted parameters and the ELBO trajectory track the oracle.
    Stated tolerance: 2e-4 absolute on mu/omega/alpha after `steps` ADAM steps, 1e-6 relative on the ELBO."""
    noise = np.random.default_rng(K).normal(size=(steps, K, fx.n - 1)).astype(np.float32)
    ora = oracle.fit_lsn_ptt(fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval, fx.efflens, fx.parent_idxs, fx.js,
                             num_steps=steps, num_mc_samples=K, noise=noise, gradonly=False, elbo_fix=True)
    dev = pb.approximate_likelihood(pb.LogitSkewNormalPTTApprox(), _sample(pb, fx), tree_topology=(fx.parent_idxs, fx.js),
                                    num_steps=steps, num_mc_samples=K, noise=noise, gradonly=False, want_elbo=True)
    for key in ("mu", "omega", "alpha"):
        assert np.abs(dev[key] - ora[key]).max() <= 2e-4, key
    assert relerr(dev["elbo"], ora["elbo"]) <= 1e-6
    assert "node_parent_idxs" not in dev                       # topology was an input (l-a.jl:618)
    # and with gradonly (the default) the ELBO is identically 0 as in the reference (SURVEY App. C2)
    dev0 = pb.approximate_likelihood(pb.LogitSkewNormalPTTApprox(), _sample(pb, fx), tree_topology=(fx.parent_idxs, fx.js),
                                     num_steps=steps, num_mc_samples=K, noise=noise, want_elbo=True)
    assert np.all(dev0["elbo"] == 0.0)
    for key in ("mu", "omega", "alpha"):
        assert np.abs(dev0[key] - ora[key]).max() <= 2e-4, key


def test_piecewise_calls_between_steps_do_not_disturb_the_fit(pb, fx):
    """run_steps(a); <piecewise entry points, same and different K>; run_steps(b) == run_steps(a + b): the piecewise
    calls overwrite (or re-create) the step's work buffers, so the next step must redo its own reparameterisation."""
    K, a, b = 6, 7, 9
    noise = np.random.default_rng(3).normal(size=(a + b, K, fx.n - 1)).astype(np.float32)

    def make():
        h = pb.Handle(num_mc_samples=K, num_steps=a + b, noise_mode=1)
        h.set_sample(_sample(pb, fx))
        h.set_tree(fx.parent_idxs, fx.js)
        h.set_noise(noise, a + b)
        h.init_params()
        return h

    h = make()
    h.run_steps(a + b)
    h.sync()
    want = h.get_params()
    h.close()
    rng = np.random.default_rng(4)
    for Kp in (K, 3, 1):
        h = make()
        h.run_steps(a)
        h.sync()
        ys = rng.uniform(0.2, 0.8, size=(Kp, fx.n - 1))
        xs, _ = h.ptt_transform(ys)
        h.loglik_grad(xs, gradonly=False)
        h.ptt_transform_gradients(ys, rng.normal(size=(Kp, fx.n)))
        h.run_steps(b)
        h.sync()
        got = h.get_params()
        h.close()
        for w, g in zip(want, got):
            assert np.array_equal(w, g), Kp


def test_set_sample_in_one_call_equals_the_three_calls(pb, fx, small_synth):
    """polee_set_sample (matrix + efflens + tree; the host tree preparation on a second thread beside the upload) leaves
    the handle in the state polee_set_matrix_csc + polee_set_efflens + polee_set_tree do: identical fits; a bad tree is
    reported with the reference's message class and leaves the handle usable."""
    import polee_b200._lib as L
    cases = [(_sample(pb, fx), (fx.parent_idxs, fx.js)), (_synth_sample(pb, small_synth), small_synth["tree"])]
    for sample, tree in cases:
        outs = []
        for one_call in (False, True):
            h = pb.Handle(num_mc_samples=6, num_steps=12, seed=99)
            if one_call:
                h.set_sample(sample, None, tree)
            else:
                h.set_sample(sample)
                h.set_tree(*tree)
            outs.append(h.fit())
            if one_call:          # the same handle again, the other way round: state is replaced cleanly
                h.set_sample(sample, None, tree)
                again = h.fit()
                for k in ("mu", "omega", "alpha"):
                    assert np.array_equal(again[k], outs[-1][k])
            h.close()
        for k in ("mu", "omega", "alpha"):
            assert np.array_equal(outs[0][k], outs[1][k]), k
    h = pb.Handle(num_mc_samples=2, num_steps=3)
    bad = fx.parent_idxs.copy()
    bad[5] = 600                                       # parent index after the child
    with pytest.raises(pb.PoleeError) as e:
        h.set_sample(_sample(pb, fx), None, (bad, fx.js))
    assert e.value.code == L.POLEE_EBADTREE
    h.set_sample(_sample(pb, fx), None, (fx.parent_idxs, fx.js))
    assert np.all(np.isfinite(h.fit()["mu"]))
    h.close()
    out = pb.approximate_likelihood(pb.LogitSkewNormalPTTApprox(), _sample(pb, fx),
                                    tree_topology=(fx.parent_idxs, fx.js), num_steps=5)
    assert np.all(np.isfinite(out["mu"]))


def test_progress_callback_and_random_treemethod(pb, fx):
    """polee_set_progress reports finished steps (the reference's "Optimizing" bar, l-a.jl:495,574); treemethod
    "random" (rand_tree_nodes, src/hclust.jl:439-454) builds a seeded random tree and returns its topology."""
    seen = []
    h = pb.Handle(num_mc_samples=6, num_steps=60)
    h.set_sample(_sample(pb, fx))
    h.set_tree(fx.parent_idxs, fx.js)
    h.set_progress(lambda done, total: seen.append((done, total)), every=25)
    h.fit()
    assert seen == [(25, 60), (50, 60), (60, 60)]
    h.set_progress(None)
    h.close()
    a = pb.approximate_likelihood(pb.LogitSkewNormalPTTApprox("random"), _sample(pb, fx), num_steps=20, seed=5)
    b = pb.approximate_likelihood(pb.LogitSkewNormalPTTApprox("random"), _sample(pb, fx), num_steps=20, seed=5)
    assert a["node_parent_idxs"].shape == (2 * fx.n - 1,) and np.array_equal(np.sort(a["node_js"][a["node_js"] > 0]), np.arange(1, fx.n + 1))
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert all(np.all(np.isfinite(a[k])) for k in ("mu", "omega", "alpha"))
    with pytest.raises(ValueError):
        pb.approximate_likelihood(pb.LogitSkewNormalPTTApprox("nonsense"), _sample(pb, fx), num_steps=2)


def test_default_fit_reproduces_reference_prep_file(pb, fx, oracle):
    """Device Philox noise, default options: lands where the reference's own prep.h5 does (SURVEY 8c tolerance)."""
    from conftest import sample_loglik
    fit = pb.approximate_likelihood(pb.LogitSkewNormalPTTApprox(), _sample(pb, fx), tree_topology=(fx.parent_idxs, fx.js))
    lp_ref, xm_ref = sample_loglik(oracle, fx, fx.mu, fx.omega, fx.alpha, ndraws=300, seed=0)
    lp_new, xm_new = sample_loglik(oracle, fx, fit["mu"], fit["omega"], fit["alpha"], ndraws=300, seed=0)
    assert abs(lp_new - lp_ref) < 30.0 and abs(lp_new - (-327172.0)) < 45.0
    big = xm_ref > 1e-3
    assert np.corrcoef(np.log(xm_new[big]), np.log(xm_ref[big]))[0, 1] > 0.985
    assert np.median(np.abs(xm_new[big] - xm_ref[big]) / xm_ref[big]) < 0.05
    assert np.corrcoef(fit["mu"], fx.mu)[0, 1] > 0.995
    # same seed -> bit-identical result (deterministic path: no atomics, fixed reduction trees)
    fit2 = pb.approximate_likelihood(pb.LogitSkewNormalPTTApprox(), _sample(pb, fx), tree_topology=(fx.parent_idxs, fx.js))
    assert all(np.array_equal(fit[k], fit2[k]) for k in ("mu", "omega", "alpha"))


def test_sequential_treemethod_and_output_topology(pb, fx):
    out = pb.approximate_likelihood(pb.LogitSkewNormalPTTApprox("sequential"), _sample(pb, fx), num_steps=30)
    from polee_b200.api import sequential_tree
    pi, js = sequential_tree(fx.n)
    assert np.array_equal(out["node_parent_idxs"], pi) and np.array_equal(out["node_js"], js)   # l-a.jl:618-621
    assert all(np.all(np.isfinite(out[k])) for k in ("mu", "omega", "alpha"))
    # treemethod "cluster" (the reference's default, l-a.jl:435): the tree comes from the hclust restatement and is
    # returned with the parameters; the fit on it is as good as on the reference's own tree for this matrix
    clu = pb.approximate_likelihood(pb.LogitSkewNormalPTTApprox("cluster"), _sample(pb, fx), num_steps=150)
    hp, hj = pb.hclust(_sample(pb, fx))
    assert np.array_equal(clu["node_parent_idxs"], hp) and np.array_equal(clu["node_js"], hj)
    assert all(np.all(np.isfinite(clu[k])) for k in ("mu", "omega", "alpha"))


@pytest.mark.parametrize("exact", [True, False])
def test_optimize_ptt(pb, fx, oracle, exact):
    """approximate_likelihood(::OptimizePTTApprox): point estimate on the :sequential tree.  A depth-312 chain
    amplifies last-bit differences of the gradient over the ADAM steps, so the comparison is on the objective
    reached and, loosely, on the abundant transcripts."""
    steps = 60
    xo = oracle.fit_optimize_ptt(fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval, fx.efflens, steps)
    h = pb.Handle(approx=1, num_steps=steps, exact_accumulation=exact)
    h.set_sample(_sample(pb, fx))
    x_dev = h.fit_optimize_ptt()
    h.close()
    assert abs(x_dev.astype(np.float64).sum() - 1.0) < 1e-4
    M = oracle.Model(fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval)
    lp_d, _ = M.log_likelihood(x_dev, gradonly=False)
    lp_o, _ = M.log_likelihood(xo, gradonly=False)
    assert abs(lp_d - lp_o) <= 1e-4 * abs(lp_o)
    big = xo > 1e-4
    assert np.median(np.abs(x_dev[big] - xo[big]) / xo[big]) < (1e-3 if exact else 1e-2)


@pytest.mark.parametrize("exact", [0, 1])
def test_optimize_ptt_first_steps_tight(pb, fx, oracle, exact):
    """OptimizePTTApprox step by step (l-a.jl:149-242): after 1, 2 and 3 ADAM steps the device's x equals the oracle's
    elementwise -- before the depth-312 chain has had time to amplify last-bit differences of the gradient."""
    for steps in (1, 2, 3):
        xo = oracle.fit_optimize_ptt(fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval, fx.efflens, steps)
        h = pb.Handle(approx=1, num_steps=steps, exact_accumulation=exact)
        h.set_sample(_sample(pb, fx))
        x_dev = h.fit_optimize_ptt()
        h.close()
        err = np.abs(x_dev.astype(np.float64) - xo) / np.maximum(xo, 1e-30)
        # the first ADAM step moves every coordinate by ~ +-lr g / (|g| + 1e-8): coordinates whose gradient is ~ 0 are
        # sensitive to its last bits, hence a looser bound on the maximum than on the bulk
        assert np.median(err) <= 1e-6 and err.max() <= 2e-4, (steps, np.median(err), err.max())


def test_synthetic_sample_all_paths(pb, small_synth, oracle):
    s = small_synth
    K = 8
    sample = _synth_sample(pb, s)
    pi, js = s["tree"]
    rng = np.random.default_rng(9)
    xs = rng.dirichlet(np.ones(s["n"]), K).astype(np.float32).clip(1e-10)
    h = pb.Handle(num_mc_samples=K, noise_mode=1, num_steps=25, gradonly=False)
    h.set_sample(sample)
    h.set_tree(pi, js)
    lp, g = h.loglik_grad(xs, gradonly=False)
    M = oracle.Model(s["m"], s["n"], s["colptr"], s["rowval"], s["nzval"])
    for k in (0, K - 1):
        lp_o, g_o = M.log_likelihood(xs[k], gradonly=False)
        assert abs(lp[k] - lp_o) <= 1e-8 * abs(lp_o) and relerr(g[k], g_o) <= 1e-5
    noise = rng.normal(size=(25, K, s["n"] - 1)).astype(np.float32)
    dev = h.fit(noise=noise, want_elbo=True)
    ora = oracle.fit_lsn_ptt(s["m"], s["n"], s["colptr"], s["rowval"], s["nzval"], s["efflens"], pi, js, num_steps=25,
                             num_mc_samples=K, noise=noise, gradonly=False, elbo_fix=True)
    for key in ("mu", "omega", "alpha"):
        assert np.abs(dev[key] - ora[key]).max() <= 2e-4, key
    assert relerr(dev["elbo"], ora["elbo"]) <= 1e-6
    h.close()


def test_long_rows_and_empty_columns(pb, oracle):
    """Config-4-shaped rows (up to 512 entries), columns spanning many K2 segments, empty columns."""
    from polee_b200 import synth
    s = synth.to_numpy_sample(synth.make_sample(6000, 3000, seed=5, long_rows=True))
    s["n"] += 7                                                   # trailing empty columns (fixture: 29 of 313 empty)
    s["colptr"] = np.concatenate([s["colptr"], np.full(7, s["colptr"][-1], np.uint32)])
    s["efflens"] = np.concatenate([s["efflens"], np.full(7, 1000, np.float32)])
    rows = np.bincount(s["rowval"] - 1, minlength=s["m"])
    cols = np.diff(s["colptr"].astype(np.int64))
    assert rows.max() > 256 and cols.max() > 256 and (cols == 0).any()
    sample = _synth_sample(pb, s)
    xs = np.random.default_rng(1).dirichlet(np.ones(s["n"]), 2).astype(np.float32).clip(1e-10)
    lp, g = pb.log_likelihood(sample, xs, gradonly=False)
    M = oracle.Model(s["m"], s["n"], s["colptr"], s["rowval"], s["nzval"])
    for k in range(2):
        lp_o, g_o = M.log_likelihood(xs[k], gradonly=False)
        assert abs(lp[k] - lp_o) <= 1e-8 * abs(lp_o)
        assert np.array_equal(g[k] == 0, g_o == 0)               # empty columns give exactly 0
        nz = g_o != 0
        assert relerr(g[k][nz], g_o[nz]) <= 1e-5


def test_non_finite_gradient_is_reported(pb, fx):
    """likelihood-approximation.jl:559 `@assert all_finite` -> POLEE_ENONFINITE with the failing step."""
    import polee_b200._lib as L
    bad = fx.nzval.copy()
    bad[0] = np.nan
    h = pb.Handle(num_mc_samples=2, num_steps=3)
    h.set_sample(pb.RNASeqSample(fx.m, fx.n, fx.colptr, fx.rowval, bad, fx.efflens))
    h.set_tree(fx.parent_idxs, fx.js)
    with pytest.raises(pb.PoleeError) as e:
        h.fit()
    assert e.value.code == L.POLEE_ENONFINITE and "step 1" in str(e.value)
    h.close()


def test_approx_likelihood_sampler(pb, fx, oracle):
    """Random.rand!(::ApproxLikelihoodSampler, xs) (src/approx-sampler.jl:37-44) on the device: draws from the
    reference's own fitted approximation (prep.h5) reproduce the survey's probe statistics (mean log-likelihood of
    draws -327172 +- 30) and every draw is a point of the simplex."""
    als = pb.ApproxLikelihoodSampler(draws_per_launch=16)
    als.set_transform((fx.parent_idxs, fx.js), fx.mu, np.exp(fx.omega), fx.alpha)
    xs = als.rand(400, seed=1)
    assert xs.shape == (400, fx.n) and np.all(xs > 0)
    np.testing.assert_allclose(xs.astype(np.float64).sum(1), 1.0, atol=2e-5)
    M = oracle.Model(fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval)
    lps = [M.log_likelihood(np.maximum(x, np.float32(1e-10)), gradonly=False)[0] for x in xs[:300]]
    assert abs(np.mean(lps) - (-327172.0)) < 30.0
    xs2 = als.rand(400, seed=1)
    assert np.array_equal(xs, xs2)                       # counter-based noise: same seed, same draws
    assert not np.array_equal(xs[:16], xs[16:32])         # batches use different Philox counters
    # moments agree with the CPU restatement of rand! (conftest.sample_loglik) on the abundant transcripts
    from conftest import sample_loglik
    _, xm = sample_loglik(oracle, fx, fx.mu, fx.omega, fx.alpha, ndraws=400, seed=3)
    big = xm > 1e-3
    assert np.median(np.abs(xs.mean(0)[big] - xm[big]) / xm[big]) < 0.05


def test_large_sequential_tree_scan_path(pb, oracle):
    """Caterpillar trees with >= 4096 nodes take the blocked-scan kernels (tree_chain.cu).  They re-associate the
    Float64 products and carry the backward recurrences in Float64, so the comparison with the serial reference
    sweep is to rounding error: x <= 1e-12 relative, y_grad <= 2e-5 of its scale (the reference itself rounds G to
    Float32 at every one of the n-1 spine nodes)."""
    from polee_b200.api import sequential_tree
    n, K = 6000, 3
    pi, js = sequential_tree(n)
    rng = np.random.default_rng(2)
    # ys of a near-uniform composition (what the fit starts from): u_k stays O(1/n), no underflow
    x0 = rng.dirichlet(np.ones(n) * 5.0, K).astype(np.float32)
    to = oracle.PTT(pi, js)
    ys = np.stack([to.inverse_transform(x0[k])[0] for k in range(K)])
    t = pb.PolyaTreeTransform(pi, js)
    xs, ladj = t.transform(ys, compute_ladj=True)
    assert t.handle.layout_info()["tree_route"] == "chain"
    # with the trees of test_tree_forward_backward_bit_exact, every route is taken
    assert set(_TREE_ROUTES.values()) | {"chain"} == {"chain", "dfs", "path", "levels_smem", "levels_global"}
    x_grad = rng.normal(size=(K, n)) * 100
    yg = t.transform_gradients(ys, x_grad)
    yg0 = t.transform_gradients_no_ladj(ys, x_grad)
    for k in range(K):
        xo, ladj_o = to.transform(ys[k], True)
        assert relerr(xs[k], xo) <= 2e-7                  # Float32 output of a Float64 product differing by ~1e-16
        assert abs(ladj[k] - ladj_o) <= 1e-10 * abs(ladj_o)
        ygo = to.transform_gradients(ys[k], x_grad[k])
        assert np.abs(yg[k] - ygo).max() <= 2e-5 * np.abs(ygo).max()
        ygo0 = to.transform_gradients_no_ladj(ys[k], x_grad[k])
        assert np.abs(yg0[k] - ygo0).max() <= 2e-5 * np.abs(ygo0).max()


def test_optimize_ptt_large_sequential(pb, small_synth, oracle):
    """optimize_likelihood on n = 1500 takes the level-synchronous path, on a padded n >= 2048 the scan path; both
    must reach the oracle's objective."""
    s = small_synth
    sample = _synth_sample(pb, s)
    steps = 40
    xo = oracle.fit_optimize_ptt(s["m"], s["n"], s["colptr"], s["rowval"], s["nzval"], s["efflens"], steps)
    M = oracle.Model(s["m"], s["n"], s["colptr"], s["rowval"], s["nzval"])
    lp_o, _ = M.log_likelihood(xo, gradonly=False)
    for env in ("1000000000", "1"):                      # force level-synchronous / force scan kernels
        import os
        os.environ["POLEE_CHAIN_MIN_NODES"] = env
        h = pb.Handle(approx=1, num_steps=steps)
        h.set_sample(sample)
        x_dev = h.fit_optimize_ptt()
        h.close()
        lp_d, _ = M.log_likelihood(x_dev, gradonly=False)
        assert abs(lp_d - lp_o) <= 2e-4 * abs(lp_o), env
        assert abs(x_dev.astype(np.float64).sum() - 1.0) < 1e-4
    os.environ.pop("POLEE_CHAIN_MIN_NODES")


def _gene_groups(n, seed=3):
    """synthetic gene -> transcripts map: contiguous genes of 1..6 transcripts, a few transcripts in no gene"""
    rng = np.random.default_rng(seed)
    groups, i = {}, 1
    while i <= n:
        k = int(rng.integers(1, 7))
        ids = list(range(i, min(i + k, n + 1)))
        if rng.random() > 0.1:                       # ~10 % of the transcripts have no gene_id (l-a.jl:480)
            groups["gene%d" % len(groups)] = ids
        i += k
    return groups


@pytest.mark.gpu
@pytest.mark.parametrize("K", [6, 8])
def test_gene_noninformative_prior(pb, fx, oracle, K):
    """gene_noninformative_prior! (likelihood.jl:114-159) inside one step of draws and inside a fit."""
    genes = _gene_groups(fx.n)
    rng = np.random.default_rng(20 + K)
    h = pb.Handle(num_mc_samples=K, noise_mode=1, num_steps=2)
    h.set_sample(_sample(pb, fx))
    h.set_tree(fx.parent_idxs, fx.js)
    mu, om, al = h.get_params()
    al = (rng.normal(size=fx.n - 1) * 0.1).astype(np.float32)
    h.set_params(mu, om, al)
    zs0 = rng.normal(size=(K, fx.n - 1)).astype(np.float32)
    base = h.lsn_draws(zs0)
    h.set_gene_groups(genes)
    d = h.lsn_draws(zs0)
    acc = {k: np.zeros(fx.n - 1, np.float32) for k in ("mu_grad", "omega_grad", "alpha_grad")}
    for k in range(K):
        o = oracle.lsn_draw(fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval, fx.efflens, fx.parent_idxs, fx.js, mu, om, al,
                            zs0[k], gene_transcripts=genes)
        o0 = oracle.lsn_draw(fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval, fx.efflens, fx.parent_idxs, fx.js, mu, om, al,
                             zs0[k])
        prior = o["x_grad"] - o0["x_grad"]                     # the prior's own contribution
        assert np.abs(prior).max() > 0
        got = d["x_grad"][k] - base["x_grad"][k]
        assert np.abs(got - prior).max() <= 1e-5 * np.abs(prior).max() + 1e-9 * np.abs(o["x_grad"]).max()
        assert np.abs(d["x_grad"][k] - o["x_grad"]).max() <= 1e-5 * np.abs(o["x_grad"]).max()
        for key in acc:
            acc[key] += o[key]
    for key in acc:
        ref = acc[key] / np.float32(K)
        assert np.abs(d[key] - ref).max() <= 1e-5 * np.abs(ref).max(), key
    h.set_gene_groups(None)                                    # cleared -> back to the plain gradient, bit for bit
    again = h.lsn_draws(zs0)
    assert np.array_equal(again["x_grad"], base["x_grad"])
    # error behaviour: the prior needs the effective-length adjustment; a transcript may sit in one gene only
    with pytest.raises(pb.PoleeError):
        h.set_gene_groups([[1, 2], [2, 3]])
    with pytest.raises(pb.PoleeError):
        h.set_gene_groups([[0, 1]])
    h.close()
    h2 = pb.Handle(num_mc_samples=K, use_efflen_jacobian=False, num_steps=2)
    h2.set_sample(_sample(pb, fx))
    h2.set_tree(fx.parent_idxs, fx.js)
    h2.set_gene_groups(genes)
    with pytest.raises(pb.PoleeError):
        h2.run_steps(1)
    h2.close()
    # the fit: same noise, prior on -> tracks the oracle, and differs from the fit without the prior
    steps = 40
    noise = np.random.default_rng(K).normal(size=(steps, K, fx.n - 1)).astype(np.float32)
    ora = oracle.fit_lsn_ptt(fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval, fx.efflens, fx.parent_idxs, fx.js,
                             num_steps=steps, num_mc_samples=K, noise=noise, gene_transcripts=genes)
    kw = dict(tree_topology=(fx.parent_idxs, fx.js), num_steps=steps, num_mc_samples=K, noise=noise)
    dev = pb.approximate_likelihood(pb.LogitSkewNormalPTTApprox(), _sample(pb, fx), gene_noninformative=True,
                                    gene_transcripts=genes, **kw)
    plain = pb.approximate_likelihood(pb.LogitSkewNormalPTTApprox(), _sample(pb, fx), **kw)
    for key in ("mu", "omega", "alpha"):
        assert np.abs(dev[key] - ora[key]).max() <= 2e-4, key
    assert np.abs(dev["mu"] - plain["mu"]).max() > 1e-3
    with pytest.warns(UserWarning):                            # l-a.jl:489-492: flag dropped without gene information
        same = pb.approximate_likelihood(pb.LogitSkewNormalPTTApprox(), _sample(pb, fx), gene_noninformative=True, **kw)
    assert np.array_equal(same["mu"], plain["mu"])


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 6, 8])
def test_split_and_fused_layouts_agree(pb, fx, small_synth, oracle, K, monkeypatch):
    """The two device layouts of the matrix (SELL + CSC pair vs. fused row tiles, matrix_setup.cu) are two
    implementations of the same pAt_mul_B! / pAt_mulinv_B! pair (sparse.jl:6-40): each within 1e-5 of the oracle,
    within 1e-6 of each other, each run-to-run identical; also with row counts (likelihood.jl:59-85) and for the
    row-wise 1/p output."""
    rng = np.random.default_rng(40 + K)
    for (m, n, colptr, rowval, nzval, eff, tree) in (
            (fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval, fx.efflens, (fx.parent_idxs, fx.js)),
            (small_synth["m"], small_synth["n"], small_synth["colptr"], small_synth["rowval"], small_synth["nzval"],
             small_synth["efflens"], small_synth["tree"])):
        sample = pb.RNASeqSample(m, n, colptr, rowval, nzval, eff)
        xs = rng.dirichlet(np.ones(n), K).astype(np.float32).clip(1e-10)
        ks = rng.integers(1, 5, size=m).astype(np.int64)
        M = oracle.Model(m, n, colptr, rowval, nzval)
        out = {}
        for layout in ("split", "fused"):
            monkeypatch.setenv("POLEE_LAYOUT", layout)
            h = pb.Handle(num_mc_samples=K, gradonly=False)
            h.set_sample(sample)
            h.set_tree(*tree)
            lp, g = h.loglik_grad(xs, gradonly=False)
            lp2, g2 = h.loglik_grad(xs, gradonly=False)
            assert np.array_equal(g, g2) and np.array_equal(lp, lp2)          # deterministic
            w = np.zeros(m, np.float32)
            h.check(h.lib.polee_frag_prob_recip(h.h, xs[0].ctypes.data_as(pb.api._P), w.ctypes.data_as(pb.api._P)))
            h.close()
            hk = pb.Handle(num_mc_samples=K, gradonly=False)
            hk.set_sample(sample, ks)
            hk.set_tree(*tree)
            lpk, gk = hk.loglik_grad(xs, gradonly=False)
            hk.close()
            out[layout] = (lp, g, w, lpk, gk)
            for k in (0, K - 1):
                lp_o, g_o = M.log_likelihood(xs[k], gradonly=False)
                assert abs(lp[k] - lp_o) <= 1e-8 * abs(lp_o) and relerr(g[k], g_o) <= 1e-5, layout
                lpk_o, gk_o = M.log_likelihood(xs[k], gradonly=False, ks=ks)
                assert abs(lpk[k] - lpk_o) <= 1e-8 * abs(lpk_o) and relerr(gk[k], gk_o) <= 1e-5, layout
        a, b = out["split"], out["fused"]
        assert relerr(a[1], b[1]) <= 1e-6 and relerr(a[0], b[0]) <= 1e-9      # rows > 4 entries: Float32 vs Float64 row sums
        assert relerr(a[2], b[2]) <= 5e-7                                       # 1/p per row, original row order
        assert relerr(a[4], b[4]) <= 1e-6


@pytest.mark.gpu
def test_exact_factorization_on_device(pb, fx, small_synth, oracle):
    """polee_exact_factorization vs the restated tools/exact-factorization.jl: identical unique rows, counts and CSC
    arrays (bit for bit; rows numbered by first occurrence), and the factored likelihood of the compressed sample
    equals the plain likelihood of the original."""
    rng = np.random.default_rng(77)
    # the fixture as is (2 % duplicates), and a synthetic sample with every row repeated 1-4 times
    s = small_synth
    X = []
    import scipy.sparse as sp
    A = sp.csc_matrix((s["nzval"], s["rowval"].astype(np.int64) - 1, s["colptr"].astype(np.int64) - 1),
                      shape=(s["m"], s["n"])).tocsr()
    reps = rng.integers(1, 5, size=2000)
    rows = np.repeat(rng.integers(0, s["m"], size=2000), reps)
    rng.shuffle(rows)
    B = A[rows].tocsc()
    B.sort_indices()
    dup = (B.shape[0], B.shape[1], (B.indptr + 1).astype(np.uint32), (B.indices + 1).astype(np.uint32),
           B.data.astype(np.float32), s["efflens"])
    for (m, n, colptr, rowval, nzval, eff) in ((fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval, fx.efflens), dup):
        sample = pb.RNASeqSample(m, n, colptr, rowval, nzval, eff)
        comp, counts = pb.exact_factorization(sample)
        mu, cp, rv, nz, cnt = oracle.exact_factorization(m, n, colptr, rowval, nzval)
        assert comp.m == mu and counts.sum() == m
        assert np.array_equal(counts, cnt) and np.array_equal(comp.colptr, cp)
        assert np.array_equal(comp.rowval, rv) and np.array_equal(comp.nzval.view(np.uint32), nz.view(np.uint32))
        xs = rng.dirichlet(np.ones(n), 2).astype(np.float32).clip(1e-10)
        tree = pb.sequential_tree(n) if hasattr(pb, "sequential_tree") else pb.api.sequential_tree(n)
        h0 = pb.Handle(num_mc_samples=2, gradonly=False)
        h0.set_sample(sample); h0.set_tree(*tree)
        lp0, g0 = h0.loglik_grad(xs, gradonly=False)
        h0.close()
        h1 = pb.Handle(num_mc_samples=2, gradonly=False)
        h1.set_sample(comp, counts); h1.set_tree(*tree)
        lp1, g1 = h1.loglik_grad(xs, gradonly=False)
        h1.close()
        assert relerr(lp1, lp0) <= 1e-10 and relerr(g1, g0) <= 1e-6
    assert dup[0] > 2 * comp.m * 0.9                                  # the synthetic case really was ~2.5x redundant
