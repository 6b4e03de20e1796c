"""The step loop's launch mechanics change how kernels overlap, never what they compute.

* Programmatic dependent launch (POLEE_PDL, read when a handle is created): a fit with it on is bit-identical to one with
  it off, and the captured step graphs carry programmatic edges exactly when it is on.  Each setting runs in its own
  process.
* The multi-step graph of polee_run_steps: any step count gives the bits of the same steps enqueued without a graph,
  and a progress callback sees the calls it saw with one graph launch per step."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIT_STEPS = 30


def _fixture_sample(pb):
    from conftest import Fixture
    fx = Fixture()
    return pb.RNASeqSample(fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval, fx.efflens), (fx.parent_idxs, fx.js)


def _synth_sample(pb):
    """~1 M rows x 20 000 transcripts (generated on the device, seeded) and a balanced-by-gene tree"""
    from polee_b200 import synth
    s = synth.make_sample(1 << 20, 20_000, seed=20260002, device="cuda:0")
    tree = synth.balanced_tree(20_000, s["gene_sizes"].cpu().numpy())
    ns = synth.to_numpy_sample(s)
    return pb.RNASeqSample(ns["m"], ns["n"], ns["colptr"], ns["rowval"], ns["nzval"], ns["efflens"]), tree


def _fit(pb, sample, tree, steps, use_cuda_graph=True):
    h = pb.Handle(num_mc_samples=6, num_steps=steps, gradonly=False, use_cuda_graph=use_cuda_graph)
    h.set_sample(sample, tree_topology=tree)
    out = h.fit(want_elbo=True)
    out["edges"] = np.array([h.layout_info()[k] for k in ("graph_programmatic_edges",
                                                          "multi_step_graph_programmatic_edges")])
    h.close()
    return out


def _fit_in_child(which, pdl, tmp_path):
    """a FIT_STEPS-step fit in a fresh process with POLEE_PDL=pdl"""
    out = os.path.join(str(tmp_path), "%s_pdl%d.npz" % (which, pdl))
    env = dict(os.environ, POLEE_PDL=str(pdl))
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), which, out]
    r = subprocess.run(cmd, env=env, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout
    return dict(np.load(out))


@pytest.mark.parametrize("which", ["fixture", "synth_1m"])
def test_pdl_fit_bit_identical(which, tmp_path):
    on, off = _fit_in_child(which, 1, tmp_path), _fit_in_child(which, 0, tmp_path)
    for key in ("mu", "omega", "alpha", "elbo"):
        assert np.array_equal(on[key], off[key]), key
    assert np.all(np.isfinite(on["elbo"])) and np.any(on["elbo"] != 0.0)
    one, multi = on["edges"]
    assert one > 0 and multi >= 8 * one, on["edges"]
    if which == "synth_1m":   # DFS-run forward: the step boundary k3_elem -> k3d_tree_fwd is programmatic as well
        assert multi == 8 * one + 7, on["edges"]
    assert list(off["edges"]) == [0, 0]


@pytest.fixture(scope="module")
def fixture_sample():
    import polee_b200 as pb
    return (pb,) + _fixture_sample(pb)


@pytest.mark.parametrize("steps", [1, 7, 8, 9, 17, 500])
def test_multi_step_graph_bit_identical(fixture_sample, steps):
    pb, sample, tree = fixture_sample
    graph, plain = _fit(pb, sample, tree, steps), _fit(pb, sample, tree, steps, use_cuda_graph=False)
    for key in ("mu", "omega", "alpha", "elbo"):
        assert np.array_equal(graph[key], plain[key]), key
    assert list(plain["edges"]) == [-1, -1]
    if steps >= 3 + 8:   # three single steps (uncaptured, captured, replayed), then whole chunks of 8
        assert graph["edges"][1] >= 0


def _refits(pb, sample, tree, use_cuda_graph):
    """on ONE handle: two whole fits, then a warm start from the first fit's parameters after polee_sample, each long
    enough (20 steps) that the multi-step graph captured by the first fit replays in the later ones"""
    steps = 20
    h = pb.Handle(num_mc_samples=6, num_steps=steps, gradonly=False, use_cuda_graph=use_cuda_graph)
    h.set_sample(sample, tree_topology=tree)
    first = h.fit(want_elbo=True)
    second = h.fit(want_elbo=True)
    h.sample(4, seed=5)   # leaves its own draws in the step buffers
    h.set_params(first["mu"], first["omega"], first["alpha"])
    h.run_steps(steps)
    h.sync()
    warm = dict(zip(("mu", "omega", "alpha"), h.get_params()))
    h.close()
    return first, second, warm


def test_refit_on_one_handle_bit_identical(fixture_sample):
    """init_params / set_params / polee_sample leave the next step's draws to be made again; the multi-step graph must
    not step on the stale ones"""
    pb, sample, tree = fixture_sample
    graph, plain = _refits(pb, sample, tree, True), _refits(pb, sample, tree, False)
    for g, p in zip(graph, plain):
        for key in p:
            assert np.array_equal(g[key], p[key]), key
    for key in ("mu", "omega", "alpha", "elbo"):   # init_params starts the same fit over
        assert np.array_equal(graph[0][key], graph[1][key]), key
    assert not np.array_equal(graph[2]["mu"], graph[0]["mu"])


@pytest.mark.parametrize("every", [3, 8])
def test_progress_callback_sequence(fixture_sample, every):
    pb, sample, tree = fixture_sample
    steps = 29
    seen = []
    h = pb.Handle(num_mc_samples=6, num_steps=steps, gradonly=False)
    h.set_sample(sample, tree_topology=tree)
    h.set_progress(lambda done, total: seen.append((done, total)), every=every)
    h.init_params()
    h.run_steps(steps)
    h.sync()
    params = h.get_params()
    h.close()
    assert seen == [(s, steps) for s in range(1, steps + 1) if s % every == 0 or s == steps]
    plain = _fit(pb, sample, tree, steps, use_cuda_graph=False)
    for key, v in zip(("mu", "omega", "alpha"), params):
        assert np.array_equal(v, plain[key]), key


if __name__ == "__main__":
    # child of test_pdl_fit_bit_identical: <fixture | synth_1m> <out.npz>
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import polee_b200 as pb
    sample, tree = (_fixture_sample if sys.argv[1] == "fixture" else _synth_sample)(pb)
    res = _fit(pb, sample, tree, FIT_STEPS)
    np.savez(sys.argv[2], **{k: res[k] for k in ("mu", "omega", "alpha", "elbo", "edges")})
