"""A whole logit-skew-normal step, and short fits, on every kernel route of the tree at every padded draw width,
against the oracle.

tree_route (tree_kernels.cu) serves a tree with one of five kernel sets -- chain, dfs, path, levels_smem,
levels_global -- chosen from the tree's shape and from KP, the draw count padded to 1, 2, 4, 8 or 16.  Each route's
forward writes its own rows of the S and log-Jacobian partial sums and each backward applies the effective-length
Jacobian its own way, so each (route, KP) pair is a separate piece of code for the step.  CATALOGUE names one tree
and one K per pair, the padded K = 3, 5, 6 and 12 included, plus trees whose route changes with KP.

The CPU test restates the route rules on the host schedule (tree_host.cu) and checks that the catalogue reaches every
pair; the GPU tests check that the device takes the predicted route and computes what the oracle computes."""
import collections
import os
import subprocess
import sys

import numpy as np
import pytest

gpu = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if __name__ == "__main__":          # a child of test_pdl_fit_bit_identical: the package and conftest from the tree
    sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
M_ROWS = 20_000
ROUTES = ("chain", "dfs", "path", "levels_smem", "levels_global")
KPS = (1, 2, 4, 8, 16)
NO_CHAIN = str(10 ** 9)            # POLEE_CHAIN_MIN_NODES: a caterpillar of any size keeps the level kernels

# the device constants the route rules read (common.cuh, api.cu, tree_kernels.cu)
ROUTE_SMEM_LIMIT = 200 * 1024      # what tree_route allows any route's kernels
MAX_SMEM_PER_CTA = 227 * 1024      # the sm_100 opt-in limit of a CTA's shared memory
TREE_BIN_NODES = 512
DFS_MAX_DEPTH, DFS_RUN, DFS_RUNS_PER_CTA = 96, 64, 16
PATH_GROUP, PATH_MAX_GANC, PATH_MAX_SUFFIX, PATH_MAX_ENTRIES = 128, 1024, 16384, 64 << 20
CHAIN_MIN_NODES = 4096
SNODE_BYTES, DNODE_BYTES = 16, 8


# ------------------------------------------------------------------------------------------------ trees
def _children(pi):
    """0-based right / left child of every node: the first child seen is the right one (src/ptt.jl:104-110)"""
    N = len(pi)
    right, left = np.full(N, -1, np.int64), np.full(N, -1, np.int64)
    for i in range(1, N):
        p = pi[i] - 1
        if right[p] < 0:
            right[p] = i
        else:
            left[p] = i
    return right, left


def children_first(pi, js):
    """The same tree with a node's two children numbered together when the node is reached (then the right child's
    subtree, then the left child's).  Parents still come before children, but the order is not DFS pre-order, so
    tree_host builds root-path tables for it instead of the DFS-run inputs."""
    N = len(pi)
    right, left = _children(pi)
    new = np.zeros(N, np.int64)
    order, stack = [0], [0]
    while stack:
        v = stack.pop()
        if js[v] == 0:
            new[right[v]], new[left[v]] = len(order), len(order) + 1
            order += [right[v], left[v]]
            stack += [left[v], right[v]]
    pi2, js2 = np.zeros(N, np.int32), np.zeros(N, np.int32)
    for v in range(N):
        js2[new[v]] = js[v]
        if v:
            pi2[new[v]] = new[np.int64(pi[v]) - 1] + 1
    return pi2, js2


def deep_preorder_tree(n_spine=88, sub_leaves=16):
    """A spine of n_spine nodes with a balanced sub_leaves-leaf subtree off each one, in DFS pre-order: depth 93, so
    k3d_tree_fwd's stacks fit the 200 KB up to KP = 8 and not at KP = 16"""
    from polee_b200 import synth

    def bal(items):
        while len(items) > 1:
            items = [(items[i], items[i + 1]) for i in range(0, len(items) - 1, 2)] + \
                    ([items[-1]] if len(items) % 2 else [])
        return items[0]

    j, subs = 1, []
    for _ in range(n_spine):
        subs.append(bal(list(range(j, j + sub_leaves))))
        j += sub_leaves
    node = j
    for s in reversed(subs):
        node = (node, s)                      # tree_from_nested emits the right (second) element first
    return synth.tree_from_nested(node, j)


def _fixture_tree():
    from conftest import Fixture
    fx = Fixture()
    return fx.parent_idxs, fx.js


def _trees():
    from polee_b200 import synth
    from polee_b200.api import sequential_tree
    return {
        "fixture": _fixture_tree,
        "random_2000": lambda: synth.random_tree(2000, 5),
        "children_first_1000": lambda: children_first(*synth.random_tree(1000, 7)),
        "sequential_313": lambda: sequential_tree(313),
        "spine_1225": lambda: synth.spine_tree(1200, 100),
        "sequential_6000": lambda: sequential_tree(6000),
        "sequential_2500": lambda: sequential_tree(2500),
        "deep_preorder": deep_preorder_tree,
        "sequential_900": lambda: sequential_tree(900),
    }


TREES = _trees()
# trees that run with POLEE_CHAIN_MIN_NODES raised: a large caterpillar on the level kernels
RAISED_CHAIN_MIN = {"sequential_6000"}

Case = collections.namedtuple("Case", "tree K route")
CATALOGUE = [
    Case("fixture", 1, "dfs"), Case("random_2000", 2, "dfs"), Case("fixture", 3, "dfs"),
    Case("random_2000", 5, "dfs"), Case("fixture", 12, "dfs"), Case("random_2000", 16, "dfs"),
    Case("children_first_1000", 1, "path"), Case("sequential_313", 2, "path"), Case("children_first_1000", 3, "path"),
    Case("sequential_313", 6, "path"), Case("children_first_1000", 16, "path"),
    Case("spine_1225", 1, "levels_smem"), Case("spine_1225", 2, "levels_smem"), Case("spine_1225", 4, "levels_smem"),
    Case("spine_1225", 8, "levels_smem"), Case("spine_1225", 12, "levels_smem"),
    Case("sequential_6000", 1, "levels_global"), Case("sequential_6000", 2, "levels_global"),
    Case("sequential_6000", 3, "levels_global"), Case("sequential_6000", 5, "levels_global"),
    Case("sequential_6000", 16, "levels_global"),
    Case("sequential_2500", 1, "chain"), Case("sequential_2500", 2, "chain"), Case("sequential_2500", 4, "chain"),
    Case("sequential_2500", 6, "chain"), Case("sequential_2500", 12, "chain"),
    # the route changes with KP: DFS-run stacks of depth 93 outgrow the shared memory at KP = 16
    Case("deep_preorder", 8, "dfs"), Case("deep_preorder", 16, "levels_smem"),
    # root-path tables that need more shared memory at KP = 16 than a CTA can have
    Case("sequential_900", 6, "path"), Case("sequential_900", 16, "levels_smem"),
]


def _case_id(c):
    return "%s-K%d" % (c.tree, c.K)


def pad_k(K):
    return 1 << (K - 1).bit_length()


# ------------------------------------------------------------------------------ the route rules, restated
def tree_stats(pi, js):
    """What tree_route reads of a tree, restated from TreeHost::build_from_lrf (tree_host.cu)"""
    pi, js = np.asarray(pi, np.int64), np.asarray(js, np.int64)
    N = len(pi)
    n = (N + 1) // 2
    right, left = _children(pi)
    internal = js == 0
    kidx = np.cumsum(internal) - 1
    parent = pi - 1
    depth = np.zeros(N, np.int64)
    for i in range(1, N):
        depth[i] = depth[parent[i]] + 1
    size, sub_depth = np.ones(N, np.int64), depth.copy()    # subtree sizes, deepest node of every subtree
    for i in range(N - 1, 0, -1):
        size[parent[i]] += size[i]
        sub_depth[parent[i]] = max(sub_depth[parent[i]], sub_depth[i])
    max_depth = int(depth.max())
    st = {"n": n, "N": N, "max_depth": max_depth}
    ii = np.nonzero(internal)[0]
    preorder_nodes = n >= 2 and bool(np.all(right[ii] == ii + 1)) and bool(np.all(left[ii] == ii + 1 + size[ii + 1]))
    st["preorder"] = preorder_nodes and max_depth <= DFS_MAX_DEPTH
    cta_nodes = DFS_RUN * DFS_RUNS_PER_CTA
    st["dfs_max_nk"] = max(int(internal[c:c + cta_nodes].sum()) for c in range(0, N, cta_nodes)) if st["preorder"] else 0
    # root-path tables (only when the DFS-run inputs are not built)
    st["path_tables"], st["max_ganc"], st["max_gsuf"] = False, 0, 0
    if not st["preorder"] and n >= 2 and depth.sum() <= PATH_MAX_ENTRIES:
        def path(i):                      # root first: k of the ancestor << 1 | 1 when the path goes to its left child
            out = []
            while i > 0:
                p = parent[i]
                out.append(int(kidx[p]) << 1 | int(left[p] == i))
                i = p
            return out[::-1]

        ok, mg, ms = True, 0, 0
        for g0 in range(0, N, PATH_GROUP):
            paths = [path(i) for i in range(g0, min(N, g0 + PATH_GROUP))]
            cp = len(paths[0])
            for p in paths[1:]:
                c, lim = 0, min(cp, len(p))
                while c < lim and p[c] == paths[0][c]:
                    c += 1
                cp = c
            suffix_ks = {e >> 1 for p in paths for e in p[cp:]}
            na, ns = cp + len(suffix_ks), sum(len(p) - cp for p in paths)
            mg, ms = max(mg, na), max(ms, ns)
            if na > PATH_MAX_GANC or ns > PATH_MAX_SUFFIX:
                ok = False
                break
        if ok:
            st["path_tables"], st["max_ganc"], st["max_gsuf"] = True, mg, ms
    # caterpillar: spine node k at 2k, its right child the leaf at 2k + 1, its left child the next spine node
    cat = n >= 2 and js[N - 1] > 0
    for i in ii:
        if not cat:
            break
        cat = i % 2 == 0 and right[i] == i + 1 and left[i] == i + 2 and js[i + 1] > 0
    st["caterpillar"] = bool(cat)
    # the cut into a top part (subtrees of more than TREE_BIN_NODES nodes) and bottom bins of whole subtrees
    is_top = size > TREE_BIN_NODES
    bins, fill = [], 0                   # per bin: [nodes, levels]
    for r in range(N):
        if is_top[r] or (r > 0 and not is_top[parent[r]]):
            continue
        if not bins or fill + size[r] > TREE_BIN_NODES:
            bins.append([0, 0])
            fill = 0
        fill += size[r]
        bins[-1][0] += int(size[r])
        bins[-1][1] = max(bins[-1][1], int(sub_depth[r] - depth[r]) + 1)
    st["bottom_nodes"] = max((b[0] for b in bins), default=0)
    st["bottom_levels"] = max((b[1] for b in bins), default=0)
    top = np.nonzero(is_top)[0]
    exch = [c for v in top if internal[v] for c in (left[v], right[v]) if not is_top[c]]
    st["top_nodes"] = len(top) + len(exch)
    st["top_levels"] = int(max(depth[list(top) + exch].max() + 1, 0)) if len(top) else 0
    return st


def dfs_fwd_smem(st, KP):
    """dynamic shared memory of k3d_tree_fwd (tree_kernels.cu dfs_fwd_smem)"""
    return (st["max_depth"] + 2) * DFS_RUNS_PER_CTA * KP * 8 + ((max(st["dfs_max_nk"], 1) + 1) & ~1) * KP * 8 + \
        DFS_RUNS_PER_CTA * (DFS_RUN + 2) * DNODE_BYTES


def path_fwd_smem(st, KP):
    """dynamic shared memory of k3p_tree_fwd (tree_kernels.cu path_fwd_smem)"""
    return st["max_ganc"] * (16 * KP + 2) + 16 + 2 * st["max_gsuf"]


def predicted_route(st, KP, chain_min_nodes=CHAIN_MIN_NODES):
    """tree_route (tree_kernels.cu) on the restated schedule"""
    if st["caterpillar"] and st["N"] >= chain_min_nodes:
        return "chain"
    kpc = min(KP, 8)
    bins_fit = st["bottom_nodes"] * (SNODE_BYTES + 24 * kpc) + 4 * (st["bottom_levels"] + 2) <= ROUTE_SMEM_LIMIT and \
        st["top_nodes"] * (SNODE_BYTES + 24) + 4 * (st["top_levels"] + 2) <= ROUTE_SMEM_LIMIT
    if not bins_fit:
        return "levels_global"
    if st["preorder"] and KP <= 16 and dfs_fwd_smem(st, KP) <= ROUTE_SMEM_LIMIT:
        return "dfs"
    if st["path_tables"] and path_fwd_smem(st, KP) <= ROUTE_SMEM_LIMIT:
        return "path"
    return "levels_smem"


_STATS = {}


def _stats(tree):
    if tree not in _STATS:
        _STATS[tree] = tree_stats(*TREES[tree]())
    return _STATS[tree]


def _chain_min(tree):
    return int(NO_CHAIN) if tree in RAISED_CHAIN_MIN else CHAIN_MIN_NODES


def test_catalogue_reaches_every_route_at_every_width():
    """The restated route rules send every catalogue case where the catalogue says, and the catalogue covers every
    (route, KP) pair, the padded widths and the trees whose route depends on KP."""
    for c in CATALOGUE:
        assert predicted_route(_stats(c.tree), pad_k(c.K), _chain_min(c.tree)) == c.route, c
    pairs = {(c.route, pad_k(c.K)) for c in CATALOGUE}
    assert pairs == {(r, kp) for r in ROUTES for kp in KPS}, sorted(pairs)
    assert {1, 3, 5, 6, 12, 16} <= {c.K for c in CATALOGUE}
    by_tree = collections.defaultdict(set)
    for c in CATALOGUE:
        by_tree[c.tree].add(c.route)
    assert by_tree["deep_preorder"] == {"dfs", "levels_smem"} and by_tree["sequential_900"] == {"path", "levels_smem"}
    st = _stats("deep_preorder")
    assert st["preorder"] and 90 <= st["max_depth"] <= DFS_MAX_DEPTH
    assert dfs_fwd_smem(st, 8) <= ROUTE_SMEM_LIMIT < dfs_fwd_smem(st, 16)


def test_sequential_900_path_tables_outgrow_shared_memory_at_16_draws():
    """Why the sequential_900 case exists: the caterpillar of 900 leaves gets root-path tables (a group has up to 899
    ancestors), and k3p_tree_fwd would need more than the opt-in shared memory of a CTA for them at KP = 16.  The path
    route must therefore not be taken there (it was, before tree_route checked the path kernel's shared memory)."""
    st = _stats("sequential_900")
    assert st["path_tables"] and st["max_ganc"] == 899
    assert path_fwd_smem(st, 8) <= ROUTE_SMEM_LIMIT
    assert path_fwd_smem(st, 16) > MAX_SMEM_PER_CTA
    for tree in ("children_first_1000", "sequential_313"):       # the path-route trees fit at every width
        assert not _stats(tree)["preorder"] and path_fwd_smem(_stats(tree), 16) <= ROUTE_SMEM_LIMIT


# ------------------------------------------------------------------------------------------- GPU tests
_SAMPLES = {}


def _sample(n):
    """a synthetic sample of M_ROWS rows over n transcripts (seeded by n): (RNASeqSample, numpy arrays)"""
    if n not in _SAMPLES:
        import polee_b200 as pb
        from polee_b200 import synth
        s = synth.to_numpy_sample(synth.make_sample(M_ROWS, n, seed=n))
        _SAMPLES[n] = (pb.RNASeqSample(s["m"], s["n"], s["colptr"], s["rowval"], s["nzval"], s["efflens"]), s)
    return _SAMPLES[n]


def _tree(name):
    pi, js = TREES[name]()
    return np.asarray(pi, np.int32), np.asarray(js, np.int32)


@pytest.fixture
def chain_env(monkeypatch):
    """sets POLEE_CHAIN_MIN_NODES for a tree (read when the tree is uploaded)"""
    def set_for(tree):
        if tree in RAISED_CHAIN_MIN:
            monkeypatch.setenv("POLEE_CHAIN_MIN_NODES", NO_CHAIN)
        else:
            monkeypatch.delenv("POLEE_CHAIN_MIN_NODES", raising=False)
    return set_for


def _max_abs(a, b):
    return float(np.max(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64))))


def _relerr(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))


def _leaf_factor_differences(pi, js, ys_a, ys_b):
    """[K][n]: for every draw and leaf, the sum along the leaf's root path of the relative differences between the
    factors the transform multiplies -- y (into the left child) and 1 - y (into the right child) -- under ys_a and
    ys_b.  To first order, the relative difference of the leaf's x."""
    right, left = _children(pi)
    N, K = len(pi), ys_a.shape[0]
    rel = np.zeros((N, K))
    k = 0
    for i in range(N):
        if js[i] == 0:
            a, b = ys_a[:, k], ys_b[:, k]
            rel[left[i]] = rel[i] + np.abs(a - b) / b
            rel[right[i]] = rel[i] + np.abs((1.0 - a) - (1.0 - b)) / (1.0 - b)
            k += 1
    out = np.zeros((K, (N + 1) // 2))
    leaves = np.nonzero(np.asarray(js) > 0)[0]
    out[:, np.asarray(js)[leaves] - 1] = rel[leaves].T
    return out


@gpu
@pytest.mark.parametrize("gradonly", [False, True])
@pytest.mark.parametrize("case", CATALOGUE, ids=_case_id)
def test_one_step_matches_oracle(oracle, chain_env, case, gradonly):
    """likelihood-approximation.jl:511-559 for K injected-noise draws at non-trivial parameters, on the case's route:
    the tolerances of test_gpu_parity.test_one_step_of_draws_matches_oracle."""
    import polee_b200 as pb
    pi, js = _tree(case.tree)
    n, K = (len(pi) + 1) // 2, case.K
    sample, s = _sample(n)
    chain_env(case.tree)
    rng = np.random.default_rng(1000 * K + n)
    h = pb.Handle(num_mc_samples=K, noise_mode=1, gradonly=gradonly, num_steps=2)
    h.set_sample(sample, tree_topology=(pi, js))
    mu, om, _ = h.get_params()
    om = (om + rng.uniform(-0.3, 0.3, n - 1)).astype(np.float32)
    al = (rng.normal(size=n - 1) * 0.1).astype(np.float32)
    h.set_params(mu, om, al)
    zs0 = rng.normal(size=(K, n - 1)).astype(np.float32)
    d = h.lsn_draws(zs0)
    assert h.layout_info()["tree_route"] == case.route
    h.close()
    acc = {k: np.zeros(n - 1) for k in ("mu_grad", "omega_grad", "alpha_grad")}
    elbo = 0.0
    to = oracle.PTT(pi, js)
    draws = [oracle.lsn_draw(s["m"], n, s["colptr"], s["rowval"], s["nzval"], s["efflens"], pi, js, mu, om, al, zs0[k],
                             gradonly=gradonly) for k in range(K)]
    # x: the route's forward of the device's own ys is the reference's transform! of them (the chain scans: to
    # rounding, see test_large_sequential_tree_scan_path).  Against the oracle's draw, a leaf's x differs by what the
    # few-ulp differences of ys (Float32 expf / sinhf / asinhf: CUDA vs glibc) make of the factors on its root path:
    # y ~ 1 - 1/n on a caterpillar's spine, so a 1-ulp change of y is a relative change of ~1e-7 n in 1 - y, far above
    # the 2e-5 that bounds x on the fixture's shallow tree.  The bound below is that first-order propagation (+ the
    # Float32 rounding of both x).
    x_bound = _leaf_factor_differences(pi, js, d["ys"], np.stack([o["ys"] for o in draws])) * 1.01 + 2.5e-7
    for k, o in enumerate(draws):
        assert np.all(o["xs"] > 1e-10), "a clamped leaf: the case's parameters spread too far"
        assert _relerr(d["ys"][k], o["ys"]) <= 2e-6, k            # Float32 expf / sinhf / asinhf: CUDA vs glibc
        xt = np.clip(to.transform(d["ys"][k])[0], np.float32(1e-10), np.float32(1 - 1e-10))
        assert _relerr(d["xs"][k], xt) <= (2e-7 if case.route == "chain" else 0.0), k
        assert np.all(np.abs(d["xs"][k].astype(np.float64) - o["xs"]) <= x_bound[k] * o["xs"]), k
        assert _max_abs(d["x_grad"][k], o["x_grad"]) <= 1e-5 * np.abs(o["x_grad"]).max(), k
        # the chain scans re-associate the Float64 products of a spine of n - 1 nodes, where the reference rounds G
        # to Float32 at every node (test_gpu_parity.test_large_sequential_tree_scan_path)
        yg_tol = 2e-5 if case.route == "chain" else 1e-5
        assert _max_abs(d["y_grad"][k], o["y_grad"]) <= yg_tol * np.abs(o["y_grad"]).max(), k
        for key in acc:
            acc[key] += o[key]
        elbo += o["elbo"]
    for key in acc:
        ref = acc[key] / K
        assert _max_abs(d[key], ref) <= 1e-5 * np.abs(ref).max(), key
    if gradonly:
        assert d["elbo"] == 0.0
    else:
        assert abs(d["elbo"] - elbo / K) <= 1e-7 * abs(elbo / K)


# one case per route for the fits: a tree and what its route is at both K = 6 and K = 16
FIT_TREES = {"dfs": "random_2000", "path": "children_first_1000", "levels_smem": "spine_1225",
             "levels_global": "sequential_6000", "chain": "sequential_2500"}
# ADAM steps of the fits compared with the oracle.  The device's ys differ from the reference's by a Float32 ulp here
# and there (CUDA's expf vs glibc's); on a deep spine, where y ~ 1 - 1/(n - k), such an ulp is a relative change of
# ~6e-8 (n - k) in a leaf's x and gradient, which the ADAM steps then amplify: the trajectories part by more than 2e-4
# after some 20 steps on these trees (and on the caterpillar of 6 000 leaves at 16 draws after some 5), and after ~17
# steps both the device's and the reference's ELBO reach -inf on the deep ones.  The fits are shortened accordingly.
FIT_STEPS = {"dfs": 10, "path": 20, "levels_smem": 10, "levels_global": 3, "chain": 10}


def _noise(steps, K, n, seed):
    return np.random.default_rng(seed).normal(size=(steps, K, n - 1)).astype(np.float32)


def _device_fit(tree, K, steps, noise, use_cuda_graph=True):
    import polee_b200 as pb
    pi, js = _tree(tree)
    sample, _ = _sample((len(pi) + 1) // 2)
    h = pb.Handle(num_mc_samples=K, num_steps=steps, gradonly=False, noise_mode=1, use_cuda_graph=use_cuda_graph)
    h.set_sample(sample, tree_topology=(pi, js))
    out = h.fit(noise=noise, want_elbo=True)
    info = h.layout_info()
    h.close()
    out["route"] = info["tree_route"]
    out["edges"] = np.array([info["graph_programmatic_edges"], info["multi_step_graph_programmatic_edges"]])
    return out


@gpu
@pytest.mark.parametrize("K", [6, 16])
@pytest.mark.parametrize("route", ROUTES)
def test_short_fit_matches_oracle(oracle, chain_env, route, K):
    """FIT_STEPS ADAM steps with injected noise track the oracle on each route: 2e-4 absolute on mu, omega and alpha,
    1e-6 relative on the ELBO trajectory (test_gpu_parity.test_fit_trajectory_matches_oracle_with_injected_noise)."""
    tree, steps = FIT_TREES[route], FIT_STEPS[route]
    assert predicted_route(_stats(tree), pad_k(K), _chain_min(tree)) == route
    chain_env(tree)
    pi, js = _tree(tree)
    n = (len(pi) + 1) // 2
    _, s = _sample(n)
    noise = _noise(steps, K, n, K + n)
    dev = _device_fit(tree, K, steps, noise)
    assert dev["route"] == route
    ora = oracle.fit_lsn_ptt(s["m"], n, s["colptr"], s["rowval"], s["nzval"], s["efflens"], pi, js, num_steps=steps,
                             num_mc_samples=K, noise=noise, gradonly=False, elbo_fix=True)
    for key in ("mu", "omega", "alpha"):
        assert _max_abs(dev[key], ora[key]) <= 2e-4, key
    assert _relerr(dev["elbo"], ora["elbo"]) <= 1e-6


@gpu
@pytest.mark.parametrize("steps", [7, 8, 9, 17])
@pytest.mark.parametrize("route", ROUTES)
def test_graph_and_plain_fits_bit_identical(chain_env, route, steps):
    """The step graphs (one step, and the multi-step graph of 8) replay exactly what the uncaptured steps compute, on
    every route: step counts on both sides of a chunk."""
    tree, K = FIT_TREES[route], 6
    chain_env(tree)
    n = (len(TREES[tree]()[0]) + 1) // 2
    noise = _noise(steps, K, n, steps)
    graph, plain = _device_fit(tree, K, steps, noise), _device_fit(tree, K, steps, noise, use_cuda_graph=False)
    assert graph["route"] == plain["route"] == route
    for key in ("mu", "omega", "alpha", "elbo"):
        assert np.array_equal(graph[key], plain[key]), key


PDL_STEPS, PDL_K = 12, 6         # 3 single steps, then one multi-step graph of 8; a finite ELBO throughout


def _pdl_fit_in_child(route, pdl, tmp_path):
    """a PDL_STEPS-step fit on the route's tree in a fresh process with POLEE_PDL=pdl (read when a handle is made)"""
    out = os.path.join(str(tmp_path), "%s_pdl%d.npz" % (route, pdl))
    env = dict(os.environ, POLEE_PDL=str(pdl))
    env.pop("POLEE_CHAIN_MIN_NODES", None)
    if FIT_TREES[route] in RAISED_CHAIN_MIN:
        env["POLEE_CHAIN_MIN_NODES"] = NO_CHAIN
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), route, out]
    r = subprocess.run(cmd, env=env, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout
    return dict(np.load(out))


@gpu
@pytest.mark.parametrize("route", ["path", "levels_smem", "chain"])
def test_pdl_fit_bit_identical(route, tmp_path):
    """Programmatic dependent launch changes how the step's kernels overlap, not what they compute, on the routes
    whose forward is a plain launch and whose backward is a PDL launch."""
    on, off = _pdl_fit_in_child(route, 1, tmp_path), _pdl_fit_in_child(route, 0, tmp_path)
    assert str(on["route"]) == str(off["route"]) == route
    for key in ("mu", "omega", "alpha", "elbo"):
        assert np.array_equal(on[key], off[key]), key
    assert np.all(np.isfinite(on["elbo"])) and np.any(on["elbo"] != 0.0)
    assert on["edges"][0] > 0 and list(off["edges"]) == [0, 0], (on["edges"], off["edges"])


@gpu
@pytest.mark.parametrize("route,chain_min", [("levels_global", NO_CHAIN), ("chain", "1")])
def test_optimize_ptt_first_steps_tight(oracle, monkeypatch, route, chain_min):
    """OptimizePTTApprox (l-a.jl:149-242) on the sequential tree it builds, after 1, 2 and 3 ADAM steps, on the level
    kernels in global memory and on the chain scans: the bounds of
    test_gpu_parity.test_optimize_ptt_first_steps_tight on the bulk, and on the maximum where n allows it."""
    import polee_b200 as pb
    n = 6000 if route == "levels_global" else 1500       # 1 500 spine nodes still fit the shared-memory level kernels
    # ys = logistic(z) is Float32 (l-a.jl:196) and y ~ 1 - 1/(n - k) on the spine: a 1-ulp difference of y (CUDA's
    # expf vs glibc's) is a relative difference of 2^-24 (n - k) in the factor 1 - y of the leaf below it.  The
    # fixture's 2e-4 on the maximum is a few such ulps at n = 313; the bound scales with n.  The median stays 1e-6.
    max_bound = max(2e-4, 8 * n * 2.0 ** -24)
    sample, s = _sample(n)
    monkeypatch.setenv("POLEE_CHAIN_MIN_NODES", chain_min)
    for steps in (1, 2, 3):
        xo = oracle.fit_optimize_ptt(s["m"], n, s["colptr"], s["rowval"], s["nzval"], s["efflens"], steps)
        h = pb.Handle(approx=1, num_steps=steps)
        h.set_sample(sample)
        x_dev = h.fit_optimize_ptt()
        assert h.layout_info()["tree_route"] == route
        h.close()
        err = np.abs(x_dev.astype(np.float64) - xo) / np.maximum(xo, 1e-30)
        assert np.median(err) <= 1e-6 and err.max() <= max_bound, (steps, np.median(err), err.max())


if __name__ == "__main__":
    # child of test_pdl_fit_bit_identical: <route> <out.npz>
    route, path = sys.argv[1], sys.argv[2]
    tree = FIT_TREES[route]
    n = (len(TREES[tree]()[0]) + 1) // 2
    res = _device_fit(tree, PDL_K, PDL_STEPS, _noise(PDL_STEPS, PDL_K, n, 1))
    np.savez(path, **{k: res[k] for k in ("mu", "omega", "alpha", "elbo", "edges", "route")})
