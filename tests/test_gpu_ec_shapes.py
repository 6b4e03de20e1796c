"""The equivalence-class likelihood pass (`k_ec_lik` + `k_ec_combine1/2`, ec_kernels.cu; layout from ec_setup.cu) at
every class shape it dispatches, against a plain Float64 restatement of the same products.

The matrix is designed, not sampled: for every class width L in 1..64 there are classes whose row count R hits each
case the kernel treats differently (one row, a partial block, one full block, a block and one row more, several full
blocks, exactly one full task, one task and one row), a hub column with more than FT_UNIT partials (so the second
combine stage runs), pairs of classes that differ only in their last column, and shuffled rows.  The tests run every K
in 1..16 in both class arithmetics, pin the layout counts to what the Python restatement of the layout predicts,
and check that the grid size, the draw batching, row weights, the 1/p output, the mix with the general layouts and the
upload path do not change the results beyond what the arithmetic allows.  A mismatch names the class shape (L, q, R)
it comes from."""
import numpy as np
import pytest

# ---------------------------------------------------------------- the layout arithmetic of common.cuh, restated
EC_MAX_L = 64
EC_V_BYTES = 8192
EC_MAX_NBT = 32
EC_MIN_ROWS_DEFAULT = 12
FT_UNIT = 64


def ec_q(L):
    return 1 if L <= 8 else 2 if L <= 16 else 4 if L <= 32 else 8


def ec_lh(L):
    return -(-L // ec_q(L))


def ec_nbt(L):
    return max(1, min(EC_MAX_NBT, EC_V_BYTES // (ec_lh(L) * 128)))


def ec_hdr_bytes(L):
    return (16 + 8 * ec_q(L) * ec_lh(L) + 15) & ~15


def row_count_cases(L):
    """The row counts of a class of width L that take different paths: rpb = 32 / q rows per block, `full` rows fill
    one task of ec_nbt(L) blocks."""
    rpb = 32 // ec_q(L)
    full = ec_nbt(L) * rpb
    return {"1": 1, "rpb-1": rpb - 1, "rpb": rpb, "2rpb+1": 2 * rpb + 1, "3rpb": 3 * rpb, "full": full,
            "full+1": full + 1}


class EcClass:
    def __init__(self, L, R, case, cols):
        self.L, self.R, self.case, self.cols = L, R, case, cols
        self.q, self.lh = ec_q(L), ec_lh(L)
        self.hub = False

    def blocks(self):
        return -(-self.R // (32 // self.q))

    def tasks(self):
        return -(-self.blocks() // ec_nbt(self.L))

    def __str__(self):
        if self.L > EC_MAX_L:
            return "L=%d R=%d (general layouts)" % (self.L, self.R)
        return "L=%d q=%d LH=%d R=%d (%s)%s" % (self.L, self.q, self.lh, self.R, self.case, " hub" if self.hub else "")


class Design:
    """A CSC sample (1-based uint32 colptr / rowval, float32 nzval) built class by class."""

    def __init__(self, n, classes, rng, hub, isolated=False):
        import scipy.sparse as sp
        self.n, self.classes, self.hub, self.isolated = n, classes, hub, isolated
        self.m = sum(c.R for c in classes)
        rows, cols, vals, row_class = [], [], [], []
        r0 = 0
        lo, hi = np.log(1.0001e-12), np.log(1e-2)          # log-uniform, as synth.py bounds the values
        for ci, c in enumerate(classes):
            rows.append(np.repeat(np.arange(r0, r0 + c.R), c.L))
            cols.append(np.tile(c.cols, c.R))
            vals.append(np.exp(rng.uniform(lo, hi, c.R * c.L)).astype(np.float32))
            row_class.append(np.full(c.R, ci))
            r0 += c.R
        perm = rng.permutation(self.m)                     # shuffled: the classes interleave
        rows = perm[np.concatenate(rows)]
        self.row_class = np.empty(self.m, np.int64)
        self.row_class[perm] = np.concatenate(row_class)
        A = sp.csc_matrix((np.concatenate(vals), (rows, np.concatenate(cols))), shape=(self.m, n))
        A.sort_indices()
        self.colptr = (A.indptr + 1).astype(np.uint32)
        self.rowval = (A.indices + 1).astype(np.uint32)
        self.nzval = A.data.astype(np.float32)
        self.A = A.astype(np.float64).tocsr()              # the reference's products: Float32 values, Float64 sums
        self.AT = A.T.astype(np.float64).tocsr()
        self.efflens = np.ones(n, np.float32)

    def sample(self, pb):
        return pb.RNASeqSample(self.m, self.n, self.colptr, self.rowval, self.nzval, self.efflens)

    def classes_of_column(self, j):
        return [c for c in self.classes if j in c.colset]


def _random_cols(rng, pool, L, hub):
    cols = rng.choice(pool, L - (hub is not None), replace=False)
    if hub is not None:
        cols = np.append(cols, hub)
    return np.sort(cols)


def make_design(seed=20261020, n=2000, wide=False, isolated=False):
    """Every L in 1..64 x every row-count case; with `wide`, also classes of width 65..80 (general layouts only).
    96 classes contain the hub column; classes (L, "full") of six widths are twins of (L, "rpb") but for the last
    column; a few columns are in no class.

    isolated: the same class shapes, but every class on columns of its own (n becomes ~15 000, no hub): then a wrong
    gradient entry belongs to exactly one class, and a failure names the broken shapes exactly."""
    d = _make_shared(seed, n, wide)
    if not isolated:
        return d
    nxt, empty = 0, lambda j: j % 250 == 7
    for c in d.classes:
        cols = []
        while len(cols) < c.L:
            if not empty(nxt):
                cols.append(nxt)
            nxt += 1
        c.cols = np.array(cols)
        c.colset = set(cols)
        c.hub = False
    return Design(nxt + 8, d.classes, np.random.default_rng(seed + 1), hub=-1, isolated=True)


def _make_shared(seed, n, wide):
    rng = np.random.default_rng(seed)
    hub = n // 2
    empty = np.arange(7, n, 250)
    pool = np.setdiff1d(np.arange(n), np.append(empty, hub))
    specs = [(L, case, R) for L in range(1, EC_MAX_L + 1) for case, R in row_count_cases(L).items()]
    if wide:
        specs += [(L, "wide", int(rng.integers(1, 6))) for L in range(EC_MAX_L + 1, 81)]
    with_hub = set(rng.choice([i for i, s in enumerate(specs) if 2 <= s[0] <= EC_MAX_L], 96, replace=False).tolist())
    twins = {3, 8, 12, 24, 48, 64}
    classes, seen, by_case = [], set(), {}
    for i, (L, case, R) in enumerate(specs):
        while True:
            if case == "full" and L in twins:
                cols = by_case[(L, "rpb")].cols.copy()
                later = pool[(pool > (cols[-2] if L > 1 else -1)) & (pool != cols[-1])]
                cols[-1] = rng.choice(later)
            else:
                cols = _random_cols(rng, pool, L, hub if i in with_hub else None)
            if tuple(cols) not in seen:
                break
        seen.add(tuple(cols))
        c = EcClass(L, R, case, cols)
        c.colset = set(cols.tolist())
        c.hub = hub in c.colset
        by_case[(L, case)] = c
        classes.append(c)
    return Design(n, classes, rng, hub)


def predict_layout(d, min_rows=None):
    """layout_info() of the design as ec_setup.cu builds it.  min_rows: POLEE_EC_MIN_ROWS, or None for the default
    policy (every class when the padded blobs stay below 8 bytes per entry, else classes of >= 12 rows)."""
    def table(min_r):
        t = dict(rows=0, nnz=0, tasks=0, blocks=0, parts=0, bytes=0, taken=[])
        for c in d.classes:
            if c.R < min_r or c.L > EC_MAX_L:
                continue
            nb, nt = c.blocks(), c.tasks()
            t["rows"] += c.R
            t["nnz"] += c.R * c.L
            t["tasks"] += nt
            t["blocks"] += nb
            t["parts"] += nt * c.L
            t["bytes"] += nt * ec_hdr_bytes(c.L) + nb * c.lh * 128
            t["taken"].append(c)
        return t
    t = table(min_rows if min_rows is not None else 1)
    if min_rows is None and t["bytes"] > 8 * t["nnz"]:
        t = table(EC_MIN_ROWS_DEFAULT)
    if t["tasks"] == 0:
        return dict(ec_rows=0, ec_nnz=0, ec_classes=0, ec_tasks=0, ec_blob_bytes=0, ec_partials=0, ec_row_slots=0,
                    general_rows=d.m), t
    return dict(ec_rows=t["rows"], ec_nnz=t["nnz"], ec_classes=len(d.classes), ec_tasks=t["tasks"],
                ec_blob_bytes=t["bytes"], ec_partials=t["parts"], ec_row_slots=32 * t["blocks"],
                general_rows=d.m - t["rows"]), t


def column_partials(d, taken):
    cnt = np.zeros(d.n, np.int64)
    for c in taken:
        cnt[c.cols] += c.tasks()
    return cnt


# ---------------------------------------------------------------- the Float64 reference
def reference(d, xs, ks=None, rows=None):
    """p = A x, lp = sum_i k_i log p_i, g = A^T (k / p), w = 1 / p, all in Float64 from the Float32 inputs.
    rows: a row mask; then also the share of those rows in lp and g."""
    x = np.atleast_2d(xs).astype(np.float64)
    p = d.A @ x.T                                           # (m, K)
    k = np.ones(d.m) if ks is None else np.asarray(ks, np.float64)
    lp = (k[:, None] * np.log(p)).sum(0)
    g = (d.AT @ (k[:, None] / p)).T
    if rows is None:
        return lp, g, 1.0 / p.T
    kr = k * rows
    return lp, g, 1.0 / p.T, (kr[:, None] * np.log(p)).sum(0), (d.AT @ (kr[:, None] / p)).T


def draws(K, n, seed):
    """K draws, rotating through Dirichlet(0.5) clipped to 1e-10, the uniform 1/n and x ~ 10^U(-10, 0) normalised."""
    rng = np.random.default_rng(seed)
    xs = np.empty((K, n), np.float32)
    for k in range(K):
        kind = (K + k) % 3
        if kind == 0:
            xs[k] = rng.dirichlet(np.full(n, 0.5)).clip(1e-10)
        elif kind == 1:
            xs[k] = np.float32(1) / np.float32(n)
        else:
            x = 10.0 ** rng.uniform(-10, 0, n)
            xs[k] = x / x.sum()
    return xs


def _relerr(got, want):
    """|got - want| / |want| elementwise; where want is 0 the result is 0 if got is exactly 0, else inf."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        e = np.where(want != 0, np.abs(got - want) / np.abs(want), np.where(got == 0, 0.0, np.inf))
    return np.nan_to_num(e, nan=np.inf)


def _summary(classes, limit=6):
    kinds = sorted({(c.q, c.lh) for c in classes})
    cases = sorted({c.case for c in classes})
    return "%d classes, (q, LH) kinds %s, row cases %s: %s%s" % (
        len(classes), kinds, cases, "; ".join(str(c) for c in classes[:limit]), " ..." if len(classes) > limit else "")


def _tolerance(tol, ref, part=None, tol_part=None):
    """Relative tolerance per entry: tol on the share of the class rows, tol_part on the share `part` of the rows in
    the general layouts (their own arithmetic; every term of a sum has the sign of the sum, so the shares are in 0..1)."""
    if part is None:
        return np.full(np.shape(ref), tol)
    with np.errstate(divide="ignore", invalid="ignore"):
        share = np.where(ref != 0, np.abs(part) / np.abs(ref), 0.0)
    return tol * (1.0 - share) + tol_part * share


def check_grad(d, g, g_ref, tol, what, g_general=None, tol_general=None):
    """g vs the reference on every draw and column; on failure, name the worst column's classes (and, when every class
    has columns of its own, every class with a column off)."""
    e = _relerr(g, g_ref)                                   # (K, n)
    t = _tolerance(tol, g_ref, g_general, tol_general)
    if np.all(e <= t):
        return float(e.max())
    k, j = np.unravel_index(int(np.argmax(e / t)), e.shape)
    msg = "%s: x_grad[%d][%d] = %.17g, reference %.17g (relative error %.3e > %.1e); column %d%s is in %s" % (
        what, k, j, g[k][j], g_ref[k][j], e[k, j], t[k, j], j, " (the hub)" if j == d.hub else "",
        _summary(d.classes_of_column(j)))
    if d.isolated:
        off = (e > t).any(0)
        msg += ". Classes with a column off: " + _summary([c for c in d.classes if off[c.cols].any()], 10)
    raise AssertionError(msg)


def check_rows(d, w, w_ref, tol, what, general=None, tol_general=None):
    """1/p per row: finite, positive (a row nobody wrote reads 0), within tol of the reference (tol_general on the rows
    of the mask `general`); name the row's class."""
    w = np.asarray(w, np.float64)
    e = np.where(np.isfinite(w) & (w > 0), _relerr(w, w_ref), np.inf)
    t = np.full(d.m, tol) if general is None else np.where(general, tol_general, tol)
    if np.all(e <= t):
        return float(e.max())
    i = int(np.argmax(e / t))
    bad = sorted({int(c) for c in d.row_class[e > t]})
    raise AssertionError("%s: 1/p of row %d = %.9g, reference %.17g (relative error %.3e > %.1e%s); row of class %s. "
                         "Classes with a row off: %s" % (what, i, w[i], w_ref[i], e[i], t[i],
                                                         ", never written" if w[i] == 0 else "",
                                                         d.classes[d.row_class[i]], _summary([d.classes[c] for c in bad])))


def check_lp(lp, lp_ref, tol, what, lp_general=None, tol_general=None):
    e = _relerr(lp, lp_ref)
    t = _tolerance(tol, lp_ref, lp_general, tol_general)
    assert np.all(e <= t), "%s: lp relative error %s > %s (lp %s, reference %s)" % (what, e, t, lp, lp_ref)
    return float(e.max())


# tolerances: exact_accumulation = 0 (Float32 class arithmetic) and 2 (Float64, RCP64H + one Newton step)
TOL = {0: {"g": 1e-5, "lp": 1e-8, "w": 1e-5}, 2: {"g": 1e-10, "lp": 1e-12, "w": 1e-7}}
# rows the classes do not take run in the general layouts, whose arithmetic is not the class kernel's: with
# exact_accumulation = 2 they use the reference's order (each product and frag_probs rounded to Float32, ~1e-7 from
# Float64).  Their share of a result is held to the gates the suite applies to those layouts against the oracle.
TOL_GENERAL = {"g": 1e-5, "lp": 1e-8, "w": 1e-5}


# ---------------------------------------------------------------- CPU: the design reaches what it claims to
def test_design_covers_every_class_shape():
    d = make_design()
    cases = {}
    for c in d.classes:
        cases.setdefault(c.L, {})[c.case] = c.R
    for L in range(1, EC_MAX_L + 1):
        assert cases[L] == row_count_cases(L), L
        assert len(set(cases[L].values())) == 7, L          # seven distinct row counts per width
    assert len({tuple(c.cols) for c in d.classes}) == len(d.classes)
    twins = [(a, b) for a in d.classes for b in d.classes
             if a.L == b.L and a.L > 1 and a.case == "rpb" and b.case == "full" and np.array_equal(a.cols[:-1], b.cols[:-1])]
    assert len(twins) == 6 and all(a.cols[-1] != b.cols[-1] for a, b in twins)
    info, t = predict_layout(d)
    assert info["ec_rows"] == d.m and info["general_rows"] == 0     # below 8 B per entry: the policy takes every class
    assert t["bytes"] < 8 * t["nnz"]
    kinds = {(c.lh, c.q) for c in t["taken"]}
    assert len(kinds) == 20                                 # LH 1..4 with q = 1, LH 5..8 with q = 1, 2, 4, 8
    parts = column_partials(d, t["taken"])
    assert parts[d.hub] > FT_UNIT and sum(c.hub for c in d.classes) >= 80
    assert (np.diff(d.colptr.astype(np.int64)) == 0).sum() >= 8      # columns in no class
    # the sample is a valid CSC of the design: row lengths and the reference's products
    assert np.array_equal(np.bincount(d.rowval - 1, minlength=d.m), [d.classes[c].L for c in d.row_class])
    assert d.nzval.min() >= np.float32(1.0001e-12) and d.nzval.max() <= np.float32(1e-2)
    xs = draws(3, d.n, 0)
    lp, g, w = reference(d, xs)
    assert np.allclose((xs.astype(np.float64) * g).sum(1), d.m, rtol=1e-12)   # sum_j x_j g_j = m
    mixed = make_design(wide=True)
    mi, _ = predict_layout(mixed, min_rows=EC_MIN_ROWS_DEFAULT)
    assert mi["ec_rows"] > 0 and mi["general_rows"] > 0 and mi["ec_rows"] + mi["general_rows"] == mixed.m
    assert {c.L for c in mixed.classes if c.R < EC_MIN_ROWS_DEFAULT} >= set(range(1, EC_MAX_L + 1))
    iso = make_design(isolated=True)
    assert [(c.L, c.R) for c in iso.classes] == [(c.L, c.R) for c in d.classes]
    per_col = np.bincount(np.concatenate([c.cols for c in iso.classes]), minlength=iso.n)
    assert per_col.max() == 1 and (per_col == 0).sum() >= 8                # one class per column, some empty columns
    assert predict_layout(iso)[0]["ec_tasks"] == info["ec_tasks"]


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def pb():
    import polee_b200
    return polee_b200


@pytest.fixture(scope="module")
def design():
    return make_design()


@pytest.fixture(scope="module")
def isolated():
    return make_design(isolated=True)


@pytest.fixture(scope="module")
def mixed():
    return make_design(wide=True)


def _handle(pb, d, K, exact, ks=None):
    h = pb.Handle(num_mc_samples=K, exact_accumulation=exact)
    h.set_sample(d.sample(pb), ks)
    h.set_tree_sequential(d.n)                              # loglik_grad sizes its work buffers from a tree
    return h


@pytest.mark.gpu
@pytest.mark.parametrize("columns", ["shared", "isolated"])
@pytest.mark.parametrize("exact", [0, 2])
def test_every_k_against_float64_reference(pb, design, isolated, exact, columns):
    d, tol = design if columns == "shared" else isolated, TOL[exact]
    h = _handle(pb, d, 8, exact)
    info = h.layout_info()
    want, _ = predict_layout(d)
    assert {k: info[k] for k in want} == want
    for K in range(1, 17):
        xs = draws(K, d.n, 100 + K)
        lp, g = h.loglik_grad(xs, gradonly=False)
        lp_r, g_r, _ = reference(d, xs)
        check_grad(d, g, g_r, tol["g"], "exact=%d K=%d" % (exact, K))
        check_lp(lp, lp_r, tol["lp"], "exact=%d K=%d" % (exact, K))
        lp2, g2 = h.loglik_grad(xs, gradonly=False)
        assert np.array_equal(lp, lp2) and np.array_equal(g, g2), "K=%d: repeat call differs" % K
    h.close()


@pytest.mark.gpu
@pytest.mark.parametrize("exact", [0, 2])
def test_grid_size_does_not_change_a_bit(pb, design, exact, monkeypatch):
    """Each task writes its own partial slot, so the number of CTAs must not matter.  POLEE_EC_CTAS=1 makes every warp
    run ~40-60 tasks through all LH kinds: the pipeline's refills and phase bits carry across tasks and kinds."""
    d = design
    xs16 = draws(16, d.n, 7)
    out = {}
    for ctas in (None, "1", "3"):
        if ctas is None:
            monkeypatch.delenv("POLEE_EC_CTAS", raising=False)
        else:
            monkeypatch.setenv("POLEE_EC_CTAS", ctas)       # read when the work buffers are sized
        h = _handle(pb, d, 8, exact)
        res = [h.loglik_grad(xs16[:K], gradonly=False) for K in (1, 3, 5, 8, 16)]
        res.append(h.frag_prob_recip(xs16[2]))
        h.close()
        out[ctas] = res
    for ctas in ("1", "3"):
        for a, b in zip(out[None], out[ctas]):
            for u, v in zip(a if isinstance(a, tuple) else (a,), b if isinstance(b, tuple) else (b,)):
                assert np.array_equal(u, v), "POLEE_EC_CTAS=%s changes the result" % ctas
    lp_r, g_r, _ = reference(d, xs16)
    check_grad(d, out["1"][-2][1], g_r, TOL[exact]["g"], "exact=%d POLEE_EC_CTAS=1" % exact)


@pytest.mark.gpu
@pytest.mark.parametrize("exact", [0, 2])
def test_draw_alone_equals_draw_in_batch(pb, design, exact):
    """Per draw, the class kernel does the same arithmetic whatever KD; only the Float64 order of k_ec_combine2 and of the
    lp reduction depends on KP."""
    d = design
    xs = draws(16, d.n, 11)
    h = _handle(pb, d, 1, exact)
    lp16, g16 = h.loglik_grad(xs, gradonly=False)
    lp8, g8 = h.loglik_grad(xs[:8], gradonly=False)
    for k in range(16):
        lp1, g1 = h.loglik_grad(xs[k], gradonly=False)
        for lpb, gb, K in ((lp16, g16, 16), (lp8, g8, 8)):
            if k < K:
                check_grad(d, g1, gb[k:k + 1], 1e-12, "exact=%d draw %d alone vs in K=%d" % (exact, k, K))
                check_lp(lp1, lpb[k:k + 1], 1e-12, "exact=%d draw %d alone vs in K=%d" % (exact, k, K))
    h.close()


@pytest.mark.gpu
@pytest.mark.parametrize("exact", [0, 2])
def test_row_weights(pb, design, exact):
    d, tol = design, TOL[exact]
    ks = np.random.default_rng(5).integers(1, 9, d.m)
    h = _handle(pb, d, 6, exact, ks)
    for K in (1, 6, 16):
        xs = draws(K, d.n, 200 + K)
        lp, g = h.loglik_grad(xs, gradonly=False)
        lp_r, g_r, _ = reference(d, xs, ks)
        check_grad(d, g, g_r, tol["g"], "exact=%d weighted K=%d" % (exact, K))
        check_lp(lp, lp_r, tol["lp"], "exact=%d weighted K=%d" % (exact, K))
    h.close()


@pytest.mark.gpu
@pytest.mark.parametrize("exact", [0, 2])
def test_frag_prob_recip_every_row(pb, design, exact):
    """1/p through the class layout, scattered back to the rows' original positions."""
    d = design
    h = _handle(pb, d, 1, exact)
    xs = draws(3, d.n, 300)
    for k in range(3):
        w = h.frag_prob_recip(xs[k])
        _, _, w_r = reference(d, xs[k])
        check_rows(d, w, w_r[0], TOL[exact]["w"], "exact=%d draw kind %d" % (exact, (3 + k) % 3))
    h.close()


@pytest.mark.gpu
@pytest.mark.parametrize("exact", [0, 2])
def test_classes_and_general_layouts_mixed(pb, mixed, exact, monkeypatch):
    """POLEE_EC_MIN_ROWS=12 and rows of width 65..80: the general pass runs first, the class pass adds into g and lp."""
    monkeypatch.setenv("POLEE_EC_MIN_ROWS", "12")
    d = mixed
    h = _handle(pb, d, 8, exact)
    info = h.layout_info()
    want, t = predict_layout(d, min_rows=12)
    assert {k: info[k] for k in want} == want
    assert info["ec_rows"] > 0 and info["general_rows"] > 0 and info["ec_rows"] + info["general_rows"] == d.m
    _check_with_general_rows(h, d, exact, t, (1, 3, 8, 16), 400, "mixed")
    h.close()


def _check_with_general_rows(h, d, exact, layout, Ks, seed, what):
    """loglik_grad and frag_prob_recip vs the reference when some rows are in the general layouts: the class rows' share
    is held to the class arithmetic's tolerance, the general rows' share to TOL_GENERAL."""
    tol = TOL[exact]
    taken = {id(c) for c in layout["taken"]}
    general = np.array([id(c) not in taken for c in d.classes])[d.row_class]
    assert general.sum() == d.m - layout["rows"]
    for K in Ks:
        xs = draws(K, d.n, seed + K)
        lp, g = h.loglik_grad(xs, gradonly=False)
        lp_r, g_r, _, lp_g, g_g = reference(d, xs, rows=general)
        tag = "%s exact=%d K=%d" % (what, exact, K)
        check_grad(d, g, g_r, tol["g"], tag, g_g, TOL_GENERAL["g"])
        check_lp(lp, lp_r, tol["lp"], tag, lp_g, TOL_GENERAL["lp"])
    x = draws(1, d.n, seed + 99)
    check_rows(d, h.frag_prob_recip(x[0]), reference(d, x)[2][0], tol["w"], "%s exact=%d" % (what, exact), general,
               TOL_GENERAL["w"])


def _width_design(widths, R, seed):
    rng = np.random.default_rng(seed)
    n = 300
    classes = []
    for L in widths:
        c = EcClass(L, R, "wide" if L > EC_MAX_L else "limit", np.sort(rng.choice(n, L, replace=False)))
        c.colset = set(c.cols.tolist())
        classes.append(c)
    return Design(n, classes, rng, hub=-1)


@pytest.mark.gpu
@pytest.mark.parametrize("exact", [0, 2])
def test_class_width_limit(pb, exact):
    """L = 64 is a class, L = 65 is not; a matrix with only wider rows has no class task and still matches."""
    for widths, ec_rows in (((64, 65), 40), (tuple(range(65, 81)), 0)):
        d = _width_design(widths, 40, len(widths))
        h = _handle(pb, d, 8, exact)
        info = h.layout_info()
        want, t = predict_layout(d)
        assert {k: info[k] for k in want} == want
        assert info["ec_rows"] == ec_rows and info["general_rows"] == d.m - ec_rows
        assert (info["ec_tasks"] == 0) == (ec_rows == 0)
        _check_with_general_rows(h, d, exact, t, (1, 8), 500, "widths %s" % (widths[:2],))
        h.close()


@pytest.mark.gpu
def test_device_upload_equals_host_upload(pb, design):
    import torch
    d = design
    ks = np.random.default_rng(6).integers(1, 9, d.m)
    xs = draws(6, d.n, 600)
    cp = torch.from_numpy(d.colptr.view(np.int32)).cuda()
    rv = torch.from_numpy(d.rowval.view(np.int32)).cuda()
    nz = torch.from_numpy(d.nzval).cuda()
    kd = torch.from_numpy(ks.astype(np.int64)).cuda()
    torch.cuda.synchronize()
    for weights in (None, ks):
        res = []
        for device_upload in (False, True):
            h = pb.Handle(num_mc_samples=6)
            if device_upload:
                h.set_matrix_device(d.m, d.n, cp.data_ptr(), rv.data_ptr(), nz.data_ptr(),
                                    kd.data_ptr() if weights is not None else 0)
            else:
                h.set_sample(d.sample(pb), weights)
            h.set_tree_sequential(d.n)
            res.append(h.loglik_grad(xs, gradonly=False) + (h.frag_prob_recip(xs[0]),))
            h.close()
        for a, b in zip(*res):
            assert np.array_equal(a, b), "weights=%s" % (weights is not None)
    del cp, rv, nz, kd
