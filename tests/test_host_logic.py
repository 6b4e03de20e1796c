"""CPU tests of the host side: the C-ABI library loads and exports what include/polee_b200.h declares, fails
loudly without a GPU (no fallback), and the pure-host helpers (tree arrays, partitioning, generator) are exact."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT, Fixture


@pytest.fixture(scope="module")
def lib():
    from polee_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build_library()
    return _lib.load_library()


def test_library_exports_every_declared_symbol(lib):
    from polee_b200 import _lib
    header = open(os.path.join(ROOT, "include", "polee_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(polee_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 35
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    for sym in declared:
        assert hasattr(lib, sym), sym


def test_no_cpu_fallback_create_fails_without_gpu(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from polee_b200 import _lib
    import polee_b200 as pb
    h = C.c_void_p()
    o = _lib.PoleeOpts()
    assert lib.polee_opts_default(C.byref(o)) == 0
    assert (o.num_steps, o.num_mc_samples, o.gradonly, o.use_efflen_jacobian) == (500, 6, 1, 1)
    rc = lib.polee_create(C.byref(h), C.byref(o))
    assert rc == _lib.POLEE_ECUDA and not h.value
    assert b"no CPU fallback" in lib.polee_last_error(None)
    with pytest.raises(pb.PoleeError):
        pb.Handle()
    with pytest.raises(pb.PoleeError):   # the hsb ops have no fallback either
        pb.hsb(np.zeros((1, 2), np.float32), [1, -1, -1, -1, -1], [2, -1, -1, -1, -1], [-1, 0, 1, -1, -1][:5])


def test_null_handle_is_an_argument_error_not_a_crash(lib):
    """Every handle entry point checks its handle first (no device needed to say so): the one-call set-up included."""
    from polee_b200 import _lib
    z = C.c_void_p(None)
    u32, f32, i32 = (C.c_uint32 * 2)(1, 1), (C.c_float * 1)(1.0), (C.c_int32 * 1)(0)
    assert lib.polee_set_sample(z, C.c_int64(1), C.c_int64(1), u32, u32, f32, None, f32, i32, i32) == _lib.POLEE_EINVAL
    assert lib.polee_set_tree(z, C.c_int64(1), i32, i32) == _lib.POLEE_EINVAL
    assert lib.polee_run_steps(z, C.c_int32(1)) == _lib.POLEE_EINVAL
    assert lib.polee_destroy(z) == _lib.POLEE_OK


def test_product_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "polee_b200")):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                src = open(os.path.join(dirpath, fn)).read()
                assert "polee_oracle" not in src and "oracle/" not in src, os.path.join(dirpath, fn)


def test_make_inverse_ptt_params_exact(lib, fx, oracle):
    import polee_b200 as pb
    l, r, f = pb.make_inverse_ptt_params(fx.parent_idxs, fx.js)
    lo, ro, fo = oracle.make_inverse_ptt_params(fx.parent_idxs, fx.js)
    assert np.array_equal(l, lo) and np.array_equal(r, ro) and np.array_equal(f, fo)
    assert l[0] > r[0] == 1 and f[0] == -1


def test_sequential_tree_matches_list_nodes(oracle):
    from polee_b200.api import sequential_tree
    for n in (2, 3, 17, 313):
        pi, js = sequential_tree(n)
        po, jo = oracle.list_nodes(n)
        assert np.array_equal(pi, po) and np.array_equal(js, jo)


def test_partition_rows_equal_nnz(lib, fx):
    import polee_b200 as pb
    sample = pb.RNASeqSample(fx.m, fx.n, fx.colptr, fx.rowval, fx.nzval, fx.efflens)
    rows = np.bincount(fx.rowval - 1, minlength=fx.m)
    for parts in (1, 2, 4, 8):
        b = pb.partition_rows(sample, parts)
        assert b[0] == 0 and b[-1] == fx.m and np.all(np.diff(b) > 0)
        per = np.add.reduceat(rows, b[:-1])
        assert per.sum() == len(fx.rowval) and per.max() - per.min() <= 2 * rows.max()
        blocks = [pb.api.row_block(sample, int(b[i]), int(b[i + 1])) for i in range(parts)]
        assert sum(len(s.rowval) for s in blocks) == len(fx.rowval)
        assert all(s.rowval.min() == 1 and s.rowval.max() == s.m for s in blocks)


def test_synthetic_generator_invariants(small_synth, oracle):
    s = small_synth
    m, n = s["m"], s["n"]
    colptr, rowval, nzval = s["colptr"], s["rowval"], s["nzval"]
    assert colptr[0] == 1 and colptr[-1] == len(rowval) + 1 and np.all(np.diff(colptr.astype(np.int64)) >= 0)
    col_of = np.repeat(np.arange(n), np.diff(colptr.astype(np.int64)))
    key = col_of.astype(np.int64) * (m + 1) + rowval
    assert np.all(np.diff(key) > 0)                                   # sorted, no duplicate (row, col)
    rows = np.bincount(rowval - 1, minlength=m)
    assert rows.min() >= 1 and 3.0 < rows.mean() < 5.5                # every row non-empty, mean length ~ 4
    assert nzval.min() > 1e-12 and nzval.dtype == np.float32          # MIN_FRAG_PROB floor (constants.jl:45)
    assert s["efflens"].min() >= 1.0
    pi, js = s["tree"]
    t = oracle.PTT(pi, js)                                            # valid DFS tree: transform sums to one
    x, _ = t.transform(np.full(n - 1, 0.37))
    assert abs(x.astype(np.float64).sum() - 1.0) < 1e-5
    assert sorted(js[js > 0].tolist()) == list(range(1, n + 1))


def test_tree_builders_follow_the_dfs_contract(oracle):
    """SURVEY App. B: node 1 is the root, parent < child, right child = idx + 1, subtrees contiguous."""
    from polee_b200 import synth
    for pi, js in (synth.random_tree(200, 1), synth.balanced_tree(77), synth.balanced_tree(10, [3, 1, 6])):
        N = len(js)
        assert pi[0] == 0 and np.all(pi[1:] < np.arange(2, N + 1))
        idx = oracle.PTT(pi, js).index()
        internal = np.nonzero(idx[0] == 0)[0]
        assert np.all(idx[2, internal] == internal + 2)


def test_julia_glue_binds_only_exported_symbols():
    from polee_b200 import _lib
    src = open(os.path.join(ROOT, "julia", "PoleeB200.jl")).read()
    used = set(re.findall(r":(polee_[a-z0-9_]+)", src))
    assert used and used <= set(_lib.EXPORTS), used - set(_lib.EXPORTS)


def test_opts_struct_layout_matches_header_in_python_and_julia():
    header = open(os.path.join(ROOT, "include", "polee_b200.h")).read()
    body = re.search(r"typedef struct polee_opts \{(.*?)\} polee_opts;", header, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = re.findall(r"(int32_t|uint64_t|double)\s+(\w+);", body)
    from polee_b200 import _lib
    py = [(n, t) for n, t in _lib.PoleeOpts._fields_]
    cmap = {"int32_t": C.c_int32, "uint64_t": C.c_uint64, "double": C.c_double}
    assert [(n, cmap[t]) for t, n in fields] == py
    jl = open(os.path.join(ROOT, "julia", "PoleeB200.jl")).read()
    jbody = re.search(r"mutable struct PoleeOpts(.*?)PoleeOpts\(\) = new\(\)", jl, flags=re.S).group(1)
    jfields = re.findall(r"(\w+)::(Int32|UInt64|Float64)", jbody)
    jmap = {"int32_t": "Int32", "uint64_t": "UInt64", "double": "Float64"}
    assert [(n, jmap[t]) for t, n in fields] == jfields


class _H5Image:
    """An HDF5 file laid out the way libhdf5 (through HDF5.jl) lays out the reference's test/dataset/*.h5, built byte by
    byte from the format specification: superblock v0, v1 object headers (optionally split by a continuation block),
    new-style groups (link messages in the object header, or dense storage in a fractal heap), contiguous scalars,
    chunked + deflate arrays indexed by a v1 B-tree of two levels.  write_prep emits none of these group and array
    encodings, so only this image exercises the reader paths those files take.  Checksums are left zero and the name
    index of a dense group is left undefined: the reader uses neither."""

    def __init__(self):
        from polee_b200 import h5min
        self.h5, self.f = h5min, h5min._File()

    def header(self, msgs, split=None):
        """v1 object header of (type, body) messages; from index `split` on they go to a continuation block"""
        import struct
        enc = [self.h5._msg(t, b) for t, b in msgs]
        if split is None:
            return self.f.append(self.h5._object_header(enc))
        rest = b"".join(enc[split:])
        head = b"".join(enc[:split]) + self.h5._msg(0x10, struct.pack("<QQ", self.f.append(rest), len(rest)))
        return self.f.append(struct.pack("<BBHII4x", 1, 0, len(enc) + 1, 1, len(head)) + head)

    def scalar(self, v):
        return self.f.dataset(np.int64(v))

    def chunked(self, arr, chunk, fanout=4, split=None):
        """1-D dataset in deflate-compressed chunks of `chunk` elements (the last one stored whole, zero padded)"""
        import struct
        import zlib
        arr = np.ascontiguousarray(arr)
        leaves = []
        for off in range(0, len(arr), chunk):
            part = np.zeros(chunk, arr.dtype)
            part[:len(arr) - off] = arr[off:off + chunk]
            z = zlib.compress(part.tobytes(), 6)
            leaves.append((len(z), off, self.f.append(z)))

        def node(level, entries):   # entries: (bytes of the first chunk below, its element offset, child address)
            b = b"TREE" + struct.pack("<BBHQQ", 1, level, len(entries), self.h5.UNDEF, self.h5.UNDEF)
            for nbytes, off, child in entries:
                b += struct.pack("<IIQQQ", nbytes, 0, off, 0, child)
            return self.f.append(b + struct.pack("<IIQQ", 0, 0, len(arr), 0))

        level0 = [leaves[i][:2] + (node(0, leaves[i:i + fanout]),) for i in range(0, len(leaves), fanout)]
        root = node(1, level0) if len(level0) > 1 else level0[0][2]
        deflate = struct.pack("<BB6x", 1, 1) + struct.pack("<HHHHI4x", 1, 0, 0, 1, 6)   # filter 1, level 6
        msgs = [(0x01, self.h5._dataspace_msg(arr.shape)), (0x03, self.h5._dtype_msg(arr.dtype)),
                (0x05, struct.pack("<BBBB", 2, 2, 2, 0)), (0x0B, deflate),
                (0x08, struct.pack("<BBBQII", 3, 2, 2, root, chunk, arr.dtype.itemsize))]
        return self.header(msgs, split)

    @staticmethod
    def link(name, addr, flags=0x10):
        """link message v1 to a hard link; flags 0x10: UTF-8 character set field (what HDF5.jl asks for), 0x04:
        creation order field"""
        import struct
        b = struct.pack("<BB", 1, flags) + (b"\0" * 8 if flags & 0x04 else b"") + (b"\x01" if flags & 0x10 else b"")
        return b + struct.pack("<B", len(name)) + name.encode() + struct.pack("<Q", addr)

    def compact_group(self, links, split=None):
        import struct
        u = self.h5.UNDEF
        msgs = [(0x02, struct.pack("<BBQQ", 0, 0, u, u)), (0x0A, b"\0\0")]
        msgs += [(0x06, self.link(k, a, 0x14 if i % 2 else 0x10)) for i, (k, a) in enumerate(links.items())]
        return self.header(msgs, split)

    def dense_group(self, links):
        """links as managed objects of a fractal heap whose root is one direct block"""
        import struct
        u = self.h5.UNDEF
        objs = b"".join(self.link(k, a) for k, a in links.items())
        size = 512
        while size < len(objs) + 21:
            size *= 2
        dblock = self.f.append(b"FHDB" + struct.pack("<BQI", 0, 0, 0) + objs.ljust(size - 21, b"\0") + b"\0" * 4)
        frhp = self.f.append(b"FRHP" + struct.pack("<BHHBIQQQQQQQQQQQQ", 0, 7, 0, 0x02, 4096, 0, u, size - 21 - len(objs),
                                                   u, size, size, size, len(links), 0, 0, 0, 0)
                             + struct.pack("<HQQHHQH", 4, size, 65536, 32, 1, dblock, 0) + b"\0" * 4)
        self.f.buf[dblock + 5:dblock + 13] = struct.pack("<Q", frhp)                  # the block's heap header
        return self.header([(0x02, struct.pack("<BBQQ", 0, 0, frhp, u)), (0x0A, b"\0\0")])

    def write(self, path, root):
        """superblock v0 whose root symbol table entry caches nothing (a new-style root group)"""
        import struct
        f = self.f
        f.buf += b"\0" * (-len(f.buf) % 8)
        sb = self.h5.SIGNATURE + struct.pack("<BBBBBBBBHHI", 0, 0, 0, 0, 0, 8, 8, 0, 4, 16, 0)
        sb += struct.pack("<QQQQ", 0, self.h5.UNDEF, len(f.buf), self.h5.UNDEF) + struct.pack("<QQII16x", 0, root, 0, 0)
        f.buf[:96] = sb
        with open(path, "wb") as fh:
            fh.write(bytes(f.buf))
        return bytes(f.buf)


def test_h5min_prep_roundtrip_and_reference_files(tmp_path):
    """SURVEY 8f-3: the harness-side reader/writer of Polee's two HDF5 formats.  write_prep -> read_prep round trip
    (the file write_approximation produces, likelihood-approximation.jl:61-87), structural checks on the bytes, and
    the reference fixture (tests/golden) in files laid out as the reference's own test/dataset/*.h5 (_H5Image) decodes
    to the committed golden arrays: the likelihood matrix with link messages in the root group, chunked + deflate
    arrays and a continuation block, the prep file with its root group in a fractal heap."""
    import struct
    from polee_b200 import h5min
    rng = np.random.default_rng(1)
    n, m = 313, 19743
    params = {"mu": rng.normal(size=n - 1).astype(np.float32), "omega": rng.normal(size=n - 1).astype(np.float32),
              "alpha": rng.normal(size=n - 1).astype(np.float32),
              "node_parent_idxs": rng.integers(0, 2 * n - 1, 2 * n - 1).astype(np.int32),
              "node_js": rng.integers(0, n, 2 * n - 1).astype(np.int32)}
    eff = rng.uniform(1, 5000, n).astype(np.float32)
    path = str(tmp_path / "x.prep.h5")
    size = h5min.write_prep(path, params, n, m, eff, gfffilename="genes.gff3", gffhash="q83vEjRWeJA=", date="2026-10-17",
                            args="prep-sample a b")
    raw = open(path, "rb").read()
    assert len(raw) == size and raw[:8] == b"\x89HDF\r\n\x1a\n" and raw[8] == 0 and raw[13] == 8 and raw[14] == 8
    assert struct.unpack_from("<Q", raw, 40)[0] == size                        # end-of-file address
    back = h5min.read_prep(path)
    assert back["n"] == n and back["m"] == m and back["n"].dtype == np.int64
    assert np.array_equal(back["effective_lengths"], eff)
    for k, v in params.items():
        assert back[k].dtype == v.dtype and np.array_equal(back[k], v)
    md = back["metadata"]
    assert md["version"] == 2 and md["approximation"] == "Polee.LogitSkewNormalPTTApprox"
    assert md["gfffilename"] == "genes.gff3" and md["gffhash"] == "q83vEjRWeJA=" and md["args"] == "prep-sample a b"
    fx = Fixture()
    img = _H5Image()
    links = {"m": img.scalar(fx.m), "n": img.scalar(fx.n), "colptr": img.chunked(fx.colptr, 64),
             "rowval": img.chunked(fx.rowval, 4096, split=3), "nzval": img.chunked(fx.nzval, 4096),
             "effective_lengths": img.chunked(fx.efflens, 313)}
    raw = img.write(str(tmp_path / "lm.h5"), img.compact_group(links, split=4))
    assert raw.count(b"TREE\x01\x01") == 3 and raw.count(b"TREE\x01\x00") == 9         # two-level chunk indexes
    lm = h5min.read_likelihood_matrix(str(tmp_path / "lm.h5"))
    assert (lm["m"], lm["n"]) == (fx.m, fx.n) and np.array_equal(lm["colptr"], fx.colptr)
    assert np.array_equal(lm["rowval"], fx.rowval) and np.array_equal(lm["nzval"], fx.nzval)
    assert np.array_equal(lm["effective_lengths"], fx.efflens)
    img = _H5Image()
    links = {"n": img.scalar(fx.n), "m": img.scalar(fx.m), "effective_lengths": img.chunked(fx.efflens, 100),
             "mu": img.chunked(fx.mu, 128, split=2), "omega": img.chunked(fx.omega, 128),
             "alpha": img.chunked(fx.alpha, 128), "node_parent_idxs": img.chunked(fx.parent_idxs, 256),
             "node_js": img.chunked(fx.js, 256), "metadata": img.compact_group({})}
    raw = img.write(str(tmp_path / "pp.h5"), img.dense_group(links))
    assert b"FHDB" in raw and b"FRHP" in raw
    pp = h5min.read_prep(str(tmp_path / "pp.h5"))
    assert np.array_equal(pp["mu"], fx.mu) and np.array_equal(pp["node_js"], fx.js) and pp["n"] == fx.n
    assert np.array_equal(pp["omega"], fx.omega) and np.array_equal(pp["alpha"], fx.alpha)
    assert np.array_equal(pp["node_parent_idxs"], fx.parent_idxs) and pp["m"] == fx.m
    assert np.array_equal(pp["effective_lengths"], fx.efflens) and pp["metadata"] == {}


def test_hclust_host_restatement(oracle):
    """SURVEY 8f-4: polee_hclust (C++ host code behind the C ABI, no GPU) against the independent Python restatement of
    hclust + order_nodes (src/hclust.jl:193-319, 361-389) under the same explicit tie policy: identical trees; the
    tree is a valid PolyaTreeTransform input (every transcript once, DFS order, right branch first); transcripts that
    share reads end up closer in the tree than transcripts that do not."""
    import polee_b200 as pb
    from polee_b200 import synth
    fx = Fixture()
    cases = [(fx.m, fx.n, fx.colptr, fx.rowval)]
    s = synth.to_numpy_sample(synth.make_sample(6000, 400, seed=3))
    cases.append((s["m"], s["n"], s["colptr"], s["rowval"]))
    for m, n, colptr, rowval in cases:
        smp = pb.RNASeqSample(m, n, colptr, rowval, np.ones(len(rowval), np.float32), np.ones(n, np.float32))
        pi, js = pb.hclust(smp)
        pi_o, js_o = oracle.hclust_tree(m, n, colptr, rowval)
        assert np.array_equal(pi, pi_o) and np.array_equal(js, js_o)
        N = 2 * n - 1
        assert pi[0] == 0 and np.all(pi[1:] >= 1) and np.all(pi[1:] < np.arange(2, N + 1))      # parents precede children
        assert sorted(js[js > 0]) == list(range(1, n + 1)) and (js == 0).sum() == n - 1
        kids = np.bincount(pi[1:], minlength=N + 1)
        assert np.all(kids[1:][js == 0] == 2) and np.all(kids[1:][js > 0] == 0)
        t = oracle.PTT(pi, js)                                                                  # the reference's constructor rule
        assert t.n == n
    # degenerate inputs: a single transcript, two transcripts, empty columns (transcripts without compatible reads end up
    # in the "remainder" joins, hclust.jl:243-262)
    def mk(m, n, cols):
        colptr, rowval = [1], []
        for c in cols:
            rowval += sorted(c)
            colptr.append(len(rowval) + 1)
        return pb.RNASeqSample(m, n, np.array(colptr, np.uint32), np.array(rowval, np.uint32),
                               np.ones(len(rowval), np.float32), np.ones(n, np.float32))
    for smp in (mk(3, 1, [[1, 2, 3]]), mk(3, 2, [[1, 2], [2, 3]]), mk(4, 5, [[1, 2], [], [2, 3], [], [4]]),
                mk(2, 3, [[], [1, 2], []])):
        pi2, js2 = pb.hclust(smp)
        po, jo = oracle.hclust_tree(smp.m, smp.n, smp.colptr, smp.rowval)
        assert np.array_equal(pi2, po) and np.array_equal(js2, jo)
        assert sorted(js2[js2 > 0]) == list(range(1, smp.n + 1)) and pi2[0] == 0
    # the two isoforms sharing the most reads in the fixture are siblings or cousins: tree distance <= 4
    depth = np.zeros(len(pi) + 1, int)
    for i in range(2, len(pi) + 1):
        depth[i] = depth[pi[i - 1]] + 1
    import scipy.sparse as sp
    X = sp.csc_matrix((np.ones(len(rowval)), rowval.astype(np.int64) - 1, colptr.astype(np.int64) - 1), shape=(m, n))
    G = (X.T @ X).toarray().astype(float)
    sz = np.diag(G).copy()
    np.fill_diagonal(G, 0)
    a, b = np.unravel_index(np.argmax(G / (sz[:, None] + sz[None, :] - G + 1e-9)), G.shape)
    pos = {int(j): i + 1 for i, j in enumerate(js) if j > 0}

    def ancestors(i):
        out = []
        while i:
            out.append(i)
            i = pi[i - 1]
        return out
    A, B = ancestors(pos[a + 1]), ancestors(pos[b + 1])
    common = next(x for x in A if x in B)
    assert (A.index(common) + B.index(common)) <= 4


def test_speculative_replay_of_a_float32_accumulator_is_exact():
    """The algorithm of k4_ladj_chain (hsb_ops.cu), restated in numpy: InvHSB's `ladj -= log(u)` is a Float32
    accumulator fed with Float64 terms (src/tensorflow_ext/hsb_ops.cpp:211,234), i.e. a chain of roundings
    acc <- Float32(Float64(acc) - l).  While acc stays in one binade a step moves it by rint(-l / ulp) ulps whatever acc
    is, so a block of steps can be formed by a prefix sum and then VERIFIED step by step with the reference's own rule;
    the steps before the first mismatch are exact by induction, the mismatching one is redone by the scalar rule.
    Checked here against the plain serial loop, bit for bit, on data with binade crossings, ties, zeros, sign changes
    and non-finite values."""
    def serial(ls):
        acc = np.float32(0)
        for l in ls:
            acc = np.float32(np.float64(acc) - l)
        return acc

    def speculative(ls, width=256):
        acc, k, scalar_steps = np.float32(0), 0, 0
        with np.errstate(all="ignore"):
            while k < len(ls):
                l = ls[k:k + width]
                fin = acc != 0 and np.isfinite(acc)
                e = np.frexp(np.abs(acc))[1] if fin else 0
                ulp, inv_ulp = (np.ldexp(1.0, e - 24), np.ldexp(1.0, 24 - e)) if fin else (0.0, 0.0)
                P = np.cumsum(np.rint(-l * inv_ulp))
                cand = (np.float64(acc) + ulp * P).astype(np.float32)
                pred = np.concatenate([[acc], cand[:-1]]).astype(np.float32)
                ok = (pred.astype(np.float64) - l).astype(np.float32) == cand
                f = len(l) if ok.all() else int(np.argmin(ok))
                if f > 0:
                    acc = cand[f - 1]
                if f < len(l):
                    acc = np.float32(np.float64(acc) - l[f])
                    scalar_steps += 1
                    f += 1
                k += f
        return acc, scalar_steps

    rng = np.random.default_rng(11)
    cases = {
        "log u of a simplex (what InvHSB feeds it)": np.log(rng.dirichlet(np.ones(20000) * 0.3).clip(1e-300)),
        "mixed signs and magnitudes": rng.normal(size=5000) * 10.0 ** rng.integers(-12, 6, 5000),
        "ties: multiples of half an ulp": np.ldexp(rng.integers(-8, 9, 4000).astype(np.float64), -20) + 0.0,
        "zeros and tiny terms": np.where(rng.random(3000) < 0.5, 0.0, rng.normal(size=3000) * 1e-30),
        "an infinity in the middle": np.concatenate([rng.normal(size=300), [-np.inf], rng.normal(size=300)]),
    }
    for name, ls in cases.items():
        ls = np.ascontiguousarray(ls, np.float64)
        with np.errstate(all="ignore"):
            want = serial(ls)
        got, scalar_steps = speculative(ls)
        assert want.tobytes() == got.tobytes() or (np.isnan(want) and np.isnan(got)), name
        if name.startswith("log u"):
            assert scalar_steps < 200, scalar_steps   # binade changes and the first steps only: ~80 x fewer chain steps
