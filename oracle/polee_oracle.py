"""ctypes binding of the test oracle (oracle/libpolee_oracle.so, oracle/_ref/libref_hsb_ops.so).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  Nothing under polee_b200/ may import this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libpolee_oracle.so")
_REF = os.path.join(_HERE, "_ref", "libref_hsb_ops.so")

c_i64, c_u64, c_int, c_dbl = C.c_int64, C.c_uint64, C.c_int, C.c_double
P = C.c_void_p


def build(force=False, reference=None):
    """(Re)build the oracle; oracle/_ref only when `reference` names a checkout of the original Polee."""
    if force or not os.path.exists(_LIB) or \
            os.path.getmtime(_LIB) < os.path.getmtime(os.path.join(_HERE, "polee_oracle.c")):
        subprocess.check_call(["make", "-s", "-C", _HERE, "liboracle"])
    if reference and (force or not os.path.exists(_REF)):
        subprocess.check_call(["make", "-s", "-C", _HERE, "ref", "REFERENCE=" + os.path.abspath(reference)])


class OrcFitOpts(C.Structure):
    _fields_ = [("num_steps", c_int), ("num_mc_samples", c_int), ("gradonly", c_int),
                ("use_efflen_jacobian", c_int), ("seed", c_u64), ("noise", P), ("elbo_fix", c_int), ("genes", P)]


class OrcGenes(C.Structure):
    _fields_ = [("num_genes", c_i64), ("gene_ptr", P), ("transcripts", P)]


def make_genes(gene_transcripts):
    """{gene: [1-based transcript ids]} (or a list of id lists) -> (OrcGenes, keep-alive arrays); None -> (None, ())"""
    if not gene_transcripts:
        return None, ()
    groups = list(gene_transcripts.values()) if hasattr(gene_transcripts, "values") else list(gene_transcripts)
    ptr = np.zeros(len(groups) + 1, np.int64)
    ptr[1:] = np.cumsum([len(g) for g in groups])
    tx = np.ascontiguousarray(np.concatenate([np.asarray(g, np.int32) for g in groups]), np.int32)
    return OrcGenes(len(groups), _p(ptr), _p(tx)), (ptr, tx)


_lib = None
_ref = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB)
        _lib.orc_log_likelihood.restype = c_dbl
        _lib.orc_factored_log_likelihood.restype = c_dbl
        _lib.orc_effective_length_jacobian_adjustment.restype = c_dbl
        _lib.orc_ptt_new.restype = P
        _lib.orc_ptt_index.restype = P
        _lib.orc_ptt_transform.restype = c_dbl
        _lib.orc_ptt_inverse_transform.restype = c_dbl
        _lib.orc_sinh_asinh_transform.restype = c_dbl
        _lib.orc_logit_normal_transform.restype = c_dbl
        _lib.orc_fit_begin.restype = P
        _lib.orc_adam_learning_rate.restype = c_dbl
        _lib.orc_lsn_draw.restype = c_dbl
        _lib.orc_lsn_draw_genes.restype = c_dbl
    return _lib


def ref_lib():
    """The reference's own hsb_ops.cpp (compiled over the TF stub); None if not built."""
    global _ref
    if _ref is None and os.path.exists(_REF):
        _ref = C.CDLL(_REF)
    return _ref


def _p(a):
    return None if a is None else a.ctypes.data_as(P)


def _c(a, dt):
    return np.ascontiguousarray(a, dtype=dt)


def num_threads():
    return lib().orc_num_threads()


def set_num_threads(n=None):
    """Use n OpenMP threads (default: every core this process may run on -- the reference's wrapper script starts
    Julia with all cores, polee:8-12; torch.distributed.run would otherwise pin OMP_NUM_THREADS to 1)."""
    if n is None:
        try:
            n = len(os.sched_getaffinity(0))
        except AttributeError:
            n = os.cpu_count() or 1
    lib().orc_set_num_threads(C.c_int(int(n)))
    return num_threads()


# ------------------------------------------------------------------ sparse / likelihood
def transpose_csc(m, n, colptr, rowval, nzval):
    nnz = len(rowval)
    tc = np.empty(m + 1, np.uint32); tr = np.empty(max(nnz, 1), np.uint32); tv = np.empty(max(nnz, 1), np.float32)
    lib().orc_transpose_csc(c_i64(m), c_i64(n), _p(colptr), _p(rowval), _p(nzval), _p(tc), _p(tr), _p(tv))
    return tc, tr[:nnz], tv[:nnz]


class Model:
    """Model(m, n) + X + Xt (likelihood.jl:2-18, likelihood-approximation.jl:406-408)."""

    def __init__(self, m, n, colptr, rowval, nzval):
        self.m, self.n = int(m), int(n)
        self.colptr = _c(colptr, np.uint32); self.rowval = _c(rowval, np.uint32); self.nzval = _c(nzval, np.float32)
        self.t_colptr, self.t_rowval, self.t_nzval = transpose_csc(self.m, self.n, self.colptr, self.rowval, self.nzval)
        self.frag_probs = np.zeros(self.m, np.float64)
        self.log_frag_probs = np.zeros(self.m, np.float64)

    def log_likelihood(self, xs, gradonly=True, ks=None):
        xs = _c(xs, np.float32)
        x_grad = np.zeros(self.n, np.float64)
        args = [c_i64(self.m), c_i64(self.n), _p(self.frag_probs), _p(self.log_frag_probs), _p(self.colptr),
                _p(self.rowval), _p(self.nzval), _p(self.t_colptr), _p(self.t_rowval), _p(self.t_nzval)]
        if ks is None:
            lp = lib().orc_log_likelihood(*args, _p(xs), _p(x_grad), c_int(int(gradonly)))
        else:
            ks = _c(ks, np.int64)
            lp = lib().orc_factored_log_likelihood(*args, _p(ks), _p(xs), _p(x_grad), c_int(int(gradonly)))
        return lp, x_grad


def effective_length_jacobian_adjustment(efflens, xs, x_grad):
    efflens = _c(efflens, np.float32); xs = _c(xs, np.float32)
    xls = np.empty_like(xs)
    lib().orc_effective_length_jacobian_adjustment(c_i64(len(xs)), _p(efflens), _p(xs), _p(xls), _p(x_grad))
    return xls


def gene_noninformative_prior(efflens, xls, xs, x_grad, gene_transcripts):
    """likelihood.jl:114-159; adds to x_grad in place, returns xl_grad"""
    efflens = _c(efflens, np.float32); xs = _c(xs, np.float32); xls = _c(xls, np.float32)
    genes, _keep = make_genes(gene_transcripts)
    xl_grad = np.zeros(len(xs), np.float64)
    lib().orc_gene_noninformative_prior(c_i64(len(xs)), _p(efflens), _p(xls), _p(xl_grad), _p(xs), _p(x_grad),
                                        C.byref(genes))
    return xl_grad


def exact_factorization(m, n, colptr, rowval, nzval):
    """tools/exact-factorization.jl:31-68: one copy of every distinct row (transcript ids + Float32 values, compared
    bit for bit) and its multiplicity.  The reference numbers the unique rows in the iteration order of a Julia Dict
    (unspecified); here, and in the device implementation, by first occurrence.  Returns (m_unique, colptr, rowval,
    nzval, counts) with 1-based UInt32 CSC arrays like the input."""
    colptr = np.asarray(colptr, np.int64); rowval = np.asarray(rowval, np.int64); nzval = _c(nzval, np.float32)
    nnz = len(rowval)
    col_of = np.repeat(np.arange(n, dtype=np.int64), np.diff(colptr))
    order = np.argsort(rowval, kind="stable")                      # Xt = transpose(X): row-major, ascending transcript
    rptr = np.zeros(m + 1, np.int64)
    np.add.at(rptr, rowval, 1)
    rptr = np.cumsum(rptr)
    cols_r, vals_r = col_of[order], nzval[order]
    seen, uidx, counts = {}, np.zeros(m, np.int64), []
    for i in range(m):
        a, b = rptr[i], rptr[i + 1]
        key = (cols_r[a:b].tobytes(), vals_r[a:b].tobytes())       # :38-40
        u = seen.get(key)
        if u is None:
            u = seen[key] = len(counts)
            counts.append(0)
            uidx[i] = u + 1
        counts[u] += 1
    keep = uidx[rowval - 1] > 0                                    # the first occurrences' entries, CSC order kept
    new_rowval = uidx[rowval - 1][keep].astype(np.uint32)
    new_nzval = nzval[keep]
    cnt = np.zeros(n, np.int64)
    np.add.at(cnt, col_of[keep], 1)
    new_colptr = np.concatenate([[1], 1 + np.cumsum(cnt)]).astype(np.uint32)
    return len(counts), new_colptr, new_rowval, new_nzval, np.asarray(counts, np.int64)


def hclust_tree(m, n, colptr, rowval):
    """PolyaTreeTransform(X, :cluster): hclust + order_nodes (src/hclust.jl:193-319, 361-389) restated with heapq and
    numpy set operations.  Tie policy (unpinned in the reference, SURVEY 8c): equal Float32 similarities -> smaller
    (j1, j2) first; equal sizes in the remainder queue -> smaller node id first; neighbour lists keep first
    occurrences.  Returns (node_parent_idxs, node_js), 1-based, DFS order with the right branch first."""
    import heapq
    colptr = np.asarray(colptr, np.int64); rowval = np.asarray(rowval, np.uint32)
    K = 25
    med = np.zeros(n, np.uint32)
    for j in range(n):
        if colptr[j] != colptr[j + 1]:
            med[j] = rowval[(colptr[j] + colptr[j + 1]) // 2 - 1]
    idxs = np.argsort(med, kind="stable")
    N = 2 * n - 1
    sets = [None] * N
    left = [-1] * N; right = [-1] * N; leaf_tx = [0] * N
    dead = [False] * N; live = [False] * N
    nbr = [[] for _ in range(N)]
    for j in range(n):
        t = idxs[j]
        sets[j] = rowval[colptr[t] - 1:colptr[t + 1] - 1]
        leaf_tx[j] = int(t) + 1
        live[j] = True

    def jaccard(a, b):
        if len(a) == 0 and len(b) == 0:
            return np.float32(0)
        c = len(np.intersect1d(a, b, assume_unique=True))
        return np.float32(c / (len(a) + len(b) - c))

    def add_nbr(a, b):
        if b not in nbr[a]:
            nbr[a].append(b)

    heap = []
    for j1 in range(n):
        for j2 in range(j1 + 1, min(j1 + K, n - 1) + 1):
            s = jaccard(sets[j1], sets[j2])
            if s > 0:
                heapq.heappush(heap, (-float(s), j1, j2))
            add_nbr(j1, j2); add_nbr(j2, j1)
    nxt = n
    while heap:
        _, j1, j2 = heapq.heappop(heap)
        if dead[j1] or dead[j2]:
            continue
        k = nxt; nxt += 1
        sets[k] = np.union1d(sets[j1], sets[j2])
        left[k], right[k], live[k] = j1, j2, True
        for j in (j1, j2):
            sets[j] = None; dead[j] = True; live[j] = False
        for ja, jb in ((j1, j2), (j2, j1)):
            lst, nbr[ja] = nbr[ja], []
            for l in lst:
                if l == jb or dead[l]:
                    continue
                s = jaccard(sets[l], sets[k])
                if s != 0:
                    heapq.heappush(heap, (-float(s), l, k))
                add_nbr(l, k); add_nbr(k, l)
    rest = [(1 + len(sets[j]), j) for j in range(nxt) if live[j]]
    heapq.heapify(rest)
    while len(rest) > 1:
        a = heapq.heappop(rest); b = heapq.heappop(rest)
        k = nxt; nxt += 1
        left[k], right[k] = a[1], b[1]
        heapq.heappush(rest, (a[0] + b[0], k))
    assert nxt == N
    parent_idxs = np.zeros(N, np.int32); js = np.zeros(N, np.int32)
    parent_of = [0] * N
    stack, pos = [rest[0][1]], 0
    while stack:
        v = stack.pop()
        parent_idxs[pos] = parent_of[v]
        js[pos] = leaf_tx[v] if left[v] < 0 else 0
        pos += 1
        if left[v] >= 0:
            parent_of[left[v]] = parent_of[right[v]] = pos
            stack.append(left[v]); stack.append(right[v])
    return parent_idxs, js


# ------------------------------------------------------------------ ptt
class PTT:
    def __init__(self, parent_idxs, js):
        self.parent_idxs = _c(parent_idxs, np.int32); self.js = _c(js, np.int32)
        self.N = len(self.js); self.n = (self.N + 1) // 2
        self.h = lib().orc_ptt_new(_p(self.parent_idxs), _p(self.js), c_i64(self.N))

    def __del__(self):
        try:
            if getattr(self, "h", None):
                lib().orc_ptt_free(P(self.h)); self.h = None
        except Exception:  # interpreter shutdown
            pass

    def index(self):
        buf = (C.c_int32 * (4 * self.N)).from_address(lib().orc_ptt_index(P(self.h)))
        return np.frombuffer(buf, np.int32).reshape(self.N, 4).T.copy()  # 4 x N like Julia

    def transform(self, ys, compute_ladj=False):
        ys = _c(ys, np.float64); xs = np.zeros(self.n, np.float32)
        ladj = lib().orc_ptt_transform(P(self.h), _p(ys), _p(xs), c_int(int(compute_ladj)))
        return xs, ladj

    def transform_gradients(self, ys, x_grad):
        ys = _c(ys, np.float64); x_grad = _c(x_grad, np.float64); y_grad = np.zeros(self.n - 1, np.float32)
        lib().orc_ptt_transform_gradients(P(self.h), _p(ys), _p(y_grad), _p(x_grad))
        return y_grad

    def transform_gradients_no_ladj(self, ys, x_grad):
        ys = _c(ys, np.float64); x_grad = _c(x_grad, np.float64); y_grad = np.zeros(self.n - 1, np.float64)
        lib().orc_ptt_transform_gradients_no_ladj(P(self.h), _p(ys), _p(y_grad), _p(x_grad))
        return y_grad

    def inverse_transform(self, xs):
        xs = _c(xs, np.float32); ys = np.zeros(self.n - 1, np.float64)
        ladj = lib().orc_ptt_inverse_transform(P(self.h), _p(xs), _p(ys))
        return ys, ladj


def make_inverse_ptt_params(parent_idxs, js):
    parent_idxs = _c(parent_idxs, np.int32); js = _c(js, np.int32); N = len(js)
    l = np.empty(N, np.int32); r = np.empty(N, np.int32); f = np.empty(N, np.int32)
    lib().orc_make_inverse_ptt_params(_p(parent_idxs), _p(js), c_i64(N), _p(l), _p(r), _p(f))
    return l, r, f


def list_nodes(n):
    N = 2 * n - 1
    p = np.empty(N, np.int32); j = np.empty(N, np.int32)
    lib().orc_list_nodes(c_i64(n), _p(p), _p(j))
    return p, j


# ------------------------------------------------------------------ noise / fits
def noise_fill(seed, step, draw, nm1):
    z = np.empty(nm1, np.float32)
    lib().orc_noise_fill(c_u64(seed), c_i64(step), c_i64(draw), c_i64(nm1), _p(z))
    return z


def fit_lsn_ptt(m, n, colptr, rowval, nzval, efflens, parent_idxs, js, ks=None, num_steps=500, num_mc_samples=6,
                gradonly=True, use_efflen_jacobian=True, seed=0, noise=None, elbo_fix=False, gene_transcripts=None):
    genes, _keep = make_genes(gene_transcripts)
    colptr = _c(colptr, np.uint32); rowval = _c(rowval, np.uint32); nzval = _c(nzval, np.float32)
    efflens = _c(efflens, np.float32); parent_idxs = _c(parent_idxs, np.int32); js = _c(js, np.int32)
    if ks is not None:
        ks = _c(ks, np.int64)
    if noise is not None:
        noise = _c(noise, np.float32)
        assert noise.size == num_steps * num_mc_samples * (n - 1)
    o = OrcFitOpts(num_steps, num_mc_samples, int(gradonly), int(use_efflen_jacobian), seed, _p(noise), int(elbo_fix),
                   C.cast(C.pointer(genes), P) if genes is not None else None)
    mu = np.zeros(n - 1, np.float32); omega = np.zeros(n - 1, np.float32); alpha = np.zeros(n - 1, np.float32)
    elbo = np.zeros(num_steps, np.float64)
    st = lib().orc_fit_lsn_ptt(c_i64(m), c_i64(n), _p(colptr), _p(rowval), _p(nzval), _p(ks), _p(efflens),
                               _p(parent_idxs), _p(js), C.byref(o), _p(mu), _p(omega), _p(alpha), _p(elbo))
    if st != 0:
        raise FloatingPointError("non-finite gradient at step %d" % st)
    return {"mu": mu, "omega": omega, "alpha": alpha, "elbo": elbo}


class FitStepper:
    """orc_fit_begin / orc_fit_step: the reference loop one ADAM step at a time (CPU baseline timing)."""

    def __init__(self, m, n, colptr, rowval, nzval, efflens, parent_idxs, js, ks=None, num_mc_samples=6,
                 gradonly=True, use_efflen_jacobian=True, seed=0):
        self.keep = [_c(colptr, np.uint32), _c(rowval, np.uint32), _c(nzval, np.float32), _c(efflens, np.float32),
                     _c(parent_idxs, np.int32), _c(js, np.int32), None if ks is None else _c(ks, np.int64)]
        self.n = n
        o = OrcFitOpts(0, num_mc_samples, int(gradonly), int(use_efflen_jacobian), seed, None, 0, None)
        k = self.keep
        self.s = lib().orc_fit_begin(c_i64(m), c_i64(n), _p(k[0]), _p(k[1]), _p(k[2]), _p(k[6]), _p(k[3]), _p(k[4]),
                                     _p(k[5]), C.byref(o))

    def step(self):
        st = lib().orc_fit_step(P(self.s))
        if st != 0:
            raise FloatingPointError("non-finite gradient at step %d" % st)

    def params(self):
        mu = np.zeros(self.n - 1, np.float32); om = np.zeros_like(mu); al = np.zeros_like(mu)
        lib().orc_fit_params(P(self.s), _p(mu), _p(om), _p(al))
        return mu, om, al

    def close(self):
        if self.s:
            lib().orc_fit_end(P(self.s)); self.s = None


def lsn_draw(m, n, colptr, rowval, nzval, efflens, parent_idxs, js, mu, omega, alpha, zs0, ks=None, gradonly=True,
             use_efflen_jacobian=True, gene_transcripts=None):
    genes, _keep = make_genes(gene_transcripts)
    colptr = _c(colptr, np.uint32); rowval = _c(rowval, np.uint32); nzval = _c(nzval, np.float32)
    efflens = _c(efflens, np.float32); parent_idxs = _c(parent_idxs, np.int32); js = _c(js, np.int32)
    mu = _c(mu, np.float32); omega = _c(omega, np.float32); alpha = _c(alpha, np.float32); zs0 = _c(zs0, np.float32)
    if ks is not None:
        ks = _c(ks, np.int64)
    out = {"xs": np.zeros(n, np.float32), "ys": np.zeros(n - 1, np.float64), "x_grad": np.zeros(n, np.float64),
           "y_grad": np.zeros(n - 1, np.float32), "mu_grad": np.zeros(n - 1, np.float32),
           "omega_grad": np.zeros(n - 1, np.float32), "alpha_grad": np.zeros(n - 1, np.float32)}
    out["elbo"] = lib().orc_lsn_draw_genes(
        c_i64(m), c_i64(n), _p(colptr), _p(rowval), _p(nzval), _p(ks), _p(efflens), _p(parent_idxs), _p(js),
        c_int(int(gradonly)), c_int(int(use_efflen_jacobian)), C.byref(genes) if genes is not None else None,
        _p(mu), _p(omega), _p(alpha), _p(zs0),
        _p(out["xs"]), _p(out["ys"]), _p(out["x_grad"]), _p(out["y_grad"]), _p(out["mu_grad"]),
        _p(out["omega_grad"]), _p(out["alpha_grad"]))
    return out


def fit_optimize_ptt(m, n, colptr, rowval, nzval, efflens, num_steps=500):
    colptr = _c(colptr, np.uint32); rowval = _c(rowval, np.uint32); nzval = _c(nzval, np.float32)
    efflens = _c(efflens, np.float32); xs = np.zeros(n, np.float32)
    lib().orc_fit_optimize_ptt(c_i64(m), c_i64(n), _p(colptr), _p(rowval), _p(nzval), _p(efflens),
                               c_int(num_steps), _p(xs))
    return xs


# ------------------------------------------------------------------ hsb ops
def _hsb_args(B, n, left, right, leaf):
    N = 2 * n - 1
    out = []
    for a in (left, right, leaf):
        a = _c(a, np.int32)
        if a.ndim == 1 or a.shape[0] == 1:
            a = np.ascontiguousarray(np.broadcast_to(a.reshape(1, N), (B, N)))
        out.append(a)
    return out


def hsb(y_logit, left, right, leaf, impl="oracle", threads=1):
    y_logit = _c(y_logit, np.float32); B, nm1 = y_logit.shape; n = nm1 + 1
    l, r, f = _hsb_args(B, n, left, right, leaf)
    x = np.zeros((B, n), np.float32)
    if impl == "oracle":
        lib().orc_hsb(c_i64(B), c_i64(n), _p(y_logit), _p(l), _p(r), _p(f), _p(x))
    else:
        assert ref_lib().ref_hsb(c_i64(B), c_i64(n), _p(y_logit), _p(l), _p(r), _p(f), _p(x), c_int(threads)) == 0
    return x


def inv_hsb(x, left, right, leaf, impl="oracle", threads=1):
    x = _c(x, np.float32); B, n = x.shape
    l, r, f = _hsb_args(B, n, left, right, leaf)
    y = np.zeros((B, n - 1), np.float64); ladj = np.zeros((B, 1), np.float32)
    if impl == "oracle":
        lib().orc_inv_hsb(c_i64(B), c_i64(n), _p(x), _p(l), _p(r), _p(f), _p(y), _p(ladj))
    else:
        assert ref_lib().ref_inv_hsb(c_i64(B), c_i64(n), _p(x), _p(l), _p(r), _p(f), _p(y), _p(ladj), c_int(threads)) == 0
    return y, ladj


def inv_hsb_grad(y_grad, ladj_grad, y, ladj, left, right, leaf, impl="oracle", threads=1):
    y_grad = _c(y_grad, np.float64); y = _c(y, np.float64); B, nm1 = y.shape; n = nm1 + 1
    ladj_grad = _c(ladj_grad, np.float32).reshape(B, 1); ladj = _c(ladj, np.float32).reshape(B, 1)
    l, r, f = _hsb_args(B, n, left, right, leaf)
    bp = np.zeros((B, n), np.float32)
    if impl == "oracle":
        lib().orc_inv_hsb_grad(c_i64(B), c_i64(n), _p(y_grad), _p(ladj_grad), _p(y), _p(l), _p(r), _p(f), _p(bp))
    else:
        assert ref_lib().ref_inv_hsb_grad(c_i64(B), c_i64(n), _p(y_grad), _p(ladj_grad), _p(y), _p(ladj), _p(l),
                                          _p(r), _p(f), _p(bp), c_int(threads)) == 0
    return bp
