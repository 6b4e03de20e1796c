"""Host-side mirror of the reference's Julia interface for the hot path, over libpolee_b200.so.

Names, argument meaning and error behaviour follow the reference (file:line under the reference checkout):

  RNASeqSample                  src/rnaseq_sample.jl:6-23      (only the fields the path reads: m, n, X, effective_lengths)
  PolyaTreeTransform            src/ptt.jl:6-27, 89-116        (+ transform!/transform_gradients!/inverse_transform!)
  LogitSkewNormalPTTApprox      src/likelihood-approximation.jl:13-17
  OptimizePTTApprox             src/likelihood-approximation.jl:8
  approximate_likelihood        src/likelihood-approximation.jl:395-624 (default fit), :248-392 (factored), :149-242
  optimize_likelihood           src/likelihood-approximation.jl:23-25
  log_likelihood                src/likelihood.jl:36-56 (and factored_log_likelihood :59-85 when ks is given)
  make_inverse_ptt_params       src/ptt.jl:293-309
  hsb / inv_hsb / inv_hsb_grad  src/tensorflow_ext/hsb_ops.cpp (the op names src/polee_approx_likelihood.py uses)

Index arrays keep Julia's conventions (1-based UInt32 CSC, 1-based Int32 tree arrays); the library converts on
the device.  Everything computes on the GPU through the C ABI; nothing here is a fallback.
"""
import ctypes as C

import os

import numpy as np

from . import _lib as L

LIKAP_NUM_STEPS = 500        # src/constants.jl:64
LIKAP_NUM_MC_SAMPLES = 6     # src/constants.jl:65

_P = C.c_void_p


def _p(a):
    return None if a is None else a.ctypes.data_as(_P)


def _c(a, dt):
    return np.ascontiguousarray(a, dtype=dt)


class RNASeqSample:
    """The fields of RNASeqSample the likelihood approximation reads (src/rnaseq_sample.jl:6-23).

    X is a SparseMatrixCSC{Float32,UInt32} given by its three arrays (1-based colptr / rowval)."""

    def __init__(self, m, n, colptr, rowval, nzval, effective_lengths):
        self.m, self.n = int(m), int(n)
        self.colptr = _c(colptr, np.uint32)
        self.rowval = _c(rowval, np.uint32)
        self.nzval = _c(nzval, np.float32)
        self.effective_lengths = _c(effective_lengths, np.float32)
        assert self.colptr.shape == (self.n + 1,) and self.effective_lengths.shape == (self.n,)
        assert self.rowval.shape == self.nzval.shape == (int(self.colptr[-1]) - 1,)

    @classmethod
    def from_scipy(cls, X, effective_lengths):
        X = X.tocsc()
        X.sort_indices()
        return cls(X.shape[0], X.shape[1], X.indptr.astype(np.uint32) + 1, X.indices.astype(np.uint32) + 1,
                   X.data.astype(np.float32), effective_lengths)


class LogitSkewNormalPTTApprox:
    def __init__(self, treemethod="cluster"):
        self.treemethod = treemethod  # one of "sequential", "random", "cluster"


class OptimizePTTApprox:
    pass


class Handle:
    """Thin RAII wrapper of polee_handle."""

    def __init__(self, device=0, approx=L.APPROX_LSN_PTT, num_steps=LIKAP_NUM_STEPS,
                 num_mc_samples=LIKAP_NUM_MC_SAMPLES, gradonly=True, use_efflen_jacobian=True, seed=123456789,
                 noise_mode=L.NOISE_PHILOX, use_cuda_graph=True, exact_accumulation=False):
        self.lib = L.load_library()
        o = L.PoleeOpts()
        self.lib.polee_opts_default(C.byref(o))
        o.device, o.approx, o.num_steps, o.num_mc_samples = device, approx, num_steps, num_mc_samples
        o.gradonly, o.use_efflen_jacobian, o.seed = int(gradonly), int(use_efflen_jacobian), seed
        o.noise_mode, o.use_cuda_graph = noise_mode, int(use_cuda_graph)
        o.exact_accumulation = int(exact_accumulation)
        self.opts = o
        self.h = _P()
        rc = self.lib.polee_create(C.byref(self.h), C.byref(o))
        if rc != 0:
            raise L.PoleeError(rc, self.lib.polee_last_error(None).decode())
        self.n = self.m = None
        self.K = 1 if approx == L.APPROX_OPTIMIZE_PTT else num_mc_samples

    def close(self):
        if getattr(self, "h", None):
            self.lib.polee_destroy(self.h)
            self.h = None

    __del__ = close

    def check(self, rc):
        if rc != 0:
            raise L.PoleeError(rc, self.lib.polee_last_error(self.h).decode())

    # ---- inputs
    def set_sample(self, sample, ks=None, tree_topology=None):
        """sample.X, sample.effective_lengths and -- when given -- the tree (node_parent_idxs, node_js): with a tree this
        is ONE polee_set_sample call (host tree preparation on a second thread beside the matrix upload / layout build),
        without it polee_set_matrix_csc + polee_set_efflens as before."""
        ksa = None if ks is None else _c(ks, np.int64)
        if tree_topology is not None and os.environ.get("POLEE_SET_SAMPLE", "") == "3calls":   # experiments: the old sequence
            self.set_sample(sample, ks)
            self.set_tree(*tree_topology)
            return
        if tree_topology is not None:
            pi, js = _c(tree_topology[0], np.int32), _c(tree_topology[1], np.int32)
            assert pi.shape == js.shape and len(js) == 2 * sample.n - 1
            self.check(self.lib.polee_set_sample(self.h, C.c_int64(sample.m), C.c_int64(sample.n), _p(sample.colptr),
                                                 _p(sample.rowval), _p(sample.nzval), _p(ksa),
                                                 _p(sample.effective_lengths), _p(pi), _p(js)))
            self.m, self.n = sample.m, sample.n
            return
        self.check(self.lib.polee_set_matrix_csc(self.h, C.c_int64(sample.m), C.c_int64(sample.n), _p(sample.colptr),
                                                 _p(sample.rowval), _p(sample.nzval), _p(ksa)))
        self.m, self.n = sample.m, sample.n
        self.check(self.lib.polee_set_efflens(self.h, _p(sample.effective_lengths)))

    def set_matrix_device(self, m, n, d_colptr, d_rowval, d_nzval, d_ks=0):
        """device pointers (ints), e.g. torch tensors' data_ptr()"""
        self.check(self.lib.polee_set_matrix_csc_device(self.h, C.c_int64(m), C.c_int64(n), _P(d_colptr), _P(d_rowval),
                                                        _P(d_nzval), _P(d_ks or None)))
        self.m, self.n = m, n

    def set_efflens(self, efflens):
        self.check(self.lib.polee_set_efflens(self.h, _p(_c(efflens, np.float32))))

    def set_gene_groups(self, gene_transcripts):
        """gene_transcripts: {gene_id: [1-based transcript indices]} as built at likelihood-approximation.jl:476-487
        (or any iterable of index lists).  Empty / None clears the map."""
        groups = list(gene_transcripts.values()) if hasattr(gene_transcripts, "values") else list(gene_transcripts or [])
        ptr = np.zeros(len(groups) + 1, np.int64)
        ptr[1:] = np.cumsum([len(g) for g in groups])
        tx = _c(np.concatenate([np.asarray(g, np.int32) for g in groups]) if groups else np.zeros(0, np.int32), np.int32)
        self.check(self.lib.polee_set_gene_groups(self.h, C.c_int64(len(groups)), _p(ptr), _p(tx)))

    def set_tree(self, node_parent_idxs, node_js):
        pi, js = _c(node_parent_idxs, np.int32), _c(node_js, np.int32)
        assert pi.shape == js.shape and len(js) % 2 == 1
        n = (len(js) + 1) // 2
        self.check(self.lib.polee_set_tree(self.h, C.c_int64(n), _p(pi), _p(js)))
        self.n = n

    def set_tree_sequential(self, n):
        self.check(self.lib.polee_set_tree_sequential(self.h, C.c_int64(n)))
        self.n = n

    # ---- fit
    def fit(self, noise=None, want_elbo=False):
        nm1 = self.n - 1
        mu, om, al = (np.zeros(nm1, np.float32) for _ in range(3))
        elbo = np.zeros(self.opts.num_steps, np.float64) if want_elbo else None
        nz = None if noise is None else _c(noise, np.float32)
        if nz is not None:
            assert nz.size == self.opts.num_steps * self.K * nm1
        self.check(self.lib.polee_fit(self.h, _p(mu), _p(om), _p(al), _p(elbo), _p(nz)))
        out = {"mu": mu, "omega": om, "alpha": al}
        if want_elbo:
            out["elbo"] = elbo
        return out

    def fit_optimize_ptt(self):
        xs = np.zeros(self.n, np.float32)
        self.check(self.lib.polee_fit_optimize_ptt(self.h, _p(xs)))
        return xs

    def init_params(self):
        self.check(self.lib.polee_init_params(self.h))

    def run_steps(self, nsteps):
        self.check(self.lib.polee_run_steps(self.h, C.c_int32(nsteps)))

    def sync(self):
        self.check(self.lib.polee_sync(self.h))

    def set_progress(self, callback, every=25):
        """callback(steps_done, num_steps) after every `every` finished ADAM steps (the reference's progress bar,
        likelihood-approximation.jl:495,574); None removes it."""
        if callback is None:
            self._progress = None
            self.check(self.lib.polee_set_progress(self.h, None, None, C.c_int32(0)))
            return
        fn_t = C.CFUNCTYPE(None, C.c_int32, C.c_int32, C.c_void_p)
        self._progress = fn_t(lambda done, total, user: callback(int(done), int(total)))  # keep the thunk alive
        self.check(self.lib.polee_set_progress(self.h, self._progress, None, C.c_int32(every)))

    def get_params(self):
        nm1 = self.n - 1
        mu, om, al = (np.zeros(nm1, np.float32) for _ in range(3))
        self.check(self.lib.polee_get_params(self.h, _p(mu), _p(om), _p(al)))
        return mu, om, al

    def set_params(self, mu, omega, alpha):
        self.check(self.lib.polee_set_params(self.h, _p(_c(mu, np.float32)), _p(_c(omega, np.float32)),
                                             _p(_c(alpha, np.float32))))

    def set_noise(self, noise, num_steps):
        self.check(self.lib.polee_set_noise(self.h, _p(_c(noise, np.float32)), C.c_int64(num_steps)))

    def stream(self):
        return self.lib.polee_stream(self.h)

    def step_stats(self):
        b = [C.c_double() for _ in range(3)]
        nl = C.c_int32()
        self.check(self.lib.polee_step_stats(self.h, C.byref(b[0]), C.byref(b[1]), C.byref(b[2]), C.byref(nl)))
        return {"bytes_k1": b[0].value, "bytes_k2": b[1].value, "bytes_k3": b[2].value, "launches": nl.value}

    def layout_info(self):
        v = (C.c_int64 * 13)()
        self.check(self.lib.polee_layout_info(self.h, v, C.c_int32(13)))
        keys = ("ec_rows", "ec_nnz", "ec_classes", "ec_tasks", "ec_blob_bytes", "ec_partials", "general_rows",
                "general_nnz", "general_kind", "ec_row_slots", "tree_route", "graph_programmatic_edges",
                "multi_step_graph_programmatic_edges")
        out = dict(zip(keys, (int(x) for x in v)))
        out["general_kind"] = ("none", "split", "fused")[out["general_kind"]]
        # the kernels the tree takes at the draw count of the last call (None: no tree, or no call yet)
        r = out["tree_route"]
        out["tree_route"] = None if r < 0 else ("chain", "dfs", "path", "levels_smem", "levels_global")[r]
        return out

    def time_kernel(self, which, reps):
        ms = C.c_float()
        self.check(self.lib.polee_time_kernel(self.h, C.c_int32(which), C.c_int32(reps), C.byref(ms)))
        return ms.value

    # ---- piecewise
    def loglik_grad(self, xs, gradonly=True):
        xs = np.atleast_2d(_c(xs, np.float32))
        K, n = xs.shape
        lp = np.zeros(K, np.float64)
        g = np.zeros((K, n), np.float64)
        self.check(self.lib.polee_loglik_grad(self.h, _p(xs), C.c_int32(K), C.c_int32(int(gradonly)), _p(lp), _p(g)))
        return lp, g

    def frag_prob_recip(self, xs):
        xs = _c(xs, np.float32)
        w = np.zeros(self.m, np.float32)
        self.check(self.lib.polee_frag_prob_recip(self.h, _p(xs), _p(w)))
        return w

    def ptt_transform(self, ys, compute_ladj=False):
        ys = np.atleast_2d(_c(ys, np.float64))
        K = ys.shape[0]
        xs = np.zeros((K, self.n), np.float32)
        ladj = np.zeros(K, np.float64) if compute_ladj else None
        self.check(self.lib.polee_ptt_transform(self.h, _p(ys), C.c_int32(K), _p(xs), _p(ladj)))
        return xs, ladj

    def ptt_transform_gradients(self, ys, x_grad, with_ladj=True):
        ys = np.atleast_2d(_c(ys, np.float64))
        x_grad = np.atleast_2d(_c(x_grad, np.float64))
        K = ys.shape[0]
        yg = np.zeros((K, self.n - 1), np.float32)
        self.check(self.lib.polee_ptt_transform_gradients(self.h, _p(ys), _p(x_grad), C.c_int32(K),
                                                          C.c_int32(int(with_ladj)), _p(yg)))
        return yg

    def ptt_inverse_transform(self, xs):
        xs = np.atleast_2d(_c(xs, np.float32))
        K = xs.shape[0]
        ys = np.zeros((K, self.n - 1), np.float64)
        ladj = np.zeros(K, np.float64)
        self.check(self.lib.polee_ptt_inverse_transform(self.h, _p(xs), C.c_int32(K), _p(ys), _p(ladj)))
        return ys, ladj

    def lsn_draws(self, zs0):
        zs0 = np.atleast_2d(_c(zs0, np.float32))
        K, nm1 = zs0.shape
        n = nm1 + 1
        out = {"xs": np.zeros((K, n), np.float32), "ys": np.zeros((K, nm1), np.float64),
               "x_grad": np.zeros((K, n), np.float64), "y_grad": np.zeros((K, nm1), np.float32),
               "mu_grad": np.zeros(nm1, np.float32), "omega_grad": np.zeros(nm1, np.float32),
               "alpha_grad": np.zeros(nm1, np.float32)}
        elbo = C.c_double()
        self.check(self.lib.polee_lsn_draws(self.h, _p(zs0), C.c_int32(K), _p(out["xs"]), _p(out["ys"]),
                                            _p(out["x_grad"]), _p(out["y_grad"]), _p(out["mu_grad"]),
                                            _p(out["omega_grad"]), _p(out["alpha_grad"]), C.byref(elbo)))
        out["elbo"] = elbo.value
        return out

    def sample(self, num_samples, seed=0):
        xs = np.zeros((num_samples, self.n), np.float32)
        self.check(self.lib.polee_sample(self.h, C.c_int32(num_samples), C.c_uint64(seed), _p(xs)))
        return xs

    # ---- multi-GPU
    def comm_peer_export(self):
        """This rank's CUDA IPC handle (64 bytes) for the peer-memory all-reduce; see comm_peer_import."""
        buf = C.create_string_buffer(64)
        self.check(self.lib.polee_comm_peer_export(self.h, buf))
        return buf.raw

    def comm_peer_import(self, handles):
        """handles: the 64-byte handles of all ranks, in rank order (gathered by the caller, e.g. with
        torch.distributed.all_gather_object).  Returns False (and keeps the NCCL all-reduce) when peer access is not
        available."""
        if handles is None:   # back to the NCCL all-reduce
            self.check(self.lib.polee_comm_peer_import(self.h, None))
            return False
        blob = b"".join(handles)
        rc = self.lib.polee_comm_peer_import(self.h, C.c_char_p(blob))
        if rc == L.POLEE_ECUDA:
            return False
        self.check(rc)
        return True

    def comm_init(self, nranks, rank, unique_id):
        self.check(self.lib.polee_comm_init(self.h, C.c_int32(nranks), C.c_int32(rank), C.c_char_p(unique_id)))


def hclust(sample):
    """PolyaTreeTransform(X, :cluster) -> (node_parent_idxs, node_js): hclust + order_nodes (src/hclust.jl:193-319,
    361-389) on the host; ties broken by an explicit rule (the reference's are unspecified, SURVEY 8c)."""
    lib = L.load_library()
    N = 2 * sample.n - 1
    pi, js = np.zeros(N, np.int32), np.zeros(N, np.int32)
    rc = lib.polee_hclust(C.c_int64(sample.m), C.c_int64(sample.n), _p(sample.colptr), _p(sample.rowval), _p(pi), _p(js))
    if rc != 0:
        raise L.PoleeError(rc, "polee_hclust failed")
    return pi, js


def exact_factorization(sample, device=0):
    """tools/exact-factorization.jl:31-68 on the device: (compressed RNASeqSample, counts).  Feed the pair to
    approximate_likelihood(..., ks=counts) / Handle.set_sample(sample, ks): same likelihood, fewer rows to stream."""
    lib = L.load_library()
    nnz = len(sample.rowval)
    colptr = np.zeros(sample.n + 1, np.uint32)
    rowval = np.zeros(max(nnz, 1), np.uint32)
    nzval = np.zeros(max(nnz, 1), np.float32)
    counts = np.zeros(sample.m, np.int64)
    mu, nu = C.c_int64(), C.c_int64()
    rc = lib.polee_exact_factorization(C.c_int32(device), C.c_int64(sample.m), C.c_int64(sample.n), _p(sample.colptr),
                                       _p(sample.rowval), _p(sample.nzval), C.byref(mu), _p(colptr), _p(rowval), _p(nzval),
                                       _p(counts), C.byref(nu))
    if rc != 0:
        raise L.PoleeError(rc, "polee_exact_factorization failed")
    out = RNASeqSample(mu.value, sample.n, colptr, rowval[:nu.value].copy(), nzval[:nu.value].copy(),
                       sample.effective_lengths)
    return out, counts[:mu.value].copy()


def trim_memory(device=-1):
    """Return the device memory cached from destroyed handles to the driver (polee_trim_memory)."""
    L.load_library().polee_trim_memory(C.c_int32(device))


def comm_unique_id():
    buf = C.create_string_buffer(128)
    rc = L.load_library().polee_comm_unique_id(buf)
    if rc != 0:
        raise L.PoleeError(rc, "ncclGetUniqueId failed")
    return buf.raw


def connect_ranks(h, dist):
    """Join the handles of a row-partitioned fit (one process per GPU, `dist` = an initialised torch.distributed):
    NCCL communicator (polee_comm_init) and, unless POLEE_ALLREDUCE=nccl|f64, the peer-memory all-reduce
    (polee_comm_peer_export / _import; the IPC handles travel through dist.all_gather_object).  Returns "peer" or "nccl":
    which all-reduce the step graph will use.  Call after the matrix or the tree is set."""
    import os
    world, rank = dist.get_world_size(), dist.get_rank()
    uid = [comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    h.comm_init(world, rank, uid[0])
    if world < 2 or os.environ.get("POLEE_ALLREDUCE", "") in ("nccl", "f64"):
        return "nccl"
    handles = [None] * world
    dist.all_gather_object(handles, h.comm_peer_export())
    ok = h.comm_peer_import(handles)
    flags = [None] * world
    dist.all_gather_object(flags, bool(ok))   # every rank must take the same path
    if not all(flags):
        h.comm_peer_import(None)   # drop this rank's mapping too: all ranks stay on NCCL
        return "nccl"
    return "peer"


def partition_rows(sample, nparts):
    """Equal-nnz contiguous row blocks (SURVEY 8e): returns nparts+1 0-based half-open bounds."""
    bounds = np.zeros(nparts + 1, np.int64)
    rc = L.load_library().polee_partition_rows(C.c_int64(sample.m), C.c_int64(sample.n), _p(sample.colptr),
                                               _p(sample.rowval), C.c_int32(nparts), _p(bounds))
    if rc != 0:
        raise L.PoleeError(rc, "polee_partition_rows: bad arguments")
    return bounds


def row_block(sample, lo, hi):
    """The sub-sample holding rows [lo, hi) (0-based) and all n columns."""
    keep = (sample.rowval > lo) & (sample.rowval <= hi)
    col_of = np.repeat(np.arange(sample.n), np.diff(sample.colptr.astype(np.int64)))
    counts = np.bincount(col_of[keep], minlength=sample.n)
    colptr = np.concatenate([[1], 1 + np.cumsum(counts)]).astype(np.uint32)
    return RNASeqSample(hi - lo, sample.n, colptr, (sample.rowval[keep] - lo).astype(np.uint32), sample.nzval[keep],
                        sample.effective_lengths)


class PolyaTreeTransform:
    """PolyaTreeTransform(parent_idxs, output_idxs) (src/ptt.jl:89-116) living on the device."""

    def __init__(self, node_parent_idxs, node_js, device=0):
        self.node_parent_idxs = _c(node_parent_idxs, np.int32)
        self.node_js = _c(node_js, np.int32)
        self.handle = Handle(device=device, num_mc_samples=1)
        self.handle.set_tree(self.node_parent_idxs, self.node_js)
        self.n = self.handle.n

    @classmethod
    def sequential(cls, n, device=0):
        """PolyaTreeTransform(X, :sequential): list_nodes(n), src/hclust.jl:477-489."""
        pi, js = sequential_tree(n)
        return cls(pi, js, device)

    def transform(self, ys, compute_ladj=False):
        """transform!(t, ys, xs, Val(compute_ladj)) -> (xs, ladj)   src/ptt.jl:125-160"""
        xs, ladj = self.handle.ptt_transform(ys, compute_ladj)
        one = np.ndim(ys) == 1
        return (xs[0] if one else xs), (0.0 if ladj is None else (ladj[0] if one else ladj))

    def transform_gradients(self, ys, x_grad):
        """transform_gradients!(t, ys, y_grad, x_grad) -> y_grad   src/ptt.jl:167-209"""
        yg = self.handle.ptt_transform_gradients(ys, x_grad, True)
        return yg[0] if np.ndim(ys) == 1 else yg

    def transform_gradients_no_ladj(self, ys, x_grad):
        """transform_gradients_no_ladj!   src/ptt.jl:217-251"""
        yg = self.handle.ptt_transform_gradients(ys, x_grad, False)
        return yg[0] if np.ndim(ys) == 1 else yg

    def inverse_transform(self, xs):
        """inverse_transform!(t, xs, ys) -> (ys, ladj)   src/ptt.jl:257-285"""
        ys, ladj = self.handle.ptt_inverse_transform(xs)
        one = np.ndim(xs) == 1
        return (ys[0] if one else ys), (ladj[0] if one else ladj)


class ApproxLikelihoodSampler:
    """ApproxLikelihoodSampler (src/approx-sampler.jl:1-44): set_transform!(als, t, mu, sigma, alpha); rand!(als, xs)."""

    def __init__(self, device=0, draws_per_launch=16):
        self.handle = Handle(device=device, num_mc_samples=draws_per_launch)
        self.calls = 0
        self.plan = None

    def set_transform(self, t, mu, sigma, alpha):
        """t: PolyaTreeTransform or (node_parent_idxs, node_js); sigma = exp(omega) as in src/main.jl:833."""
        pi, js = (t.node_parent_idxs, t.node_js) if isinstance(t, PolyaTreeTransform) else t
        self.handle.set_tree(pi, js)
        omega = np.log(_c(sigma, np.float32))
        self.handle.set_params(mu, omega, alpha)
        self.tree = (_c(pi, np.int32), _c(js, np.int32))
        self.params = (_c(mu, np.float32), omega, _c(alpha, np.float32))
        if self.plan is not None:
            self.plan.close()
            self.plan = None

    def rand(self, num_samples=1, seed=None):
        """rand!(als, xs) for num_samples draws at once -> xs[num_samples][n]"""
        self.calls += 1
        return self.handle.sample(num_samples, self.calls if seed is None else seed)

    def log_prob(self, xs, want_grad=False):
        """log q(xs) of the approximation set_transform holds, in the x space rand() returns (DESIGN.md K5):
        xs [num_samples][n] -> lp [num_samples], or (lp, x_grad) with want_grad."""
        if self.plan is None:
            self.plan = HsbPlan(self.handle.n, *make_inverse_ptt_params(*self.tree), device=self.handle.opts.device)
        return self.plan.approx_log_prob(xs, *self.params, want_grad=want_grad)


def sequential_tree(n):
    """(node_parent_idxs, node_js) of list_nodes(n) after order_nodes (src/hclust.jl:477-489, 361-389)."""
    N = 2 * n - 1
    pi = np.zeros(N, np.int32)
    js = np.zeros(N, np.int32)
    pos, parent = 0, 0
    for leaf in range(1, n):
        pi[pos], js[pos] = parent, 0
        me = pos + 1
        pos += 1
        pi[pos], js[pos] = me, leaf
        pos += 1
        parent = me
    pi[pos], js[pos] = parent, n
    return pi, js


def make_inverse_ptt_params(node_parent_idxs, node_js):
    """make_inverse_ptt_params (src/ptt.jl:293-309): 0-based left/right (-1 = none) and leaf = js - 1."""
    pi, js = _c(node_parent_idxs, np.int32), _c(node_js, np.int32)
    N = len(js)
    l, r, f = (np.zeros(N, np.int32) for _ in range(3))
    rc = L.load_library().polee_make_inverse_ptt_params(C.c_int64(N), _p(pi), _p(js), _p(l), _p(r), _p(f))
    if rc != 0:
        raise L.PoleeError(rc, "make_inverse_ptt_params: bad tree arrays")
    return l, r, f


def log_likelihood(sample, xs, gradonly=True, ks=None, tree=None, device=0, exact_accumulation=False):
    """log_likelihood(frag_probs, log_frag_probs, X, Xt, xs, x_grad, Val(gradonly)) -> (lp, x_grad)
    (src/likelihood.jl:36-56; factored_log_likelihood :59-85 when ks is given)."""
    h = Handle(device=device, num_mc_samples=1, exact_accumulation=exact_accumulation)
    try:
        h.set_sample(sample, ks)
        pi, js = tree if tree is not None else sequential_tree(sample.n)
        h.set_tree(pi, js)
        lp, g = h.loglik_grad(xs, gradonly)
        return (lp[0], g[0]) if np.ndim(xs) == 1 else (lp, g)
    finally:
        h.close()


def approximate_likelihood(approx, sample, gradonly=True, tree_topology=None, use_efflen_jacobian=True,
                           gene_noninformative=False, ks=None, num_steps=LIKAP_NUM_STEPS,
                           num_mc_samples=LIKAP_NUM_MC_SAMPLES, seed=123456789, noise=None, device=0, want_elbo=False,
                           exact_accumulation=False, gene_transcripts=None):
    """approximate_likelihood(approx, sample, Val(gradonly); tree_topology_input_filename, use_efflen_jacobian,
    gene_noninformative) -> Dict  (src/likelihood-approximation.jl:395-624; :248-392 with ks; :149-242 for
    OptimizePTTApprox).

    tree_topology = (node_parent_idxs, node_js), what the reference reads from tree_topology_input_filename
    (:428-433).  Without one the tree is built as the reference does at :435: "sequential" -> list_nodes, "cluster" ->
    the hclust restatement (polee_hclust, host code; tie-breaking is unpinned in the reference, SURVEY 8c); "random" ->
    rand_tree_nodes restated on a seeded numpy generator (same distribution; Julia's RNG stream cannot be reproduced).
    gene_transcripts = {gene_id: [1-based transcript indices]} is the map the reference derives from the transcript
    metadata when gene_noninformative is set (:476-487); without it the flag is dropped with a warning (:489-492).
    """
    if gene_noninformative and not gene_transcripts:
        import warnings
        warnings.warn("'--gene-noninformative' used, but no gene information available")
        gene_noninformative = False
    if isinstance(approx, OptimizePTTApprox):
        h = Handle(device=device, approx=L.APPROX_OPTIMIZE_PTT, num_steps=num_steps)
        try:
            h.set_sample(sample)
            return {"x": h.fit_optimize_ptt()}
        finally:
            h.close()
    if not isinstance(approx, LogitSkewNormalPTTApprox):
        raise TypeError("alternative approximations stay on the reference's Julia path (SURVEY 2a)")
    built_here = tree_topology is None
    if built_here:                      # PolyaTreeTransform(X, approx.treemethod)  (:435, ptt.jl:35-52)
        if approx.treemethod == "sequential":
            tree_topology = sequential_tree(sample.n)
        elif approx.treemethod == "cluster":
            tree_topology = hclust(sample)
        elif approx.treemethod == "random":
            # rand_tree_nodes (src/hclust.jl:439-454): the same procedure (join two random subtrees until one is left)
            # on numpy's generator seeded with `seed` -- Julia's RNG stream cannot be reproduced, the distribution can
            from . import synth
            tree_topology = synth.random_tree(sample.n, seed=seed)
        else:
            raise ValueError("%r is not a supported Polya tree transform heuristic" % (approx.treemethod,))
    h = Handle(device=device, num_steps=num_steps, num_mc_samples=num_mc_samples, gradonly=gradonly,
               use_efflen_jacobian=use_efflen_jacobian, seed=seed,
               noise_mode=L.NOISE_INJECTED if noise is not None else L.NOISE_PHILOX,
               exact_accumulation=exact_accumulation)
    try:
        h.set_sample(sample, ks, tree_topology)
        if gene_noninformative:
            h.set_gene_groups(gene_transcripts)
        params = h.fit(noise=noise, want_elbo=want_elbo)
    finally:
        h.close()
    if built_here:  # :618-621
        params["node_parent_idxs"] = np.asarray(tree_topology[0], np.int32)
        params["node_js"] = np.asarray(tree_topology[1], np.int32)
    return params


def prep_many(samples, tree_topologies, devices=(0,), **fit_kwargs):
    """The sample loop of `polee prep` (src/main.jl:590-631) with whole samples sharded over GPUs: "replicas only"
    (SURVEY 8e, BASELINE config 5) -- one worker per device pulls the next sample from a queue; no collective.
    Returns the parameter dicts in input order.  Handles are independent, ctypes releases the GIL during calls."""
    import queue
    import threading

    todo = queue.Queue()
    for i, (smp, tree) in enumerate(zip(samples, tree_topologies)):
        todo.put((i, smp, tree))
    out = [None] * len(samples)
    errors = []

    def worker(dev):
        while True:
            try:
                i, smp, tree = todo.get_nowait()
            except queue.Empty:
                return
            try:
                out[i] = approximate_likelihood(LogitSkewNormalPTTApprox(), smp, tree_topology=tree, device=dev, **fit_kwargs)
            except Exception as e:  # surface after joining
                errors.append((i, e))

    threads = [threading.Thread(target=worker, args=(d,)) for d in devices]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0][1]
    return out


def optimize_likelihood(sample, device=0):
    """optimize_likelihood(sample) (src/likelihood-approximation.jl:23-25)"""
    return approximate_likelihood(OptimizePTTApprox(), sample, device=device)["x"]


# ---------------------------------------------------------------------------------------- hsb ops
def _hsb_idx(left, right, leaf, B, n):
    N = 2 * n - 1
    arrs = [_c(a, np.int32).reshape(-1, N) for a in (left, right, leaf)]
    ib = arrs[0].shape[0]
    assert all(a.shape[0] == ib for a in arrs) and ib in (1, B)
    return arrs, ib


def _hsb_check(rc):
    if rc != 0:
        raise L.PoleeError(rc, L.load_library().polee_hsb_last_error().decode())


def hsb(y_logit, left_index, right_index, leaf_index, device=0):
    """hsb(y_logit, left, right, leaf) -> x   (op HSB, src/tensorflow_ext/hsb_ops.cpp:17-120)"""
    y_logit = _c(y_logit, np.float32)
    B, nm1 = y_logit.shape
    n = nm1 + 1
    (l, r, f), ib = _hsb_idx(left_index, right_index, leaf_index, B, n)
    x = np.zeros((B, n), np.float32)
    _hsb_check(L.load_library().polee_hsb(C.c_int32(device), C.c_int64(B), C.c_int64(n), _p(y_logit), _p(l), _p(r),
                                          _p(f), C.c_int64(ib), _p(x)))
    return x


def inv_hsb(x, left_index, right_index, leaf_index, device=0):
    """inv_hsb(x, left, right, leaf) -> (y float64, ladj float32 [B,1])   (op InvHSB, hsb_ops.cpp:128-249)"""
    x = _c(x, np.float32)
    B, n = x.shape
    (l, r, f), ib = _hsb_idx(left_index, right_index, leaf_index, B, n)
    y = np.zeros((B, n - 1), np.float64)
    ladj = np.zeros((B, 1), np.float32)
    _hsb_check(L.load_library().polee_inv_hsb(C.c_int32(device), C.c_int64(B), C.c_int64(n), _p(x), _p(l), _p(r), _p(f),
                                              C.c_int64(ib), _p(y), _p(ladj)))
    return y, ladj


def inv_hsb_grad(y_grad, ladj_grad, y, ladj, left_index, right_index, leaf_index, device=0):
    """inv_hsb_grad(y_grad, ladj_grad, y, ladj, left, right, leaf) -> backprops  (op InvHSBGrad, hsb_ops.cpp:252-402)"""
    y = _c(y, np.float64)
    y_grad = _c(y_grad, np.float64)
    B, nm1 = y.shape
    n = nm1 + 1
    ladj_grad = _c(ladj_grad, np.float32).reshape(B)
    (l, r, f), ib = _hsb_idx(left_index, right_index, leaf_index, B, n)
    bp = np.zeros((B, n), np.float32)
    _hsb_check(L.load_library().polee_inv_hsb_grad(C.c_int32(device), C.c_int64(B), C.c_int64(n), _p(y_grad),
                                                   _p(ladj_grad), _p(y), _p(l), _p(r), _p(f), C.c_int64(ib), _p(bp)))
    return bp


def hsb_grad(x_grad, y_logit, left_index, right_index, leaf_index, device=0):
    """hsb_grad(x_grad, y_logit, left, right, leaf) -> y_logit_grad [B][n-1] float32: the gradient of hsb(y_logit) that
    the reference leaves as a TODO (hsb_ops.cpp:123-125); definition: include/polee_b200.h, DESIGN.md K4."""
    y_logit = _c(y_logit, np.float32)
    B, nm1 = y_logit.shape
    n = nm1 + 1
    x_grad = _c(x_grad, np.float32).reshape(B, n)
    (l, r, f), ib = _hsb_idx(left_index, right_index, leaf_index, B, n)
    out = np.zeros((B, nm1), np.float32)
    _hsb_check(L.load_library().polee_hsb_grad(C.c_int32(device), C.c_int64(B), C.c_int64(n), _p(x_grad), _p(y_logit),
                                               _p(l), _p(r), _p(f), C.c_int64(ib), _p(out)))
    return out


class HsbPlan:
    """The validated, level-scheduled tree(s) of the three HSB ops resident on the device (polee_hsb_plan_*), with the
    device-resident entry points (polee_*_device): every tensor argument is a DEVICE pointer (int), the work is
    enqueued on `stream` (a cudaStream_t as int; 0 = the legacy stream) and nothing is copied -- what the DEVICE_GPU
    registration of the TF ops binds (polee_b200/tf/hsb_ops_b200.cpp)."""

    def __init__(self, n, left_index, right_index, leaf_index, device=0):
        N = 2 * n - 1
        arrs = [_c(a, np.int32).reshape(-1, N) for a in (left_index, right_index, leaf_index)]
        self.n, self.idx_batch = n, arrs[0].shape[0]
        self.lib = L.load_library()
        self.p = C.c_void_p()
        _hsb_check(self.lib.polee_hsb_plan_create(C.byref(self.p), C.c_int32(device), C.c_int64(n), C.c_int64(self.idx_batch),
                                                  _p(arrs[0]), _p(arrs[1]), _p(arrs[2])))

    def close(self):
        if self.p:
            self.lib.polee_hsb_plan_destroy(self.p)
            self.p = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def hsb_device(self, B, d_y_logit, d_x, stream=0):
        _hsb_check(self.lib.polee_hsb_device(self.p, C.c_int64(B), C.c_void_p(d_y_logit), C.c_void_p(d_x), C.c_void_p(stream)))

    def inv_hsb_device(self, B, d_x, d_y, d_ladj, stream=0):
        _hsb_check(self.lib.polee_inv_hsb_device(self.p, C.c_int64(B), C.c_void_p(d_x), C.c_void_p(d_y), C.c_void_p(d_ladj),
                                                 C.c_void_p(stream)))

    def inv_hsb_grad_device(self, B, d_y_grad, d_ladj_grad, d_y, d_backprops, stream=0):
        _hsb_check(self.lib.polee_inv_hsb_grad_device(self.p, C.c_int64(B), C.c_void_p(d_y_grad), C.c_void_p(d_ladj_grad),
                                                      C.c_void_p(d_y), C.c_void_p(d_backprops), C.c_void_p(stream)))

    def hsb_grad_device(self, B, d_x_grad, d_y_logit, d_y_logit_grad, stream=0):
        _hsb_check(self.lib.polee_hsb_grad_device(self.p, C.c_int64(B), C.c_void_p(d_x_grad), C.c_void_p(d_y_logit),
                                                  C.c_void_p(d_y_logit_grad), C.c_void_p(stream)))

    def approx_log_prob(self, x, mu, omega, alpha, want_grad=True):
        """log q(x) of the LogitSkewNormalPTT approximation on this plan's tree(s) (polee_approx_log_prob_with_plan;
        definition: DESIGN.md K5).  x [B][n]; mu / omega / alpha [param_batch][n-1] (or [n-1]), param_batch 1 or B.
        Returns lp [B] Float64, or (lp, x_grad [B][n] Float32) with want_grad."""
        x = np.atleast_2d(_c(x, np.float32))
        B, n = x.shape
        mu, omega, alpha = (_c(a, np.float32).reshape(a.size // (n - 1) if n > 1 else 1, n - 1)
                            for a in (np.asarray(mu), np.asarray(omega), np.asarray(alpha)))
        if not mu.shape[0] == omega.shape[0] == alpha.shape[0]:
            raise ValueError("mu, omega and alpha must have the same number of rows")
        lp = np.zeros(B, np.float64)
        x_grad = np.zeros((B, n), np.float32) if want_grad else None
        _hsb_check(self.lib.polee_approx_log_prob_with_plan(self.p, C.c_int64(B), C.c_int64(mu.shape[0]), _p(x), _p(mu),
                                                            _p(omega), _p(alpha), _p(lp), _p(x_grad)))
        return (lp, x_grad) if want_grad else lp

    def approx_log_prob_device(self, B, param_batch, d_x, d_mu, d_omega, d_alpha, d_lp, d_x_grad=0, stream=0):
        """polee_approx_log_prob_device: device pointers; d_x_grad = 0 computes lp only."""
        _hsb_check(self.lib.polee_approx_log_prob_device(self.p, C.c_int64(B), C.c_int64(param_batch), C.c_void_p(d_x),
                                                         C.c_void_p(d_mu), C.c_void_p(d_omega), C.c_void_p(d_alpha),
                                                         C.c_void_p(d_lp), C.c_void_p(d_x_grad or None),
                                                         C.c_void_p(stream)))


def approx_log_prob(x, mu, omega, alpha, left_index, right_index, leaf_index, want_grad=True, device=0):
    """log q(x) of the fitted LogitSkewNormalPTT approximation (mu, omega = log sigma, alpha: one row, or one per row of
    x) on the tree(s) given as make_inverse_ptt_params arrays -> lp [B], or (lp, x_grad) with want_grad.  The density
    the reference evaluates in RNASeqApproxLikelihoodDist._log_prob (src/polee_approx_likelihood.py:367-450), in the
    fit's own x space (no effective-length rescaling); definition: DESIGN.md K5."""
    x = np.atleast_2d(_c(x, np.float32))
    plan = HsbPlan(x.shape[1], left_index, right_index, leaf_index, device)
    try:
        return plan.approx_log_prob(x, mu, omega, alpha, want_grad)
    finally:
        plan.close()


_approx_log_prob_fn = None


def approx_log_prob_torch(plan, x, mu, omega, alpha):
    """Differentiable log q(x) for a torch model: lp [B] (float64) of x [B][n] (float32, on the plan's device), computed
    by polee_approx_log_prob_device on torch's current stream.  Gradients flow into x only (grad_lp[:, None] * x_grad);
    mu / omega / alpha ([param_batch][n-1], param_batch 1 or B) are constants here."""
    global _approx_log_prob_fn
    if _approx_log_prob_fn is None:
        import torch

        class ApproxLogProb(torch.autograd.Function):
            @staticmethod
            def forward(ctx, plan, x, mu, omega, alpha):
                x = x.detach().to(torch.float32).contiguous()
                n = x.shape[1]
                mu, omega, alpha = (a.detach().to(device=x.device, dtype=torch.float32).reshape(-1, n - 1).contiguous()
                                    for a in (mu, omega, alpha))
                B = x.shape[0]
                lp = torch.empty(B, dtype=torch.float64, device=x.device)
                x_grad = torch.empty_like(x) if ctx.needs_input_grad[1] else None
                plan.approx_log_prob_device(B, mu.shape[0], x.data_ptr(), mu.data_ptr(), omega.data_ptr(),
                                            alpha.data_ptr(), lp.data_ptr(), 0 if x_grad is None else x_grad.data_ptr(),
                                            torch.cuda.current_stream(x.device).cuda_stream)
                ctx.save_for_backward(x_grad)
                return lp

            @staticmethod
            def backward(ctx, grad_lp):
                (x_grad,) = ctx.saved_tensors
                return None, (grad_lp[:, None] * x_grad).to(x_grad.dtype), None, None, None

        _approx_log_prob_fn = ApproxLogProb
    return _approx_log_prob_fn.apply(plan, x, mu, omega, alpha)


_hsb_fn = None
_inv_hsb_fn = None


def _stream_of(t):
    import torch
    return torch.cuda.current_stream(t.device).cuda_stream


def hsb_torch(plan, y_logit):
    """Differentiable HSB for a torch model: x [B][n] (float32) = hsb(y_logit [B][n-1]) on the plan's tree(s), computed
    by polee_hsb_device on torch's current stream; the backward is HSBGrad (polee_hsb_grad_device)."""
    global _hsb_fn
    if _hsb_fn is None:
        import torch

        class Hsb(torch.autograd.Function):
            @staticmethod
            def forward(ctx, plan, y_logit):
                y_logit = y_logit.detach().to(torch.float32).contiguous()
                B = y_logit.shape[0]
                x = torch.empty((B, plan.n), dtype=torch.float32, device=y_logit.device)
                plan.hsb_device(B, y_logit.data_ptr(), x.data_ptr(), _stream_of(y_logit))
                ctx.plan = plan
                ctx.save_for_backward(y_logit)
                return x

            @staticmethod
            def backward(ctx, grad_x):
                (y_logit,) = ctx.saved_tensors
                grad_x = grad_x.to(torch.float32).contiguous()
                out = torch.empty_like(y_logit)
                ctx.plan.hsb_grad_device(y_logit.shape[0], grad_x.data_ptr(), y_logit.data_ptr(), out.data_ptr(),
                                         _stream_of(y_logit))
                return None, out

        _hsb_fn = Hsb
    return _hsb_fn.apply(plan, y_logit)


def inv_hsb_torch(plan, x):
    """Differentiable InvHSB for a torch model: (y [B][n-1] float64, ladj [B][1] float32) = inv_hsb(x [B][n]) on the
    plan's tree(s), computed by polee_inv_hsb_device on torch's current stream; the backward is InvHSBGrad
    (polee_inv_hsb_grad_device), with a missing upstream gradient taken as zeros."""
    global _inv_hsb_fn
    if _inv_hsb_fn is None:
        import torch

        class InvHsb(torch.autograd.Function):
            @staticmethod
            def forward(ctx, plan, x):
                x = x.detach().to(torch.float32).contiguous()
                B = x.shape[0]
                y = torch.empty((B, plan.n - 1), dtype=torch.float64, device=x.device)
                ladj = torch.empty((B, 1), dtype=torch.float32, device=x.device)
                plan.inv_hsb_device(B, x.data_ptr(), y.data_ptr(), ladj.data_ptr(), _stream_of(x))
                ctx.plan = plan
                ctx.save_for_backward(y)
                return y, ladj

            @staticmethod
            def backward(ctx, grad_y, grad_ladj):
                (y,) = ctx.saved_tensors
                B = y.shape[0]
                grad_y = torch.zeros_like(y) if grad_y is None else grad_y.to(torch.float64).contiguous()
                grad_ladj = (torch.zeros((B,), dtype=torch.float32, device=y.device) if grad_ladj is None
                             else grad_ladj.to(torch.float32).reshape(B).contiguous())
                out = torch.empty((B, ctx.plan.n), dtype=torch.float32, device=y.device)
                ctx.plan.inv_hsb_grad_device(B, grad_y.data_ptr(), grad_ladj.data_ptr(), y.data_ptr(), out.data_ptr(),
                                             _stream_of(y))
                return None, out

        _inv_hsb_fn = InvHsb
    return _inv_hsb_fn.apply(plan, x)
