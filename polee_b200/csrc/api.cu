// api.cu -- the extern "C" surface of libpolee_b200.so (include/polee_b200.h) and the per-step
// launch sequence.  No CPU fallback anywhere: every compute entry point needs a CUDA device.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <mutex>

#include <dlfcn.h>

#include "common.cuh"
#include <chrono>
#include <thread>

using namespace polee;

#ifdef POLEE_WITH_NCCL
// NCCL is bound lazily with dlopen: single-GPU users need no NCCL at all, and a host process that already
// carries its own libnccl.so.2 (e.g. PyTorch's bundled one) keeps using exactly that copy.
namespace {
struct NcclApi {
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};
NcclApi &nccl_api() {
    static NcclApi api;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void *lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (lib) {
            api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(lib, "ncclGetUniqueId");
            api.CommInitRank = (decltype(api.CommInitRank))dlsym(lib, "ncclCommInitRank");
            api.CommDestroy = (decltype(api.CommDestroy))dlsym(lib, "ncclCommDestroy");
            api.AllReduce = (decltype(api.AllReduce))dlsym(lib, "ncclAllReduce");
            api.GetErrorString = (decltype(api.GetErrorString))dlsym(lib, "ncclGetErrorString");
            api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.AllReduce && api.GetErrorString;
        }
    }
    return api;
}
}  // namespace
#endif

static std::string g_create_error;
static std::mutex g_err_mu;

#define CK(expr) POLEE_CUDA_CHECK(h, expr)
#define CHECK_H(h)                    \
    if (!(h)) return POLEE_EINVAL;    \
    (h)->err.clear();                 \
    if (cudaSetDevice((h)->device) != cudaSuccess) return (h)->fail(POLEE_ECUDA, "cudaSetDevice failed")

constexpr int TREE_BIN_NODES = 512;  // nodes per bottom bin of the tree schedule
// steps per launch of the multi-step graph: inside it the step boundary (k3_elem -> tree forward) is a programmatic edge
// too, and one graph launch replaces STEP_GRAPH_STEPS
constexpr int STEP_GRAPH_STEPS = 8;
constexpr int STEP_GRAPH_LEAD = 3;  // steps queued before the multi-step graph is captured (polee_run_steps)

static void drop_graph(polee_handle *h) {
    if (h->graph_exec) cudaGraphExecDestroy(h->graph_exec);
    if (h->graph) cudaGraphDestroy(h->graph);
    if (h->graph_multi_exec) cudaGraphExecDestroy(h->graph_multi_exec);
    if (h->graph_multi) cudaGraphDestroy(h->graph_multi);
    h->graph_exec = nullptr;
    h->graph = nullptr;
    h->graph_multi_exec = nullptr;
    h->graph_multi = nullptr;
    h->graph_warm = false;
}

extern "C" int polee_opts_default(polee_opts *o) {
    if (!o) return POLEE_EINVAL;
    std::memset(o, 0, sizeof(*o));
    o->device = 0;
    o->approx = POLEE_APPROX_LOGIT_SKEW_NORMAL_PTT;
    o->num_steps = 500;       // LIKAP_NUM_STEPS       constants.jl:64
    o->num_mc_samples = 6;    // LIKAP_NUM_MC_SAMPLES  constants.jl:65
    o->gradonly = 1;          // Val(gradonly)=Val(true)  likelihood-approximation.jl:397
    o->use_efflen_jacobian = 1;
    o->noise_mode = POLEE_NOISE_PHILOX;
    o->seed = 123456789ull;   // main.jl:123-127
    o->max_step_mu = 2e-1;    // likelihood-approximation.jl:421-423
    o->max_step_omega = 2e-1;
    o->max_step_alpha = 2e-2;
    o->max_step_z = 1e-1;     // :166
    o->use_cuda_graph = 1;
    return POLEE_OK;
}

extern "C" int polee_device_info(int32_t device, int32_t *sm, int32_t *num_sms, int64_t *hbm_bytes) {
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, device) != cudaSuccess) return POLEE_ECUDA;
    if (sm) *sm = p.major * 10 + p.minor;
    if (num_sms) *num_sms = p.multiProcessorCount;
    if (hbm_bytes) *hbm_bytes = (int64_t)p.totalGlobalMem;
    return POLEE_OK;
}

// POLEE_SETUP_TIMING=1: where polee_create / polee_set_tree / polee_set_sample spend their time
struct HostPhaseTimer {
    bool on = getenv("POLEE_SETUP_TIMING") != nullptr;
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    void mark(const char *what) {
        if (!on) return;
        auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[polee tree ] %-28s %8.2f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

extern "C" int polee_create(polee_handle **out, const polee_opts *opts) {
    if (!out) return POLEE_EINVAL;
    *out = nullptr;
    polee_opts o;
    if (opts) o = *opts; else polee_opts_default(&o);
    auto fail = [&](int code, const std::string &msg) {
        std::lock_guard<std::mutex> lk(g_err_mu);
        g_create_error = msg;
        return code;
    };
    if (o.num_mc_samples < 1 || o.num_mc_samples > 16) return fail(POLEE_EINVAL, "num_mc_samples must be in 1..16");
    if (o.approx == POLEE_APPROX_OPTIMIZE_PTT) o.num_mc_samples = 1;
    if (o.num_steps < 0) return fail(POLEE_EINVAL, "num_steps must be >= 0");
    HostPhaseTimer pt;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(POLEE_ECUDA, std::string("no CUDA device (libpolee_b200 has no CPU fallback): ") +
                                     cudaGetErrorString(e));
    if (o.device < 0 || o.device >= count) return fail(POLEE_EINVAL, "device ordinal out of range");
    // two attribute queries, not cudaGetDeviceProperties: that call also asks the driver for clocks and the like and was
    // measured taking 3 - 290 ms on a GPU that had just gone idle (profiles/README.md, round 2, e2e set-up)
    int cc_major = 0, sm_count = 0;
    if (cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, o.device) != cudaSuccess ||
        cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, o.device) != cudaSuccess)
        return fail(POLEE_ECUDA, "cudaDeviceGetAttribute failed");
    if (cc_major != 10) return fail(POLEE_ECUDA, "libpolee_b200 is built for sm_100a only (B200); found another GPU");
    if (cudaSetDevice(o.device) != cudaSuccess) return fail(POLEE_ECUDA, "cudaSetDevice failed");
    pt.mark("create: device queries");
    polee_handle *h = new polee_handle();
    h->o = o;
    h->device = o.device;
    h->num_sms = sm_count;
    h->K = o.num_mc_samples;
    h->KP = pad_k(h->K);
    h->pdl = !(getenv("POLEE_PDL") && !strcmp(getenv("POLEE_PDL"), "0"));
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->side_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming) != cudaSuccess ||
        polee::dmalloc((void **)&h->d_step, sizeof(StepCtl)) != cudaSuccess ||
        polee::dmalloc((void **)&h->d_bad_step, sizeof(int)) != cudaSuccess ||
        polee::dmalloc((void **)&h->d_leafS_counter, sizeof(unsigned int)) != cudaSuccess ||
        cudaMemsetAsync(h->d_leafS_counter, 0, sizeof(unsigned int), h->stream) != cudaSuccess) {
        delete h;
        return fail(POLEE_ECUDA, "stream / control block allocation failed");
    }
    pt.mark("create: streams + control");
    *out = h;
    return POLEE_OK;
}

static void release_params(polee_handle *h) {
    float *ptrs[] = {h->mu, h->omega, h->alpha, h->m_mu, h->m_omega, h->m_alpha, h->v_mu, h->v_omega, h->v_alpha, h->mu0_dev};
    for (float *p : ptrs) polee::dfree(p);
    h->mu = h->omega = h->alpha = h->m_mu = h->m_omega = h->m_alpha = h->v_mu = h->v_omega = h->v_alpha = h->mu0_dev = nullptr;
}

void polee::drop_step_graph(polee_handle *h) { drop_graph(h); }

extern "C" int polee_destroy(polee_handle *h) {
    if (!h) return POLEE_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (getenv("POLEE_SETUP_TIMING")) polee::dreport("handle lifetime");
    drop_graph(h);
#ifdef POLEE_WITH_NCCL
    polee::peer_release(h);
    if (h->comm) nccl_api().CommDestroy(h->comm);
#endif
    release_work_buffers(h);
    release_matrix(h);
    release_params(h);
    h->td.release();
    polee::dfree(h->efflen); polee::dfree(h->efflen_adj); polee::dfree(h->elbo); polee::dfree(h->noise);
    polee::dfree(h->d_step); polee::dfree(h->d_bad_step); polee::dfree(h->d_leafS_counter);
    release_gene_buffers(h);
    polee::dfree(h->gene_ptr); polee::dfree(h->gene_tx);
    if (h->copy_done) cudaEventDestroy(h->copy_done);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    if (h->side_stream) cudaStreamDestroy(h->side_stream);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return POLEE_OK;
}

extern "C" int polee_trim_memory(int32_t device) {
    polee::dtrim(device);
    return POLEE_OK;
}

extern "C" const char *polee_last_error(const polee_handle *h) {
    if (h) return h->err.c_str();
    std::lock_guard<std::mutex> lk(g_err_mu);
    return g_create_error.c_str();
}

// ------------------------------------------------------------------ inputs
extern "C" int polee_set_matrix_csc_device(polee_handle *h, int64_t m, int64_t n, const uint32_t *d_colptr,
                                           const uint32_t *d_rowval, const float *d_nzval, const int64_t *d_ks) {
    CHECK_H(h);
    if (!d_colptr || (!d_rowval && m > 0) || !d_nzval) return h->fail(POLEE_EINVAL, "set_matrix: null pointer");
    if (h->have_tree && h->td.n != n) return h->fail(POLEE_EINVAL, "n differs from the tree already set");
    drop_graph(h);
    release_work_buffers(h);
    return setup_matrix_from_device_csc(h, m, n, d_colptr, d_rowval, d_nzval, d_ks, nullptr, nullptr);
}

extern "C" int polee_set_matrix_csc(polee_handle *h, int64_t m, int64_t n, const uint32_t *colptr,
                                    const uint32_t *rowval, const float *nzval, const int64_t *ks) {
    CHECK_H(h);
    if (!colptr || !rowval || !nzval) return h->fail(POLEE_EINVAL, "set_matrix: null pointer");
    if (n < 1 || m < 1) return h->fail(POLEE_EINVAL, "set_matrix: m and n must be >= 1");
    if (h->have_tree && h->td.n != n) return h->fail(POLEE_EINVAL, "n differs from the tree already set");
    if (colptr[0] != 1) return h->fail(POLEE_EINVAL, "set_matrix: colptr must be 1-based (colptr[1] == 1)");
    const int64_t nnz = (int64_t)colptr[n] - 1;
    drop_graph(h);
    release_work_buffers(h);
    uint32_t *d_colptr = nullptr, *d_rowval = nullptr;
    float *d_nzval = nullptr;
    int64_t *d_ks = nullptr;
    int rc = POLEE_OK;
    auto cleanup = [&]() { polee::dfree(d_colptr); polee::dfree(d_rowval); polee::dfree(d_nzval); polee::dfree(d_ks); };
#define CKC(expr)                                                                                     \
    do {                                                                                              \
        cudaError_t _e = (expr);                                                                      \
        if (_e != cudaSuccess) {                                                                      \
            cleanup();                                                                                \
            return h->fail(POLEE_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));          \
        }                                                                                             \
    } while (0)
    CKC(polee::dmalloc((void **)&d_colptr, sizeof(uint32_t) * (n + 1)));
    CKC(polee::dmalloc((void **)&d_rowval, sizeof(uint32_t) * std::max<int64_t>(nnz, 1)));
    CKC(polee::dmalloc((void **)&d_nzval, sizeof(float) * std::max<int64_t>(nnz, 1)));
    // the row ids go first on the compute stream (the row-length pass and both sorts need nothing else); the values
    // and counts follow on a side stream so that their transfer overlaps the first half of the layout build
    if (!h->copy_stream) CKC(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    if (!h->copy_done) CKC(cudaEventCreateWithFlags(&h->copy_done, cudaEventDisableTiming));
    CKC(cudaMemcpyAsync(d_colptr, colptr, sizeof(uint32_t) * (n + 1), cudaMemcpyHostToDevice, h->stream));
    CKC(cudaMemcpyAsync(d_rowval, rowval, sizeof(uint32_t) * nnz, cudaMemcpyHostToDevice, h->stream));
    CKC(cudaMemcpyAsync(d_nzval, nzval, sizeof(float) * nnz, cudaMemcpyHostToDevice, h->copy_stream));
    if (ks) {
        CKC(polee::dmalloc((void **)&d_ks, sizeof(int64_t) * m));
        CKC(cudaMemcpyAsync(d_ks, ks, sizeof(int64_t) * m, cudaMemcpyHostToDevice, h->copy_stream));
    }
    CKC(cudaEventRecord(h->copy_done, h->copy_stream));
#undef CKC
    rc = setup_matrix_from_device_csc(h, m, n, d_colptr, d_rowval, d_nzval, d_ks, colptr, h->copy_done);
    cudaStreamSynchronize(h->copy_stream);
    cleanup();
    return rc;
}

extern "C" int polee_set_efflens(polee_handle *h, const float *efflens) {
    CHECK_H(h);
    if (!efflens) return h->fail(POLEE_EINVAL, "set_efflens: null pointer");
    int64_t n = h->have_matrix ? h->n : (h->have_tree ? h->td.n : 0);
    if (n < 1) return h->fail(POLEE_EINVAL, "set_efflens: set the matrix or the tree first (n unknown)");
    drop_graph(h);  // a captured step holds the old buffers' addresses
    polee::dfree(h->efflen); polee::dfree(h->efflen_adj);
    h->efflen = h->efflen_adj = nullptr;
    std::vector<float> adj(n);
    for (int64_t j = 0; j < n; ++j) adj[j] = (float)n * (1.0f / efflens[j]);  // likelihood.jl:105, Float32
    CK(polee::dmalloc((void **)&h->efflen, sizeof(float) * n));
    CK(polee::dmalloc((void **)&h->efflen_adj, sizeof(float) * n));
    CK(polee::copy_sync(h->stream, h->efflen, efflens, sizeof(float) * n, cudaMemcpyHostToDevice));
    CK(polee::copy_sync(h->stream, h->efflen_adj, adj.data(), sizeof(float) * n, cudaMemcpyHostToDevice));
    h->have_efflen = true;
    return patch_leaf_records(h);
}

// Gene groups of gene_noninformative_prior! (likelihood.jl:114-159): the flattened `gene_transcripts` Dict the reference
// builds at likelihood-approximation.jl:476-493.  Only genes with more than one transcript contribute (:123).
extern "C" int polee_set_gene_groups(polee_handle *h, int64_t num_genes, const int64_t *gene_ptr, const int32_t *transcripts) {
    CHECK_H(h);
    drop_graph(h);
    release_gene_buffers(h);
    polee::dfree(h->gene_ptr); polee::dfree(h->gene_tx);
    h->gene_ptr = nullptr; h->gene_tx = nullptr; h->n_genes = 0; h->gene_n = 0;
    if (num_genes == 0) return POLEE_OK;
    if (num_genes < 0 || !gene_ptr || !transcripts) return h->fail(POLEE_EINVAL, "set_gene_groups: null pointer");
    const int64_t n = h->have_matrix ? h->n : (h->have_tree ? h->td.n : 0);
    if (n < 1) return h->fail(POLEE_EINVAL, "set_gene_groups: set the matrix or the tree first (n unknown)");
    if (gene_ptr[0] != 0) return h->fail(POLEE_EINVAL, "set_gene_groups: gene_ptr[0] must be 0");
    std::vector<int64_t> ptr{0};
    std::vector<int32_t> tx;
    std::vector<uint8_t> seen((size_t)n, 0);
    for (int64_t gidx = 0; gidx < num_genes; ++gidx) {
        const int64_t b = gene_ptr[gidx], e = gene_ptr[gidx + 1];
        if (e < b) return h->fail(POLEE_EINVAL, "set_gene_groups: gene_ptr must be non-decreasing");
        for (int64_t q = b; q < e; ++q) {
            const int64_t i = (int64_t)transcripts[q] - 1;  // 1-based ids, as the Dict values
            if (i < 0 || i >= n) return h->fail(POLEE_EINVAL, "set_gene_groups: transcript id out of range 1..n");
            if (seen[i]) return h->fail(POLEE_EINVAL, "set_gene_groups: a transcript belongs to more than one gene");
            seen[i] = 1;
        }
        if (e - b < 2) continue;
        for (int64_t q = b; q < e; ++q) tx.push_back(transcripts[q] - 1);
        ptr.push_back((int64_t)tx.size());
    }
    h->gene_n = n;
    h->n_genes = (int64_t)ptr.size() - 1;
    if (h->n_genes == 0) return POLEE_OK;  // nothing but single-transcript genes: the prior is identically zero
    CK(polee::dmalloc((void **)&h->gene_ptr, sizeof(int64_t) * ptr.size()));
    CK(polee::dmalloc((void **)&h->gene_tx, sizeof(int32_t) * tx.size()));
    CK(polee::copy_sync(h->stream, h->gene_ptr, ptr.data(), sizeof(int64_t) * ptr.size(), cudaMemcpyHostToDevice));
    CK(polee::copy_sync(h->stream, h->gene_tx, tx.data(), sizeof(int32_t) * tx.size(), cudaMemcpyHostToDevice));
    return POLEE_OK;
}

static int alloc_params(polee_handle *h) {
    release_params(h);
    const int64_t nm1 = std::max<int64_t>(h->td.n - 1, 1);
    float **ptrs[] = {&h->mu, &h->omega, &h->alpha, &h->m_mu, &h->m_omega, &h->m_alpha, &h->v_mu, &h->v_omega, &h->v_alpha, &h->mu0_dev};
    for (float **p : ptrs) {
        CK(polee::dmalloc((void **)p, sizeof(float) * nm1));
        CK(cudaMemsetAsync(*p, 0, sizeof(float) * nm1, h->stream));
    }
    return POLEE_OK;
}

// inverse_transform!(t, fill(1.0f0/n, n), ys); map!(logit, mu, ys)   likelihood-approximation.jl:451-453, on the device:
// fills h->mu0_dev (polee_init_params starts every fit from it)
static int initial_mu_device(polee_handle *h) {
    const int64_t n = h->td.n, N = h->td.N;
    if (n < 2) return POLEE_OK;
    float *x0 = nullptr;
    double *us = nullptr, *ys = nullptr;
    struct Release {
        float *&a;
        double *&b, *&c;
        ~Release() { polee::dfree(a); polee::dfree(b); polee::dfree(c); }
    } release{x0, us, ys};
    CK(polee::dmalloc((void **)&x0, sizeof(float) * n));
    CK(polee::dmalloc((void **)&us, sizeof(double) * N));
    CK(polee::dmalloc((void **)&ys, sizeof(double) * (n - 1)));
    int rc = launch_fill_f32(h, x0, n, 1.0f / (float)n);
    if (!rc) rc = launch_tree_inv(h, 1, x0, us, ys, nullptr, nullptr);
    if (!rc) rc = launch_init_params(h, ys, 1);
    cudaError_t e = cudaStreamSynchronize(h->stream);  // the temporaries go back to the cache below
    if (!rc && e != cudaSuccess) rc = h->fail(POLEE_ECUDA, std::string("initial mu: ") + cudaGetErrorString(e));
    return rc;
}

static int finish_tree(polee_handle *h, const std::string &err, HostPhaseTimer &pt) {
    if (!err.empty()) return h->fail(POLEE_EBADTREE, err);
    pt.mark("validate + schedule (host)");
    std::string e2 = upload_tree(h->th, h->td);
    if (!e2.empty()) return h->fail(POLEE_ECUDA, e2);
    pt.mark("upload");
    h->have_tree = true;
    int rc = alloc_params(h);
    if (rc) return rc;
    if ((rc = patch_leaf_records(h))) return rc;
    if ((rc = initial_mu_device(h))) return rc;
    pt.mark("initial mu (device)");
    rc = polee_init_params(h);
    pt.mark("params alloc + init");
    return rc;
}

extern "C" int polee_set_tree(polee_handle *h, int64_t n, const int32_t *node_parent_idxs, const int32_t *node_js) {
    CHECK_H(h);
    if (!node_parent_idxs || !node_js) return h->fail(POLEE_EINVAL, "set_tree: null pointer");
    if (h->have_matrix && h->n != n) return h->fail(POLEE_EINVAL, "set_tree: n differs from the matrix already set");
    drop_graph(h);
    release_work_buffers(h);
    h->have_tree = false;
    HostPhaseTimer pt;
    return finish_tree(h, h->th.build_from_parents(n, node_parent_idxs, node_js, TREE_BIN_NODES), pt);
}

// One RNASeqSample in one call: what polee_set_matrix_csc + polee_set_efflens + polee_set_tree do, with the host-side
// tree work (validation, child pointers, the kernels' schedules: pure host code over h->th, ~25 ms at 200 k transcripts)
// on a second host thread while this thread uploads the matrix and waits for the device to build its layout.  The
// device half of the tree (upload, initial mu) follows once both are done.  Same state, same results.
extern "C" int polee_set_sample(polee_handle *h, int64_t m, int64_t n, const uint32_t *colptr, const uint32_t *rowval,
                                const float *nzval, const int64_t *ks, const float *efflens,
                                const int32_t *node_parent_idxs, const int32_t *node_js) {
    CHECK_H(h);
    if (!node_parent_idxs || !node_js || !efflens) return h->fail(POLEE_EINVAL, "set_sample: null pointer");
    drop_graph(h);
    release_work_buffers(h);
    h->have_tree = false;  // nothing on this thread reads h->th / h->td until the worker has been joined
    HostPhaseTimer pt;
    std::string tree_err;
    struct Joiner {
        std::thread t;
        ~Joiner() { if (t.joinable()) t.join(); }
    } worker{std::thread([&]() {
        try {
            tree_err = h->th.build_from_parents(n, node_parent_idxs, node_js, TREE_BIN_NODES);
        } catch (const std::exception &e) {
            tree_err = std::string("tree: ") + e.what();
        }
    })};
    // a third thread loads the kernels of the ADAM step (lazy module loading would otherwise do that at their first
    // launch, with the device idle); POLEE_PRELOAD=0 turns it off
    static const bool preload = !(getenv("POLEE_PRELOAD") && !strcmp(getenv("POLEE_PRELOAD"), "0"));
    Joiner loader{preload && h->o.approx == POLEE_APPROX_LOGIT_SKEW_NORMAL_PTT ? std::thread([h]() {
        if (cudaSetDevice(h->device) != cudaSuccess) return;
        polee::preload_ec_kernels(h, h->KP, h->K);
        polee::preload_tree_kernels(h->KP);
    }) : std::thread()};
    int rc = polee_set_matrix_csc(h, m, n, colptr, rowval, nzval, ks);
    if (!rc) rc = polee_set_efflens(h, efflens);
    pt.mark("matrix + efflens (this thread)");
    worker.t.join();
    if (loader.t.joinable()) loader.t.join();
    if (rc) return rc;
    return finish_tree(h, tree_err, pt);
}

extern "C" int polee_set_tree_sequential(polee_handle *h, int64_t n) {
    CHECK_H(h);
    if (n < 1) return h->fail(POLEE_EINVAL, "set_tree_sequential: n must be >= 1");
    // list_nodes + order_nodes (hclust.jl:477-489, 361-389): root, leaf 1, I, leaf 2, ..., leaf n-1, leaf n
    const int64_t N = 2 * n - 1;
    std::vector<int32_t> pi(N), js(N);
    int64_t pos = 0;
    int32_t parent = 0;
    for (int64_t leaf = 1; leaf <= n - 1; ++leaf) {
        pi[pos] = parent; js[pos] = 0;
        int32_t me = (int32_t)(pos + 1);
        ++pos;
        pi[pos] = me; js[pos] = (int32_t)leaf;
        ++pos;
        parent = me;
    }
    pi[pos] = parent; js[pos] = (int32_t)n;
    return polee_set_tree(h, n, pi.data(), js.data());
}

// ------------------------------------------------------------------ parameters
extern "C" int polee_init_params(polee_handle *h) {
    CHECK_H(h);
    if (!h->have_tree) return h->fail(POLEE_EINVAL, "init_params: set the tree first");
    const int64_t nm1 = h->td.n - 1;
    if (nm1 > 0) {
        int rc = launch_init_params(h, nullptr, 1);  // mu0, log(0.1f0), 0: likelihood-approximation.jl:451-456
        if (rc) return rc;
        float *st[] = {h->m_mu, h->m_omega, h->m_alpha, h->v_mu, h->v_omega, h->v_alpha};
        for (float *p : st) CK(cudaMemsetAsync(p, 0, sizeof(float) * nm1, h->stream));
    }
    StepCtl c{1, 1};
    CK(polee::copy_sync(h->stream, h->d_step, &c, sizeof(c), cudaMemcpyHostToDevice));
    CK(cudaMemsetAsync(h->d_bad_step, 0, sizeof(int), h->stream));
    h->steps_enqueued = 0;
    h->reparam_ready = false;
    return POLEE_OK;
}

extern "C" int polee_get_params(polee_handle *h, float *mu, float *omega, float *alpha) {
    CHECK_H(h);
    if (!h->have_tree) return h->fail(POLEE_EINVAL, "get_params: set the tree first");
    const int64_t nm1 = h->td.n - 1;
    CK(cudaStreamSynchronize(h->stream));
    if (nm1 > 0) {
        if (mu) CK(polee::copy_sync(h->stream, mu, h->mu, sizeof(float) * nm1, cudaMemcpyDeviceToHost));
        if (omega) CK(polee::copy_sync(h->stream, omega, h->omega, sizeof(float) * nm1, cudaMemcpyDeviceToHost));
        if (alpha) CK(polee::copy_sync(h->stream, alpha, h->alpha, sizeof(float) * nm1, cudaMemcpyDeviceToHost));
    }
    return POLEE_OK;
}

extern "C" int polee_set_params(polee_handle *h, const float *mu, const float *omega, const float *alpha) {
    CHECK_H(h);
    if (!h->have_tree) return h->fail(POLEE_EINVAL, "set_params: set the tree first");
    const int64_t nm1 = h->td.n - 1;
    CK(cudaStreamSynchronize(h->stream));
    if (nm1 > 0) {
        if (mu) CK(polee::copy_sync(h->stream, h->mu, mu, sizeof(float) * nm1, cudaMemcpyHostToDevice));
        if (omega) CK(polee::copy_sync(h->stream, h->omega, omega, sizeof(float) * nm1, cudaMemcpyHostToDevice));
        if (alpha) CK(polee::copy_sync(h->stream, h->alpha, alpha, sizeof(float) * nm1, cudaMemcpyHostToDevice));
    }
    h->reparam_ready = false;
    return POLEE_OK;
}

extern "C" int polee_set_noise(polee_handle *h, const float *noise, int64_t num_steps) {
    CHECK_H(h);
    if (!h->have_tree) return h->fail(POLEE_EINVAL, "set_noise: set the tree first");
    drop_graph(h);
    h->reparam_ready = false;
    polee::dfree(h->noise);
    h->noise = nullptr;
    h->noise_steps = 0;
    if (!noise || num_steps <= 0) return POLEE_OK;
    const size_t count = (size_t)num_steps * h->K * (size_t)std::max<int64_t>(h->td.n - 1, 1);
    CK(polee::dmalloc((void **)&h->noise, sizeof(float) * count));
    CK(polee::copy_sync(h->stream, h->noise, noise, sizeof(float) * count, cudaMemcpyHostToDevice));
    h->noise_steps = num_steps;
    return POLEE_OK;
}

extern "C" void *polee_stream(polee_handle *h) { return h ? (void *)h->stream : nullptr; }

// ------------------------------------------------------------------ one ADAM step
static int ready_for_steps(polee_handle *h) {
    if (!h->have_matrix) return h->fail(POLEE_EINVAL, "no matrix: call polee_set_matrix_csc first");
    if (!h->have_tree) return h->fail(POLEE_EINVAL, "no tree: call polee_set_tree first");
    if (h->n != h->td.n) return h->fail(POLEE_EINVAL, "matrix and tree disagree on n");
    const bool need_eff = h->o.use_efflen_jacobian || h->o.approx == POLEE_APPROX_OPTIMIZE_PTT;
    if (need_eff && !h->have_efflen) return h->fail(POLEE_EINVAL, "no effective lengths: call polee_set_efflens first");
    if (h->n_genes > 0) {
        // the reference reads xls, which only effective_length_jacobian_adjustment! fills (likelihood.jl:98-101), and
        // the factored / OptimizePTT entries have no gene prior (likelihood-approximation.jl:248-251, :149-151)
        if (h->gene_n != h->n) return h->fail(POLEE_EINVAL, "gene groups were set for a different n");
        if (h->o.approx != POLEE_APPROX_LOGIT_SKEW_NORMAL_PTT || h->row_weight || h->ft_row_weight || h->ec_slot_weight)
            return h->fail(POLEE_EINVAL, "gene groups: the prior exists only in the unweighted LogitSkewNormalPTTApprox fit");
        if (!h->o.use_efflen_jacobian)
            return h->fail(POLEE_EINVAL, "gene groups need use_efflen_jacobian (the prior reads the scaled abundances it computes)");
    }
    if (h->o.noise_mode == POLEE_NOISE_INJECTED && h->o.approx == POLEE_APPROX_LOGIT_SKEW_NORMAL_PTT && !h->noise)
        return h->fail(POLEE_EINVAL, "noise_mode is INJECTED but no noise was supplied");
    int rc = ensure_work_buffers(h, h->KP);
    if (rc) return rc;
    if ((rc = ensure_gene_buffers(h, h->KP))) return rc;
    if (!h->elbo) {
        CK(polee::dmalloc((void **)&h->elbo, sizeof(double) * std::max(h->o.num_steps, 1)));
        CK(cudaMemsetAsync(h->elbo, 0, sizeof(double) * std::max(h->o.num_steps, 1), h->stream));
    }
    return POLEE_OK;
}

// log-likelihood gradient of the KP draws in h->x: the equivalence-class pass, plus -- for the rows it did not take, or
// for all rows when it is switched off -- the fused single pass or K1 + K2 on the split layout
static int launch_likelihood(polee_handle *h, int KP, int K, bool want_lp) {
    int rc;
    const bool general = h->gm > 0 || h->ec_tasks == 0;
    double *lp_out = h->g + (size_t)h->n * KP;
    if (general) {
        if (h->fused) {
            if ((rc = launch_fused(h, h->x, h->g, want_lp, h->lp_partial, nullptr, KP))) return rc;
        } else {
            if ((rc = launch_k1(h, h->x, h->w, want_lp, h->lp_partial, KP))) return rc;
            if ((rc = launch_k2(h, h->w, h->g, KP))) return rc;
        }
        if (want_lp && (rc = launch_reduce_lp(h, h->lp_partial, lp_out, KP))) return rc;
    }
    if (h->ec_tasks > 0 && (rc = launch_ec(h, h->x, h->g, general, want_lp, lp_out, nullptr, KP, K))) return rc;
    return POLEE_OK;
}

// the per-step sum of g (and, when requested, of the K log-likelihood sums) over the ranks of a row-partitioned fit
static int launch_allreduce(polee_handle *h, int KP, bool want_vals) {
#ifdef POLEE_WITH_NCCL
    if (h->nranks > 1) {
        int rc;
        // The gradient crosses NVLink as Float32 (6.4 MB instead of 12.8 MB at C3; every rank's partial g is a sum of
        // positive Float32-accurate terms, so nothing is lost that the 1e-5 gate could see); the K log-likelihood
        // sums, when requested, stay Float64.  POLEE_ALLREDUCE=f64 keeps the whole buffer in Float64.
        static const bool f64 = getenv("POLEE_ALLREDUCE") && !strcmp(getenv("POLEE_ALLREDUCE"), "f64");
        static const bool nccl_only = getenv("POLEE_ALLREDUCE") && !strcmp(getenv("POLEE_ALLREDUCE"), "nccl");
        const size_t count = (size_t)h->n * KP;
        ncclResult_t r = ncclSuccess;
        if (h->peer_ready && !f64 && !nccl_only) {
            // one kernel over NVLink peer memory (peer_allreduce.cu): narrow, reduce-scatter by loads, all-gather by
            // stores, widen; the K log-likelihood sums, when requested, still go through NCCL as Float64
            if ((rc = polee::launch_peer_allreduce(h, h->g, count))) return rc;
            if (want_vals) r = nccl_api().AllReduce(h->g + count, h->g + count, KP, ncclDouble, ncclSum, h->comm, h->stream);
        } else if (f64 || !h->g32) {
            r = nccl_api().AllReduce(h->g, h->g, count + (want_vals ? KP : 0), ncclDouble, ncclSum, h->comm, h->stream);
        } else {
            if ((rc = launch_narrow(h, h->g, h->g32, count))) return rc;
            r = nccl_api().AllReduce(h->g32, h->g32, count, ncclFloat, ncclSum, h->comm, h->stream);
            if (r == ncclSuccess && want_vals)
                r = nccl_api().AllReduce(h->g + count, h->g + count, KP, ncclDouble, ncclSum, h->comm, h->stream);
            if (r == ncclSuccess && (rc = launch_widen(h, h->g32, h->g, count))) return rc;
        }
        if (r != ncclSuccess) return h->fail(POLEE_ENCCL, std::string("ncclAllReduce: ") + nccl_api().GetErrorString(r));
    }
#else
    (void)h; (void)KP; (void)want_vals;
#endif
    return POLEE_OK;
}

// The launch sequence of one step (SURVEY 3a inner loop, batched over the K draws).  ys / zs0 of the step are
// produced by the previous step's fused update+reparam kernel (or by ensure_reparam for the first step):
//   tree fwd (top, bottom) -> mid -> K1 -> K2 (+combine) -> [lp reduce] -> [all-reduce] -> tree bwd (bottom, top)
//   -> [elbo] -> update(step s) + reparam(step s+1)
static int launch_step_sequence(polee_handle *h, bool do_adam, bool next_reparam, float *grad_out, double *xgrad_out,
                                const float *noise, int64_t noise_steps) {
    const int KP = h->KP, K = h->K;
    const bool lsn = h->o.approx == POLEE_APPROX_LOGIT_SKEW_NORMAL_PTT;
    const bool want_vals = lsn && !h->o.gradonly;
    const bool apply_eff = lsn ? (h->o.use_efflen_jacobian != 0) : true;
    int rc;
    if ((rc = launch_tree_fwd(h, KP, 1, apply_eff, want_vals))) return rc;
    // k3_mid (the S reduction and the step counters) depends only on the tree pass and is needed only by the backward
    // pass: it runs on a side stream beside the likelihood pass (a fork / join that the graph capture records too)
    CK(cudaEventRecord(h->ev_fork, h->stream));
    CK(cudaStreamWaitEvent(h->side_stream, h->ev_fork, 0));
    if ((rc = launch_mid(h, KP, do_adam ? 1 : 0, h->side_stream))) return rc;
    CK(cudaEventRecord(h->ev_join, h->side_stream));
    if ((rc = launch_likelihood(h, KP, K, want_vals))) return rc;
    CK(cudaStreamWaitEvent(h->stream, h->ev_join, 0));
    if ((rc = launch_allreduce(h, KP, want_vals))) return rc;
    if (h->n_genes > 0 && (rc = launch_gene_prior(h, KP))) return rc;
    if ((rc = launch_tree_bwd(h, KP, lsn, apply_eff, xgrad_out))) return rc;
    if (want_vals && (rc = launch_elbo(h, KP, K, true))) return rc;
    if ((rc = launch_elem(h, KP, K, true, do_adam, next_reparam, noise, noise_steps, next_reparam && want_vals, grad_out)))
        return rc;
    return POLEE_OK;
}

// first step after (re)initialisation: produce ys / zs0 for the step the counters point at
static int ensure_reparam(polee_handle *h) {
    if (h->reparam_ready) return POLEE_OK;
    const bool lsn = h->o.approx == POLEE_APPROX_LOGIT_SKEW_NORMAL_PTT;
    const float *noise = h->o.noise_mode == POLEE_NOISE_INJECTED ? h->noise : nullptr;
    int rc = launch_elem(h, h->KP, h->K, false, false, true, noise, std::max<int64_t>(h->noise_steps, 1),
                         lsn && !h->o.gradonly, nullptr);
    if (rc) return rc;
    h->reparam_ready = true;
    return POLEE_OK;
}

// nsteps consecutive steps captured into one graph.  The step number and the learning rate live in device memory
// (StepCtl), so a replay is the same as enqueueing the steps one by one.
static int capture_steps(polee_handle *h, int nsteps, cudaGraph_t *graph, cudaGraphExec_t *exec) {
    const float *noise = h->o.noise_mode == POLEE_NOISE_INJECTED ? h->noise : nullptr;
    // Relaxed: other host threads (one handle per thread in `polee prep`) may allocate, free or synchronise while
    // this thread records; the handle's streams are non-blocking, so nothing they do can join this capture.
    std::shared_lock<std::shared_mutex> cap(polee::capture_mutex());  // no device-wide sync anywhere meanwhile
    CK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeRelaxed));
    int rc = POLEE_OK;
    for (int s = 0; s < nsteps && !rc; ++s)
        rc = launch_step_sequence(h, true, true, nullptr, nullptr, noise, std::max<int64_t>(h->noise_steps, 1));
    cudaError_t e = cudaStreamEndCapture(h->stream, graph);
    if (rc) return rc;
    if (e != cudaSuccess) return h->fail(POLEE_ECUDA, std::string("graph capture: ") + cudaGetErrorString(e));
    CK(cudaGraphInstantiate(exec, *graph, 0));
    return POLEE_OK;
}

// STEP_GRAPH_STEPS steps in one graph launch; the caller has run enqueue_step at least once
static int enqueue_step_chunk(polee_handle *h) {
    int rc = ensure_reparam(h);  // init_params, set_params, polee_sample ... leave ys / zs0 for the graph to redo
    if (rc) return rc;
    if (!h->graph_multi_exec) {
        HostPhaseTimer pt;
        if ((rc = capture_steps(h, STEP_GRAPH_STEPS, &h->graph_multi, &h->graph_multi_exec))) return rc;
        pt.mark("multi-step graph: capture + inst.");
    }
    CK(cudaGraphLaunch(h->graph_multi_exec, h->stream));
    return POLEE_OK;
}

static int enqueue_step(polee_handle *h) {
    const float *noise = h->o.noise_mode == POLEE_NOISE_INJECTED ? h->noise : nullptr;
    int rc = ensure_reparam(h);
    if (rc) return rc;
    if (!h->o.use_cuda_graph) {
        rc = launch_step_sequence(h, true, true, nullptr, nullptr, noise, std::max<int64_t>(h->noise_steps, 1));
        if (rc) return rc;
        CK(cudaGetLastError());
        return POLEE_OK;
    }
    if (!h->graph_warm) {
        // the first step of a handle runs uncaptured: every kernel it needs is then loaded before a capture starts
        // (lazy module loading allocates, which a capture does not tolerate)
        HostPhaseTimer pt;
        rc = launch_step_sequence(h, true, true, nullptr, nullptr, noise, std::max<int64_t>(h->noise_steps, 1));
        if (rc) return rc;
        CK(cudaGetLastError());
        h->graph_warm = true;
        pt.mark("first step: enqueue (uncaptured)");
        return POLEE_OK;
    }
    if (!h->graph_exec) {
        HostPhaseTimer pt;
        if ((rc = capture_steps(h, 1, &h->graph, &h->graph_exec))) return rc;
        pt.mark("second step: capture + instantiate");
    }
    CK(cudaGraphLaunch(h->graph_exec, h->stream));
    return POLEE_OK;
}

extern "C" int polee_run_steps(polee_handle *h, int32_t nsteps) {
    CHECK_H(h);
    HostPhaseTimer pt;
    pt.on = pt.on && !h->graph_warm;
    int rc = ready_for_steps(h);
    if (rc) return rc;
    pt.mark("run_steps: work buffers");
    const bool progress = h->progress_cb && h->progress_every > 0;
    for (int s = 0; s < nsteps;) {
        // the multi-step graph once the one-step graph exists, while a whole chunk remains and no progress report
        // falls inside it (one may fall on its last step).  It is captured only after this call has queued
        // STEP_GRAPH_LEAD steps: its capture and instantiation (~1 ms of host time) then overlap their execution
        // instead of leaving the device idle.
        int chunk = 1;
        if (h->graph_exec && (h->graph_multi_exec || s >= STEP_GRAPH_LEAD) && nsteps - s >= STEP_GRAPH_STEPS) {
            chunk = STEP_GRAPH_STEPS;
            for (int j = 1; progress && j < STEP_GRAPH_STEPS; ++j)
                if ((h->steps_enqueued + j) % h->progress_every == 0) chunk = 1;
        }
        if ((rc = chunk > 1 ? enqueue_step_chunk(h) : enqueue_step(h))) return rc;
        h->steps_enqueued += chunk;
        s += chunk;
        if (progress && (h->steps_enqueued % h->progress_every == 0 || s == nsteps)) {
            CK(cudaStreamSynchronize(h->stream));  // the bar reports finished steps, not enqueued ones
            h->progress_cb(h->steps_enqueued, h->o.num_steps, h->progress_user);
        }
    }
    return POLEE_OK;
}

extern "C" int polee_set_progress(polee_handle *h, polee_progress_fn cb, void *user, int32_t every) {
    CHECK_H(h);
    if (cb && every < 1) return h->fail(POLEE_EINVAL, "set_progress: every must be >= 1");
    h->progress_cb = cb;
    h->progress_user = user;
    h->progress_every = cb ? every : 0;
    return POLEE_OK;
}

extern "C" int polee_sync(polee_handle *h) {
    CHECK_H(h);
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    int bad = 0;
    CK(polee::copy_sync(h->stream, &bad, h->d_bad_step, sizeof(int), cudaMemcpyDeviceToHost));
    if (bad == polee::PEER_ERR_TIMEOUT) return h->fail(POLEE_ENCCL, "peer all-reduce: a rank did not arrive within the time limit");
    if (bad) return h->fail(POLEE_ENONFINITE, "non-finite gradient at step " + std::to_string(bad));
    return POLEE_OK;
}

extern "C" int polee_get_elbo(polee_handle *h, double *elbo, int32_t nsteps) {
    CHECK_H(h);
    if (!h->elbo || !elbo) return h->fail(POLEE_EINVAL, "get_elbo: nothing recorded");
    CK(cudaStreamSynchronize(h->stream));
    CK(polee::copy_sync(h->stream, elbo, h->elbo, sizeof(double) * std::min(nsteps, std::max(h->o.num_steps, 1)), cudaMemcpyDeviceToHost));
    return POLEE_OK;
}

extern "C" int polee_fit(polee_handle *h, float *mu, float *omega, float *alpha, double *elbo_traj, const float *noise) {
    CHECK_H(h);
    if (h->o.approx != POLEE_APPROX_LOGIT_SKEW_NORMAL_PTT) return h->fail(POLEE_EINVAL, "polee_fit: handle was created for OptimizePTTApprox");
    int rc;
    if (h->o.noise_mode == POLEE_NOISE_INJECTED) {
        if (!noise && !h->noise) return h->fail(POLEE_EINVAL, "polee_fit: noise_mode is INJECTED but noise == NULL");
        if (noise && (rc = polee_set_noise(h, noise, h->o.num_steps))) return rc;
    }
    if ((rc = polee_init_params(h))) return rc;
    if ((rc = polee_run_steps(h, h->o.num_steps))) return rc;
    if ((rc = polee_sync(h))) return rc;
    if ((rc = polee_get_params(h, mu, omega, alpha))) return rc;
    if (elbo_traj) {
        if (h->o.gradonly)
            std::fill(elbo_traj, elbo_traj + h->o.num_steps, 0.0);  // reference: elbo == 0 when gradonly (SURVEY App. C2)
        else if ((rc = polee_get_elbo(h, elbo_traj, h->o.num_steps)))
            return rc;
    }
    return POLEE_OK;
}

// ------------------------------------------------------------------ layout helpers ([K][len] host <-> [len][KP] device)
template <typename T>
static int upload_kmajor(polee_handle *h, const T *host, int K, int KP, int64_t len, T *dev, T pad) {
    std::vector<T> tmp((size_t)len * KP, pad);
    for (int k = 0; k < K; ++k)
        for (int64_t i = 0; i < len; ++i) tmp[(size_t)i * KP + k] = host[(size_t)k * len + i];
    CK(cudaMemcpyAsync(dev, tmp.data(), sizeof(T) * tmp.size(), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return POLEE_OK;
}
template <typename T, typename U>
static int download_kmajor(polee_handle *h, const T *dev, int K, int KP, int64_t len, U *host) {
    std::vector<T> tmp((size_t)len * KP);
    CK(cudaStreamSynchronize(h->stream));
    CK(polee::copy_sync(h->stream, tmp.data(), dev, sizeof(T) * tmp.size(), cudaMemcpyDeviceToHost));
    for (int k = 0; k < K; ++k)
        for (int64_t i = 0; i < len; ++i) host[(size_t)k * len + i] = (U)tmp[(size_t)i * KP + k];
    return POLEE_OK;
}

static int use_kp(polee_handle *h, int K, int *KP) {
    if (K < 1 || K > 16) return h->fail(POLEE_EINVAL, "K must be in 1..16");
    *KP = pad_k(K);
    drop_graph(h);
    // every piecewise entry point comes through here and overwrites (or re-creates) ys / zs0 / x / g: the next
    // polee_run_steps must produce its own reparameterisation again instead of stepping on the caller's values
    h->reparam_ready = false;
    return ensure_work_buffers(h, *KP);
}

// after a piecewise call with a different KP, the fit's buffers are re-created lazily
extern "C" int polee_fit_optimize_ptt(polee_handle *h, float *xs) {
    CHECK_H(h);
    if (h->o.approx != POLEE_APPROX_OPTIMIZE_PTT) return h->fail(POLEE_EINVAL, "handle was not created with POLEE_APPROX_OPTIMIZE_PTT");
    if (!h->have_matrix) return h->fail(POLEE_EINVAL, "no matrix: call polee_set_matrix_csc first");
    int rc;
    if ((rc = polee_set_tree_sequential(h, h->n))) return rc;   // PolyaTreeTransform(X, :sequential)  l-a.jl:160
    if ((rc = polee_run_steps(h, h->o.num_steps))) return rc;
    if ((rc = polee_sync(h))) return rc;
    // final transform of the optimised zs  (l-a.jl:237-241)
    if ((rc = launch_reparam_fwd(h, h->KP, h->K, nullptr, 1, 0))) return rc;
    h->reparam_ready = false;
    if ((rc = launch_tree_fwd(h, h->KP, 1, 0, 0))) return rc;
    return download_kmajor<float, float>(h, h->x, 1, h->KP, h->n, xs);
}

// ------------------------------------------------------------------ piecewise entry points
extern "C" int polee_loglik_grad(polee_handle *h, const float *xs, int32_t K, int32_t gradonly, double *lp, double *x_grad) {
    CHECK_H(h);
    if (!h->have_matrix) return h->fail(POLEE_EINVAL, "no matrix: call polee_set_matrix_csc first");
    if (!h->have_tree) return h->fail(POLEE_EINVAL, "loglik_grad: set a tree first (work buffers are sized from it)");
    int KP, rc;
    if ((rc = use_kp(h, K, &KP))) return rc;
    if ((rc = upload_kmajor<float>(h, xs, K, KP, h->n, h->x, 1.0f))) return rc;
    if ((rc = launch_likelihood(h, KP, K, !gradonly))) return rc;
    CK(cudaGetLastError());
    if (x_grad && (rc = download_kmajor<double, double>(h, h->g, K, KP, h->n, x_grad))) return rc;
    if (lp) {
        if (gradonly) {
            std::fill(lp, lp + K, 0.0);
        } else {
            std::vector<double> t(KP);
            CK(cudaStreamSynchronize(h->stream));
            CK(polee::copy_sync(h->stream, t.data(), h->g + (size_t)h->n * KP, sizeof(double) * KP, cudaMemcpyDeviceToHost));
            std::copy(t.begin(), t.begin() + K, lp);
        }
    }
    CK(cudaStreamSynchronize(h->stream));
    return POLEE_OK;
}

extern "C" int polee_frag_prob_recip(polee_handle *h, const float *xs, float *w) {
    CHECK_H(h);
    if (!h->have_matrix || !h->have_tree) return h->fail(POLEE_EINVAL, "frag_prob_recip: set the matrix and a tree first");
    int KP, rc;
    if ((rc = use_kp(h, 1, &KP))) return rc;
    if ((rc = upload_kmajor<float>(h, xs, 1, KP, h->n, h->x, 1.0f))) return rc;
    const bool general = h->gm > 0 || h->ec_tasks == 0;
    float *d_w = nullptr;
    struct Release {
        float *&p;
        ~Release() { polee::dfree(p); }
    } release{d_w};
    if (h->ec_tasks > 0) {  // the class layout scatters 1/p to the rows' original positions
        CK(polee::dmalloc((void **)&d_w, sizeof(float) * (size_t)h->m * KP));
        CK(cudaMemsetAsync(d_w, 0, sizeof(float) * (size_t)h->m * KP, h->stream));
        if ((rc = launch_ec(h, h->x, h->g, false, false, nullptr, d_w, KP, 1))) return rc;
        CK(cudaStreamSynchronize(h->stream));
        std::vector<float> wp((size_t)h->m * KP);
        CK(polee::copy_sync(h->stream, wp.data(), d_w, sizeof(float) * wp.size(), cudaMemcpyDeviceToHost));
        for (int64_t i = 0; i < h->m; ++i) w[i] = wp[(size_t)i * KP];
        polee::dfree(d_w);
        d_w = nullptr;
    }
    if (!general) return POLEE_OK;
    // the general layouts hold gm rows (all of them, or the rest rows, whose original positions are in rest_row)
    std::vector<float> wr((size_t)h->gm);
    if (h->fused) {  // rows keep their order in the fused layout
        CK(polee::dmalloc((void **)&d_w, sizeof(float) * (size_t)h->gm * KP));
        rc = launch_fused(h, h->x, h->g, false, h->lp_partial, d_w, KP);
        cudaError_t e = cudaStreamSynchronize(h->stream);
        if (!rc && e != cudaSuccess) rc = h->fail(POLEE_ECUDA, std::string("frag_prob_recip: ") + cudaGetErrorString(e));
        if (rc) return rc;
        std::vector<float> wp((size_t)h->gm * KP);
        CK(polee::copy_sync(h->stream, wp.data(), d_w, sizeof(float) * wp.size(), cudaMemcpyDeviceToHost));
        for (int64_t i = 0; i < h->gm; ++i) wr[i] = wp[(size_t)i * KP];
    } else {
        if ((rc = launch_k1(h, h->x, h->w, false, h->lp_partial, KP))) return rc;
        CK(cudaStreamSynchronize(h->stream));
        std::vector<float> wp(h->m_pad);
        std::vector<uint32_t> perm(h->gm);
        CK(polee::copy_sync(h->stream, wp.data(), h->w, sizeof(float) * h->m_pad, cudaMemcpyDeviceToHost));
        CK(polee::copy_sync(h->stream, perm.data(), h->row_perm, sizeof(uint32_t) * h->gm, cudaMemcpyDeviceToHost));
        for (int64_t i = 0; i < h->gm; ++i) wr[i] = wp[perm[i]];
    }
    if (h->rest_row) {
        std::vector<uint32_t> rr((size_t)h->gm);
        CK(polee::copy_sync(h->stream, rr.data(), h->rest_row, sizeof(uint32_t) * h->gm, cudaMemcpyDeviceToHost));
        for (int64_t i = 0; i < h->gm; ++i) w[rr[i]] = wr[i];
    } else {
        std::copy(wr.begin(), wr.end(), w);
    }
    return POLEE_OK;
}

extern "C" int polee_ptt_transform(polee_handle *h, const double *ys, int32_t K, float *xs, double *ladj) {
    CHECK_H(h);
    if (!h->have_tree) return h->fail(POLEE_EINVAL, "no tree: call polee_set_tree first");
    h->n = h->td.n;
    int KP, rc;
    if ((rc = use_kp(h, K, &KP))) return rc;
    if ((rc = upload_kmajor<double>(h, ys, K, KP, h->n - 1, h->ys, 0.5))) return rc;
    if ((rc = launch_tree_fwd(h, KP, 0, 0, ladj ? 1 : 0))) return rc;
    CK(cudaGetLastError());
    if ((rc = download_kmajor<float, float>(h, h->x, K, KP, h->n, xs))) return rc;
    if (ladj) {
        const int ne = elem_ctas(h, KP);
        std::vector<double> part((size_t)h->n_tree_ctas * KP);
        CK(polee::copy_sync(h->stream, part.data(), h->ladj_partial + (size_t)2 * ne * KP, sizeof(double) * part.size(), cudaMemcpyDeviceToHost));
        for (int k = 0; k < K; ++k) {
            double s = 0.0;
            for (int t = 0; t < h->n_tree_ctas; ++t) s += part[(size_t)t * KP + k];
            ladj[k] = s;
        }
    }
    return POLEE_OK;
}

extern "C" int polee_ptt_transform_gradients(polee_handle *h, const double *ys, const double *x_grad, int32_t K,
                                             int32_t with_ladj, float *y_grad) {
    CHECK_H(h);
    if (!h->have_tree) return h->fail(POLEE_EINVAL, "no tree: call polee_set_tree first");
    h->n = h->td.n;
    int KP, rc;
    if ((rc = use_kp(h, K, &KP))) return rc;
    if ((rc = upload_kmajor<double>(h, ys, K, KP, h->n - 1, h->ys, 0.5))) return rc;
    if ((rc = upload_kmajor<double>(h, x_grad, K, KP, h->n, h->g, 0.0))) return rc;
    if ((rc = launch_tree_fwd(h, KP, 0, 0, 0))) return rc;  // us, as transform! leaves them in t.us
    if ((rc = launch_tree_bwd(h, KP, with_ladj != 0, false, nullptr))) return rc;
    CK(cudaGetLastError());
    return download_kmajor<double, float>(h, h->ygrad, K, KP, h->n - 1, y_grad);
}

// inverse_transform!  ptt.jl:257-285 on the device (k3_tree_inv: level-synchronous bottom-up sums, the reference's
// association; ladj accumulated in the reference's order)
extern "C" int polee_ptt_inverse_transform(polee_handle *h, const float *xs, int32_t K, double *ys, double *ladj) {
    CHECK_H(h);
    if (!h->have_tree) return h->fail(POLEE_EINVAL, "no tree: call polee_set_tree first");
    if (!xs || !ys) return h->fail(POLEE_EINVAL, "ptt_inverse_transform: null pointer");
    h->n = h->td.n;
    int KP, rc;
    if ((rc = use_kp(h, K, &KP))) return rc;
    const int64_t n = h->td.n, nm1 = n - 1;
    if (nm1 < 1) {
        if (ladj) for (int k = 0; k < K; ++k) ladj[k] = 0.0;
        return POLEE_OK;
    }
    // work buffers of the step double as scratch: x <- xs, us (by node), ygrad <- ys, zs <- log u, S <- ladj
    if ((rc = upload_kmajor<float>(h, xs, K, KP, n, h->x, 1.0f))) return rc;
    if ((rc = launch_tree_inv(h, KP, h->x, h->us, h->ygrad, h->zs, ladj ? h->S : nullptr))) return rc;
    CK(cudaGetLastError());
    if ((rc = download_kmajor<double, double>(h, h->ygrad, K, KP, nm1, ys))) return rc;
    if (ladj) {
        std::vector<double> l(KP);
        CK(polee::copy_sync(h->stream, l.data(), h->S, sizeof(double) * KP, cudaMemcpyDeviceToHost));
        std::copy(l.begin(), l.begin() + K, ladj);
    }
    return POLEE_OK;
}

extern "C" int polee_lsn_draws(polee_handle *h, const float *zs0, int32_t K, float *xs, double *ys, double *x_grad,
                               float *y_grad, float *mu_grad, float *omega_grad, float *alpha_grad, double *elbo) {
    CHECK_H(h);
    if (K != h->K) return h->fail(POLEE_EINVAL, "lsn_draws: K must equal opts.num_mc_samples");
    if (!zs0) return h->fail(POLEE_EINVAL, "lsn_draws: zs0 == NULL");
    int rc = ready_for_steps(h);
    if (rc == POLEE_EINVAL && !h->noise && h->o.noise_mode == POLEE_NOISE_INJECTED && h->have_matrix && h->have_tree) {
        h->err.clear();
        rc = ensure_work_buffers(h, h->KP);
        if (!rc) rc = ensure_gene_buffers(h, h->KP);
        if (!rc && !h->elbo) {
            CK(polee::dmalloc((void **)&h->elbo, sizeof(double) * std::max(h->o.num_steps, 1)));
            CK(cudaMemsetAsync(h->elbo, 0, sizeof(double) * std::max(h->o.num_steps, 1), h->stream));
        }
    }
    if (rc) return rc;
    const int KP = h->KP;
    const int64_t n = h->n, nm1 = n - 1;
    float *d_noise = nullptr;
    double *d_xg = nullptr;
    struct Release {  // the temporaries go back to the cache on every exit path
        float *&a;
        double *&b;
        ~Release() { polee::dfree(a); polee::dfree(b); }
    } release{d_noise, d_xg};
    CK(polee::dmalloc((void **)&d_noise, sizeof(float) * (size_t)K * std::max<int64_t>(nm1, 1)));
    CK(polee::dmalloc((void **)&d_xg, sizeof(double) * (size_t)n * KP));
    CK(polee::copy_sync(h->stream, d_noise, zs0, sizeof(float) * (size_t)K * nm1, cudaMemcpyHostToDevice));
    StepCtl saved, one{1, 1};
    CK(cudaStreamSynchronize(h->stream));
    CK(polee::copy_sync(h->stream, &saved, h->d_step, sizeof(saved), cudaMemcpyDeviceToHost));
    CK(polee::copy_sync(h->stream, h->d_step, &one, sizeof(one), cudaMemcpyHostToDevice));
    rc = launch_elem(h, KP, K, false, false, true, d_noise, 1, !h->o.gradonly, nullptr);
    if (!rc) rc = launch_step_sequence(h, false, false, h->grad_out, d_xg, d_noise, 1);
    h->reparam_ready = false;
    // a launch refused for its configuration shows only here: the outputs would be stale (the step counters are
    // restored below on this path too)
    cudaError_t e = cudaGetLastError();
    if (!rc && e != cudaSuccess) rc = h->fail(POLEE_ECUDA, std::string("lsn_draws: ") + cudaGetErrorString(e));
    e = cudaStreamSynchronize(h->stream);
    if (!rc && e != cudaSuccess) rc = h->fail(POLEE_ECUDA, std::string("lsn_draws: ") + cudaGetErrorString(e));
    if (!rc && xs) rc = download_kmajor<float, float>(h, h->x, K, KP, n, xs);
    if (!rc && ys) rc = download_kmajor<double, double>(h, h->ys, K, KP, nm1, ys);
    if (!rc && x_grad) rc = download_kmajor<double, double>(h, d_xg, K, KP, n, x_grad);
    if (!rc && y_grad) rc = download_kmajor<double, float>(h, h->ygrad, K, KP, nm1, y_grad);
    if (!rc && nm1 > 0) {
        if (mu_grad) polee::copy_sync(h->stream, mu_grad, h->grad_out, sizeof(float) * nm1, cudaMemcpyDeviceToHost);
        if (omega_grad) polee::copy_sync(h->stream, omega_grad, h->grad_out + nm1, sizeof(float) * nm1, cudaMemcpyDeviceToHost);
        if (alpha_grad) polee::copy_sync(h->stream, alpha_grad, h->grad_out + 2 * nm1, sizeof(float) * nm1, cudaMemcpyDeviceToHost);
    }
    if (!rc && elbo) {
        *elbo = 0.0;
        if (!h->o.gradonly) polee::copy_sync(h->stream, elbo, h->elbo, sizeof(double), cudaMemcpyDeviceToHost);
    }
    polee::copy_sync(h->stream, h->d_step, &saved, sizeof(saved), cudaMemcpyHostToDevice);
    cudaMemsetAsync(h->d_bad_step, 0, sizeof(int), h->stream);
    cudaStreamSynchronize(h->stream);
    return rc;
}

// ------------------------------------------------------------------ approx-likelihood sampler (SURVEY 8f-1)
// Random.rand!(als::ApproxLikelihoodSampler, xs)  src/approx-sampler.jl:37-44: zs = randn; sinh_asinh_transform!;
// logit_normal_transform! (no clamp); transform!(t, ys, xs).  KP draws per launch at the handle's parameters.
extern "C" int polee_sample(polee_handle *h, int32_t num_samples, uint64_t seed, float *xs) {
    CHECK_H(h);
    if (!h->have_tree) return h->fail(POLEE_EINVAL, "no tree: call polee_set_tree first");
    if (h->o.approx != POLEE_APPROX_LOGIT_SKEW_NORMAL_PTT) return h->fail(POLEE_EINVAL, "polee_sample needs a LogitSkewNormalPTTApprox handle");
    if (num_samples < 0 || (!xs && num_samples > 0)) return h->fail(POLEE_EINVAL, "polee_sample: bad arguments");
    h->n = h->td.n;
    int rc = ensure_work_buffers(h, h->KP);
    if (rc) return rc;
    const int KP = h->KP;
    h->reparam_ready = false;
    for (int done = 0, batch = 0; done < num_samples; done += KP, ++batch) {
        const int take = std::min(KP, num_samples - done);
        if ((rc = launch_elem(h, KP, KP, false, false, true, nullptr, 1, 0, nullptr, batch, seed, 0))) return rc;
        if ((rc = launch_tree_fwd(h, KP, 0, 0, 0))) return rc;
        CK(cudaGetLastError());
        if ((rc = download_kmajor<float, float>(h, h->x, take, KP, h->n, xs + (size_t)done * h->n))) return rc;
    }
    return POLEE_OK;
}

// ------------------------------------------------------------------ measurement helpers
extern "C" int polee_step_stats(polee_handle *h, double *b1, double *b2, double *b3, int32_t *launches) {
    CHECK_H(h);
    if (!h->have_matrix || !h->have_tree) return h->fail(POLEE_EINVAL, "step_stats: set the matrix and the tree first");
    // SURVEY 8(d) / BASELINE.md section 2 formulas with the padded draw count actually streamed
    const double nnz = (double)h->nnz, m = (double)h->m, n = (double)h->n, K = (double)h->KP, N = 2 * n - 1;
    // bytes the likelihood pass really streams per step with the layouts in use (what `roofline.moved` is checked against
    // ncu's dram bytes); b2 = 0 tells the caller there is no second sparse kernel
    const double gm = (double)h->gm, gnnz = (double)h->gnnz;
    double e1 = 0, e2 = 0;
    if (h->ec_tasks > 0)  // task blobs once + (task, column) partials written and read back + x gathers + g
        e1 = (double)h->ec_blob_bytes + (double)h->ec_parts * (K * (ec_math_f32(h) ? 4 : 8) * 2 + 4) + K * n * 4 + K * n * 8;
    if (h->gm > 0 || h->ec_tasks == 0) {
        if (h->fused) {
            e1 += (double)h->ft_blob_bytes + (double)h->ft_parts * (K * 4 * 2 + 4) + K * n * 8;
        } else {
            e1 += gnnz * 8 + (gm + 1) * 4 + K * n * 4 + K * gm * 4;
            e2 = gnnz * 8 + (n + 1) * 4 + K * gm * 4 + K * n * 4;
        }
    }
    if (b1) *b1 = e1;
    if (b2) *b2 = e2;
    (void)nnz; (void)m;
    if (b3) *b3 = (n - 1) * 72 + N * 16 + K * n * 8;
    if (launches) {
        const bool lsn = h->o.approx == POLEE_APPROX_LOGIT_SKEW_NORMAL_PTT;
        const bool vals = lsn && !h->o.gradonly;
        int sparse_launches = 0;
        if (h->gm > 0 || h->ec_tasks == 0)
            sparse_launches += h->fused ? 1 + (h->ft_nunits > 0) + (h->ft_nmulti > 0)
                                        : (h->n_row_tiles > 0) + (h->n_segs > 0) + (h->n_multi > 0);
        if (h->ec_tasks > 0) sparse_launches += 1 + (h->ec_nunits > 0) + (h->ec_nmulti > 0);
        int L = (h->td.top.nbins > 0) + (h->td.bottom.nbins > 0) + 1 /*mid*/ + sparse_launches +
                (h->td.top.nbins > 0) + (h->td.bottom.nbins > 0) + 1 /*update + reparam*/;
        if (vals) L += 2;
        *launches = L;
    }
    return POLEE_OK;
}

// programmatic edges of a captured graph (the PDL launches between consecutive step kernels), -1 without a graph
static int64_t programmatic_edges(cudaGraph_t g) {
    if (!g) return -1;
    size_t n = 0;
    if (cudaGraphGetEdges_v2(g, nullptr, nullptr, nullptr, &n) != cudaSuccess) return -1;
    std::vector<cudaGraphNode_t> from(n), to(n);
    std::vector<cudaGraphEdgeData> data(n);
    if (n > 0 && cudaGraphGetEdges_v2(g, from.data(), to.data(), data.data(), &n) != cudaSuccess) return -1;
    int64_t count = 0;
    for (size_t i = 0; i < n; ++i) count += data[i].type == cudaGraphDependencyTypeProgrammatic;
    return count;
}

// Which layouts hold the matrix: info[0..9] = {rows, entries, classes, tasks, blob bytes, partials} of the
// equivalence-class layout, {rows, entries} of the general layouts, general layout kind (0 none, 1 split, 2 fused),
// padded row slots of the class layout; info[10] = the tree route (TreeRoute) at the work buffers' KP, -1 without a tree
// or work buffers; info[11], info[12] = programmatic edges of the captured one-step and multi-step graphs, -1 while
// not captured.
extern "C" int polee_layout_info(polee_handle *h, int64_t *info, int32_t count) {
    CHECK_H(h);
    if (!info || count < 1) return h->fail(POLEE_EINVAL, "layout_info: bad arguments");
    const int64_t route = h->have_tree && h->work_KP > 0 ? (int64_t)tree_route(h->td, h->work_KP) : -1;
    const int64_t v[13] = {h->ec_rows, h->ec_nnz, h->ec_classes, (int64_t)h->ec_tasks, (int64_t)h->ec_blob_bytes, h->ec_parts,
                           h->gm, h->gnnz, (int64_t)((h->gm > 0 || h->ec_tasks == 0) ? (h->fused ? 2 : 1) : 0), h->ec_slots,
                           route, programmatic_edges(h->graph), programmatic_edges(h->graph_multi)};
    for (int i = 0; i < count && i < 13; ++i) info[i] = v[i];
    return POLEE_OK;
}

extern "C" int polee_time_kernel(polee_handle *h, int32_t which, int32_t reps, float *ms_avg) {
    CHECK_H(h);
    int rc = ready_for_steps(h);
    if (rc) return rc;
    if (reps < 1 || !ms_avg) return h->fail(POLEE_EINVAL, "time_kernel: bad arguments");
    if ((rc = ensure_reparam(h))) return rc;
    const int KP = h->KP, K = h->K;
    const bool lsn = h->o.approx == POLEE_APPROX_LOGIT_SKEW_NORMAL_PTT;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    const float *noise = h->o.noise_mode == POLEE_NOISE_INJECTED ? h->noise : nullptr;
    CK(cudaEventRecord(e0, h->stream));
    for (int r = 0; r < reps && !rc; ++r) {
        if (which == 1) {  // the whole likelihood pass, except on the pure split layout (K1 here, K2 under which == 2)
            rc = (h->ec_tasks > 0 || h->fused) ? launch_likelihood(h, KP, K, false)
                                               : launch_k1(h, h->x, h->w, false, h->lp_partial, KP);
        } else if (which == 2) {
            if (h->ec_tasks == 0 && !h->fused) rc = launch_k2(h, h->w, h->g, KP);  // otherwise: no second sparse kernel
        } else if (which == 3) {
            rc = launch_tree_fwd(h, KP, 1, 1, 0);
            if (!rc) rc = launch_mid(h, KP, 0);
            if (!rc) rc = launch_tree_bwd(h, KP, lsn, true, nullptr);
            if (!rc) rc = launch_elem(h, KP, K, true, false, true, noise, std::max<int64_t>(h->noise_steps, 1), 0, nullptr);
        } else if (which == 4) {  // the class kernel alone (without the second stage that adds its partials)
            if (h->ec_tasks > 0) rc = launch_ec(h, h->x, h->g, false, false, nullptr, nullptr, KP, K, true);
        } else if (which == 5) {  // the all-reduce of g alone (every rank must make the same call)
            rc = launch_allreduce(h, KP, false);
        } else {
            rc = h->fail(POLEE_EINVAL, "time_kernel: which must be 1..5");
        }
    }
    CK(cudaEventRecord(e1, h->stream));
    CK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    CK(cudaGetLastError());
    *ms_avg = ms / reps;
    return rc;
}

// ------------------------------------------------------------------ multi-GPU
extern "C" int polee_partition_rows(int64_t m, int64_t n, const uint32_t *colptr, const uint32_t *rowval, int32_t nparts,
                                    int64_t *row_bounds) {
    if (!colptr || !rowval || !row_bounds || nparts < 1 || m < 1 || n < 1) return POLEE_EINVAL;
    const int64_t nnz = (int64_t)colptr[n] - 1;
    std::vector<int64_t> cnt(m + 1, 0);
    for (int64_t e = 0; e < nnz; ++e) cnt[rowval[e]]++;  // 1-based row -> slot
    for (int64_t i = 0; i < m; ++i) cnt[i + 1] += cnt[i];
    row_bounds[0] = 0;
    for (int p = 1; p < nparts; ++p) {
        const int64_t target = nnz * p / nparts;
        int64_t r = std::lower_bound(cnt.begin(), cnt.end(), target) - cnt.begin();
        row_bounds[p] = std::min<int64_t>(std::max<int64_t>(r, row_bounds[p - 1]), m);
    }
    row_bounds[nparts] = m;
    return POLEE_OK;
}

extern "C" int polee_comm_unique_id(char id[128]) {
#ifdef POLEE_WITH_NCCL
    static_assert(sizeof(ncclUniqueId) <= 128, "ncclUniqueId does not fit");
    ncclUniqueId u;
    if (!nccl_api().ok || nccl_api().GetUniqueId(&u) != ncclSuccess) return POLEE_ENCCL;
    std::memset(id, 0, 128);
    std::memcpy(id, &u, sizeof(u));
    return POLEE_OK;
#else
    (void)id;
    return POLEE_ENCCL;
#endif
}

extern "C" int polee_comm_init(polee_handle *h, int32_t nranks, int32_t rank, const char id[128]) {
    CHECK_H(h);
#ifdef POLEE_WITH_NCCL
    if (nranks < 1 || rank < 0 || rank >= nranks) return h->fail(POLEE_EINVAL, "comm_init: bad rank / nranks");
    if (!nccl_api().ok) return h->fail(POLEE_ENCCL, "libnccl.so.2 could not be loaded");
    drop_graph(h);
    release_work_buffers(h);  // the multi-rank step needs the Float32 all-reduce buffer
    polee::peer_release(h);
    if (h->comm) { nccl_api().CommDestroy(h->comm); h->comm = nullptr; }
    h->nranks = nranks;
    h->rank = rank;
    if (nranks == 1) return POLEE_OK;
    ncclUniqueId u;
    std::memcpy(&u, id, sizeof(u));
    ncclResult_t r = nccl_api().CommInitRank(&h->comm, nranks, u, rank);
    if (r != ncclSuccess) return h->fail(POLEE_ENCCL, std::string("ncclCommInitRank: ") + nccl_api().GetErrorString(r));
    return POLEE_OK;
#else
    (void)nranks; (void)rank; (void)id;
    return h->fail(POLEE_ENCCL, "library built without NCCL");
#endif
}
