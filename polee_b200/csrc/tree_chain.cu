// tree_chain.cu -- depth-independent kernels for caterpillar ("list") trees.
//
// PolyaTreeTransform(X, :sequential) (list_nodes, src/hclust.jl:477-489) is a chain of depth n-1: internal node k has
// a leaf as right child and the next internal node as left child.  It is the tree of OptimizePTTApprox
// (src/likelihood-approximation.jl:160, run once per sample by the bias model, src/rnaseq_sample.jl:343) and of
// `--tree-method sequential`.  A level-synchronous sweep would need n-1 barrier rounds there, so for large chains
// both passes are computed as blocked scans instead (one CTA per draw, 1024 threads, each thread owns a contiguous
// piece of the spine):
//   forward   u_k = prod_{j<k} y_j                                  exclusive product scan
//   backward  G1_k = y_k G1_{k+1} + (1-y_k) g_k ,  G2_k = 1/u_k + y_k G2_{k+1}     reverse scans of affine maps
// The scans re-associate the Float64 products, and the backward recurrences are carried in Float64 instead of being
// rounded to Float32 at every node as the reference does (src/ptt.jl:196-204), so this path matches the reference to
// rounding error (tests state the tolerance), not bit for bit; small chains keep the bit-exact level-synchronous path.
#include "common.cuh"

namespace polee {

namespace {

constexpr int CH_THREADS = 1024;

// exclusive block scan of per-thread values with an associative op; identity supplied
template <typename T, typename Op>
__device__ __forceinline__ T block_exclusive_scan(T v, T identity, T *sm, Op op, bool reverse) {
    const int t = reverse ? CH_THREADS - 1 - (int)threadIdx.x : (int)threadIdx.x;
    sm[t] = v;
    __syncthreads();
    for (int d = 1; d < CH_THREADS; d <<= 1) {
        T a = sm[t];
        T b = t >= d ? sm[t - d] : identity;
        __syncthreads();
        sm[t] = t >= d ? op(b, a) : a;  // op(earlier, later)
        __syncthreads();
    }
    T r = t >= 1 ? sm[t - 1] : identity;
    __syncthreads();
    return r;
}

struct Affine {  // G -> a * G + b
    double a, b;
};

template <int KP>
__global__ void __launch_bounds__(CH_THREADS)
    k3c_chain_fwd(int64_t n, const int32_t *__restrict__ chain_leaf, const double *__restrict__ ys,
                  double *__restrict__ us /* [2n-1][KP] by node id */, float *__restrict__ x, int clamp_x, const float *__restrict__ efflen, double *__restrict__ S_partial, int want_ladj,
                  double *__restrict__ ladj_partial) {
    __shared__ double sm[CH_THREADS];
    const int k = blockIdx.x;  // draw
    const int64_t L = n - 1;
    const int64_t per = (L + CH_THREADS - 1) / CH_THREADS;
    const int64_t s = min(L, (int64_t)threadIdx.x * per), e = min(L, s + per);
    double prod = 1.0;
    for (int64_t j = s; j < e; ++j) prod *= ys[(size_t)j * KP + k];
    double u = block_exclusive_scan<double>(prod, 1.0, sm, [](double a, double b) { return a * b; }, false);
    double sacc = 0.0, lacc = 0.0;
    auto emit_leaf = [&](int leaf, double ul) {
        float xv = (float)ul;
        double d = (double)xv;
        xv = (float)(d > 1e-16 ? d : 1e-16);
        if (clamp_x) {
            d = (double)xv;
            d = fmin(fmax(d, 1e-10), 1.0 - 1e-10);
            xv = (float)d;
        }
        x[(size_t)leaf * KP + k] = xv;
        if (efflen) sacc += (double)__fdiv_rn(xv, efflen[leaf]);
    };
    for (int64_t j = s; j < e; ++j) {
        const double y = ys[(size_t)j * KP + k];
        us[(size_t)(2 * j) * KP + k] = u;
        if (want_ladj) lacc += log(u);
        emit_leaf(chain_leaf[j], (1.0 - y) * u);
        u = y * u;
        if (j == L - 1) emit_leaf(chain_leaf[L], u);
    }
    if (L == 0 && threadIdx.x == 0) emit_leaf(chain_leaf[0], 1.0);
    // block sums (fixed order)
    for (int pass = 0; pass < 2; ++pass) {
        if (pass == 0 && !S_partial) continue;
        if (pass == 1 && !want_ladj) continue;
        sm[threadIdx.x] = pass == 0 ? sacc : lacc;
        __syncthreads();
        for (int span = CH_THREADS / 2; span >= 1; span >>= 1) {
            if ((int)threadIdx.x < span) sm[threadIdx.x] += sm[threadIdx.x + span];
            __syncthreads();
        }
        if (threadIdx.x == 0) (pass == 0 ? S_partial : ladj_partial)[k] = sm[0];
        __syncthreads();
    }
}

template <int KP, bool WITH_LADJ>
__global__ void __launch_bounds__(CH_THREADS)
    k3c_chain_bwd(int64_t n, const int32_t *__restrict__ chain_leaf, const double *__restrict__ ys,
                  const double *__restrict__ us, const double *__restrict__ g, const float *__restrict__ efflen_adj,
                  const double *__restrict__ S, double *__restrict__ ygrad, double *__restrict__ xgrad_out) {
    __shared__ Affine sm1[CH_THREADS];
    __shared__ Affine sm2[CH_THREADS];
    const int k = blockIdx.x;
    const int64_t L = n - 1;
    if (L == 0) return;
    const int64_t per = (L + CH_THREADS - 1) / CH_THREADS;
    const int64_t s = min(L, (int64_t)threadIdx.x * per), e = min(L, s + per);
    const double Sk = efflen_adj ? S[k] : 1.0;
    auto leaf_grad = [&](int leaf) {
        double gv = g[(size_t)leaf * KP + k];
        if (efflen_adj) gv = gv - (double)efflen_adj[leaf] / Sk;  // likelihood.jl:105
        if (xgrad_out) xgrad_out[(size_t)leaf * KP + k] = gv;
        return (double)(float)gv;  // t.gradients[1, leaf] is Float32
    };
    // composite maps of this thread's piece: G_s = A * G_e + B  (processed from e-1 down to s)
    Affine m1{1.0, 0.0}, m2{1.0, 0.0};
    for (int64_t j = e - 1; j >= s; --j) {
        const double y = ys[(size_t)j * KP + k];
        const double gr = leaf_grad(chain_leaf[j]);
        // new map = T_j o old map,  T_j(G) = y G + (1-y) gr   /   y G + 1/u_j
        m1.a = y * m1.a;
        m1.b = y * m1.b + (1.0 - y) * gr;
        if (WITH_LADJ) {
            m2.a = y * m2.a;
            m2.b = y * m2.b + 1.0 / us[(size_t)(2 * j) * KP + k];
        }
    }
    // suffix composition over the threads after this one: apply later pieces first
    auto comp = [](Affine later, Affine earlier) {  // earlier o later : G -> earlier.a * (later.a G + later.b) + earlier.b
        return Affine{earlier.a * later.a, earlier.a * later.b + earlier.b};
    };
    const Affine suf1 = block_exclusive_scan<Affine>(m1, Affine{1.0, 0.0}, sm1, comp, true);
    Affine suf2{1.0, 0.0};
    if (WITH_LADJ) suf2 = block_exclusive_scan<Affine>(m2, Affine{1.0, 0.0}, sm2, comp, true);
    const double GL1 = leaf_grad(chain_leaf[L]);  // the last leaf (left child of the last internal node)
    double G1 = suf1.a * GL1 + suf1.b;            // G of node e (the left child of spine node e-1)
    double G2 = WITH_LADJ ? suf2.b : 0.0;         // G2 of the last leaf is 0
    for (int64_t j = e - 1; j >= s; --j) {
        const double y = ys[(size_t)j * KP + k];
        const double u = us[(size_t)(2 * j) * KP + k];
        const double gr = leaf_grad(chain_leaf[j]);
        // (left_grad + left_ladj_grad) - (right_grad + right_ladj_grad), Float32 in the reference
        const float d = WITH_LADJ ? __fsub_rn(__fadd_rn((float)G1, (float)G2), (float)gr) : __fsub_rn((float)G1, (float)gr);
        const double yg = u * (double)d;
        ygrad[(size_t)j * KP + k] = WITH_LADJ ? (double)(float)yg : yg;
        G1 = y * G1 + (1.0 - y) * gr;
        if (WITH_LADJ) G2 = 1.0 / u + y * G2;
    }
}

}  // namespace

#define CK(expr) POLEE_CUDA_CHECK(h, expr)

int launch_chain_fwd(polee_handle *h, int KP, int clamp_x, const float *eff, double *Sp, int want_ladj, double *ladj_tree) {
    DISPATCH_KP(KP, (k3c_chain_fwd<KPC><<<KP, CH_THREADS, 0, h->stream>>>(h->td.n, h->td.chain_leaf, h->ys, h->us, h->x, clamp_x, eff, Sp, want_ladj, ladj_tree)));
    return POLEE_OK;
}

int launch_chain_bwd(polee_handle *h, int KP, bool with_ladj, const float *adj, double *xgrad_out) {
    if (with_ladj) {
        DISPATCH_KP(KP, (k3c_chain_bwd<KPC, true><<<KP, CH_THREADS, 0, h->stream>>>(h->td.n, h->td.chain_leaf, h->ys, h->us, h->g,
                                                                                 adj, h->S, h->ygrad, xgrad_out)));
    } else {
        DISPATCH_KP(KP, (k3c_chain_bwd<KPC, false><<<KP, CH_THREADS, 0, h->stream>>>(h->td.n, h->td.chain_leaf, h->ys, h->us,
                                                                                  h->g, adj, h->S, h->ygrad, xgrad_out)));
    }
    return POLEE_OK;
}

}  // namespace polee
