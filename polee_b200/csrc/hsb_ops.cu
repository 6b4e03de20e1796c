// hsb_ops.cu -- K4: the three hierarchical-stick-breaking ops of the reference's TensorFlow plugin
// (src/tensorflow_ext/hsb_ops.cpp), batched over B rows, on the same level-synchronous tree engine
// as the fit (tree_host.cu).  The reference shards the batch over TF CPU threads and walks each
// tree serially (hsb_ops.cpp:87-115, 206-245, 338-398); here every (schedule bin, row) is one CTA.
//
// Index tensors are [idx_batch][2n-1] with idx_batch == B (a tree per row, as the reference op
// requires -- src/estimate.jl:357-360) or 1 (shared tree, SURVEY App. C9).  A "plan" holds the
// validated, scheduled tree(s) on the device so that callers with constant index tensors (every
// training step of a TF model) pay for the preparation once.
#include <algorithm>
#include <cstring>
#include <mutex>

#include "common.cuh"

using namespace polee;

struct polee_hsb_plan {
    int device = 0;
    int64_t n = 0, N = 0, ntrees = 0;
    TreeNode *nodes = nullptr;  // [ntrees][N]
    // phase 0 = top bins, 1 = bottom bins (concatenated over trees)
    int32_t *bin_lvl_ptr[2] = {nullptr, nullptr}, *lvl_off[2] = {nullptr, nullptr}, *sch_node[2] = {nullptr, nullptr};
    int32_t *bin_tree[2] = {nullptr, nullptr};
    int nbins[2] = {0, 0};
    int32_t *desc_order = nullptr;  // [ntrees][n-1] internal node ids in descending node order (ladj emulation)
    int32_t *bin_pos = nullptr;     // [ntrees][N] a bottom-bin node's position in its bin's schedule; -1: top node (HSBGrad)
    int max_bin_nodes = 0;          // most nodes of a bottom bin (HSBGrad's shared memory)
    std::string err;
    // scratch of the device-resident entry points (u, v / log u per row; y, y_grad and row partials of the density),
    // grown on demand and kept with the plan so a training step allocates nothing; calls on one plan are serialised by `mu`
    mutable std::mutex mu;
    mutable double *scr[3] = {nullptr, nullptr, nullptr};
    mutable size_t scr_count[3] = {0, 0, 0};
};

namespace {

std::string g_hsb_error;
std::mutex g_hsb_mu;

int hsb_fail(int code, const std::string &msg) {
    std::lock_guard<std::mutex> lk(g_hsb_mu);
    g_hsb_error = msg;
    return code;
}

constexpr int HSB_THREADS = 128;
constexpr int HSB_BIN_NODES = 4096;

struct Sched {
    const int32_t *bin_lvl_ptr, *lvl_off, *sch_node, *bin_tree;
};

__device__ __forceinline__ void bin_row(const Sched &s, int shared_tree, int &tree, int64_t &row) {
    tree = s.bin_tree[blockIdx.x];
    row = shared_tree ? (int64_t)blockIdx.y : (int64_t)tree;
}

// HSBOp::Compute  hsb_ops.cpp:87-109
__global__ void __launch_bounds__(HSB_THREADS)
    k4_hsb_fwd(Sched s, int shared_tree, const TreeNode *__restrict__ nodes_all, int64_t n, int64_t N,
               const float *__restrict__ y_logit, double *__restrict__ us, float *__restrict__ x) {
    int tree;
    int64_t row;
    bin_row(s, shared_tree, tree, row);
    const TreeNode *nodes = nodes_all + (size_t)tree * N;
    double *u = us + (size_t)row * N;
    const int l0 = s.bin_lvl_ptr[blockIdx.x], l1 = s.bin_lvl_ptr[blockIdx.x + 1] - 1;
    for (int l = l0; l < l1; ++l) {
        for (int q = s.lvl_off[l] + threadIdx.x; q < s.lvl_off[l + 1]; q += HSB_THREADS) {
            const int node = s.sch_node[q];
            const TreeNode nd = nodes[node];
            const double ui = node == 0 ? 1.0 : u[node];
            if (nd.leaf >= 0) {
                x[(size_t)row * n + nd.leaf] = (float)ui;
            } else {
                // `1.0 / (1.0 + (double) exp(-y_logit_i[k]))`: exp() resolves to the double overload
                const double y = __ddiv_rn(1.0, __dadd_rn(1.0, exp((double)(-y_logit[(size_t)row * (n - 1) + nd.k]))));
                u[nd.left] = __dmul_rn(y, ui);
                u[nd.right] = __dmul_rn(__dsub_rn(1.0, y), ui);
            }
        }
        __syncthreads();
    }
}

// InvHSBOp::Compute  hsb_ops.cpp:206-239 (bottom-up): y and log(u_j) per internal node
__global__ void __launch_bounds__(HSB_THREADS)
    k4_inv_hsb(Sched s, int shared_tree, const TreeNode *__restrict__ nodes_all, int64_t n, int64_t N,
               const float *__restrict__ x, double *__restrict__ us, double *__restrict__ y, double *__restrict__ logu) {
    int tree;
    int64_t row;
    bin_row(s, shared_tree, tree, row);
    const TreeNode *nodes = nodes_all + (size_t)tree * N;
    double *u = us + (size_t)row * N;
    const int l0 = s.bin_lvl_ptr[blockIdx.x], l1 = s.bin_lvl_ptr[blockIdx.x + 1] - 1;
    for (int l = l1 - 1; l >= l0; --l) {
        for (int q = s.lvl_off[l] + threadIdx.x; q < s.lvl_off[l + 1]; q += HSB_THREADS) {
            const int node = s.sch_node[q];
            const TreeNode nd = nodes[node];
            if (nd.leaf >= 0) {
                u[node] = (double)x[(size_t)row * n + nd.leaf];
            } else {
                const double ul = u[nd.left], ur = u[nd.right];
                const double uj = __dadd_rn(ul, ur);
                u[node] = uj;
                y[(size_t)row * (n - 1) + nd.k] = __ddiv_rn(ul, uj);
                logu[(size_t)row * (n - 1) + nd.k] = log(uj);
            }
        }
        __syncthreads();
    }
}

// `ladj_i[0] -= log(u_data[j])` for j = 2n-2 .. 0 with a FLOAT accumulator (hsb_ops.cpp:211,234): every step rounds,
// acc <- Float32(Float64(acc) - log u), so the result depends on the order and the chain cannot simply be re-associated.
// It can be SPECULATED, though: while acc stays in one binade (and no step is an exact tie) a step moves acc by a whole
// number of its ulps, q_k = rint(-log u_k / ulp), whatever acc is.  One warp per row takes 256 steps at a time: the lanes
// form q_k for 8 steps each, a shuffle scan gives the 256 candidate values, and every lane then checks ITS steps with the
// reference's own rule from the predecessor's candidate.  The steps before the first mismatch are exact by induction; the mismatching
// step (a binade change, a tie, acc == 0, non-finite values) is redone by the scalar rule, and the warp goes on from there.
constexpr int LADJ_S = 8;  // steps per lane and iteration: a warp speculates 32 x 8 = 256 steps at a time
__global__ void __launch_bounds__(128) k4_ladj_chain(int64_t B, int64_t nm1, const double *__restrict__ logu, float *__restrict__ ladj) {
    const int64_t row = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= B) return;
    const double *lu = logu + (size_t)row * nm1;
    float acc = 0.0f;
    int64_t k = nm1 - 1;  // next step (descending, as the reference's loop); lane j, slot i takes step k - (LADJ_S j + i)
    while (k >= 0) {
        const int64_t left = k + 1;
        const int cnt = left < 32 * LADJ_S ? (int)left : 32 * LADJ_S;
        double l[LADJ_S];
#pragma unroll
        for (int i = 0; i < LADJ_S; ++i) {
            const int s = lane * LADJ_S + i;
            l[i] = s < cnt ? lu[k - s] : 0.0;
        }
        int e = 0;
        (void)frexpf(fabsf(acc), &e);  // |acc| = f 2^e, f in [0.5, 1): ulp(acc) = 2^(e - 24)
        const bool fin = acc != 0.0f && isfinite(acc);
        const double ulp = fin ? ldexp(1.0, e - 24) : 0.0, inv_ulp = fin ? ldexp(1.0, 24 - e) : 0.0;
        double q[LADJ_S], tot = 0.0;  // the steps in ulps (a power-of-two scaling: exact), prefix sums inside the lane
#pragma unroll
        for (int i = 0; i < LADJ_S; ++i) {
            tot += (lane * LADJ_S + i < cnt) ? rint(-l[i] * inv_ulp) : 0.0;
            q[i] = tot;
        }
        double P = tot;  // inclusive scan of the lane totals
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double t = __shfl_up_sync(0xffffffffu, P, o);
            if (lane >= o) P += t;
        }
        const double before = P - tot;  // ulps taken by the lanes below
        float cand[LADJ_S];
#pragma unroll
        for (int i = 0; i < LADJ_S; ++i) cand[i] = (float)((double)acc + ulp * (before + q[i]));
        float pred = __shfl_up_sync(0xffffffffu, cand[LADJ_S - 1], 1);
        if (lane == 0) pred = acc;
        int first_bad = LADJ_S;  // first slot of this lane whose step does not verify by the reference's own rule
#pragma unroll
        for (int i = LADJ_S - 1; i >= 0; --i) {
            const float p = i == 0 ? pred : cand[i - 1];
            const bool ok = lane * LADJ_S + i >= cnt || (float)__dsub_rn((double)p, l[i]) == cand[i];
            if (!ok) first_bad = i;
        }
        const unsigned bad = __ballot_sync(0xffffffffu, first_bad < LADJ_S);
        const int bl = bad ? __ffs((int)bad) - 1 : 32;                       // first lane with a mismatch
        const int bi = __shfl_sync(0xffffffffu, first_bad, bl < 32 ? bl : 0);
        const int f = bl < 32 ? bl * LADJ_S + bi : 32 * LADJ_S;              // first step that did not verify
        if (f > 0) {                                                         // steps 0 .. f-1 are exact: take step f-1's value
            const int sl = (f - 1) / LADJ_S, si = (f - 1) % LADJ_S;
            float v = cand[0];
#pragma unroll
            for (int i = 1; i < LADJ_S; ++i) v = si == i ? cand[i] : v;
            acc = __shfl_sync(0xffffffffu, v, sl);
        }
        int done = f < cnt ? f : cnt;
        if (f < cnt) {                                                       // the mismatching step, by the scalar rule
            const int sl = f / LADJ_S, si = f % LADJ_S;
            double v = l[0];
#pragma unroll
            for (int i = 1; i < LADJ_S; ++i) v = si == i ? l[i] : v;
            const double lf = __shfl_sync(0xffffffffu, v, sl);
            acc = (float)__dsub_rn((double)acc, lf);
            ++done;
        }
        k -= done;
    }
    if (lane == 0) ladj[row] = acc;
}

// InvHSBGradOp::Compute  hsb_ops.cpp:338-392 (top-down)
__global__ void __launch_bounds__(HSB_THREADS)
    k4_inv_hsb_grad(Sched s, int shared_tree, const TreeNode *__restrict__ nodes_all, int64_t n, int64_t N,
                    const double *__restrict__ y_grad, const float *__restrict__ ladj_grad,
                    const double *__restrict__ yv, double *__restrict__ us, double *__restrict__ vs,
                    float *__restrict__ backprops) {
    int tree;
    int64_t row;
    bin_row(s, shared_tree, tree, row);
    const TreeNode *nodes = nodes_all + (size_t)tree * N;
    double *u = us + (size_t)row * N, *v = vs + (size_t)row * N;
    const double lg = (double)ladj_grad[row];
    const int l0 = s.bin_lvl_ptr[blockIdx.x], l1 = s.bin_lvl_ptr[blockIdx.x + 1] - 1;
    for (int l = l0; l < l1; ++l) {
        for (int q = s.lvl_off[l] + threadIdx.x; q < s.lvl_off[l + 1]; q += HSB_THREADS) {
            const int node = s.sch_node[q];
            const TreeNode nd = nodes[node];
            const double uj = node == 0 ? 1.0 : u[node];
            const double vj = node == 0 ? 0.0 : v[node];
            if (nd.leaf >= 0) {
                backprops[(size_t)row * n + nd.leaf] = (float)vj;
            } else {
                const double y = yv[(size_t)row * (n - 1) + nd.k];
                const double yg = y_grad[(size_t)row * (n - 1) + nd.k];
                const double u_left = __dmul_rn(uj, y), u_right = __dmul_rn(uj, __dsub_rn(1.0, y));
                const double dladj_du = __ddiv_rn(-1.0, uj), u_j2 = __dmul_rn(uj, uj);
                const double base = __dadd_rn(__dmul_rn(dladj_du, lg), vj);
                v[nd.left] = __dadd_rn(base, __dmul_rn(__ddiv_rn(u_right, u_j2), yg));
                v[nd.right] = __dsub_rn(base, __dmul_rn(__ddiv_rn(u_left, u_j2), yg));
                u[nd.left] = u_left;
                u[nd.right] = u_right;
            }
        }
        __syncthreads();
    }
}

// HSBGrad (the reference's op file leaves it as a TODO, hsb_ops.cpp:123-125; definition: DESIGN.md K4).  With y and u
// exactly as k4_hsb_fwd makes them, G = x_grad at a leaf and G_j = y G_l + (1 - y) G_r at an internal node (so
// G_j = sum over the leaves under j of x_grad u_leaf / u_j), and y_logit_grad_k = y (1 - y) u_j (G_l - G_r).  Every
// value depends only on a node's parent (u) or children (G), so any schedule gives the same bits.
__device__ __forceinline__ double hsb_y(float y_logit) { return __ddiv_rn(1.0, __dadd_rn(1.0, exp((double)(-y_logit)))); }

__device__ __forceinline__ double hsb_grad_node(double y, double uj, double gl, double gr, float *out) {
    *out = (float)__dmul_rn(__dmul_rn(__dmul_rn(y, __dsub_rn(1.0, y)), uj), __dsub_rn(gl, gr));
    return __dadd_rn(__dmul_rn(y, gl), __dmul_rn(__dsub_rn(1.0, y), gr));
}

// top bins (after k4_hsb_fwd wrote u and k4_hsb_grad_bin the G of the bottom-bin roots): bottom-up with u and G in global
// memory ([B][N] plan scratch, indexed by node)
__global__ void __launch_bounds__(HSB_THREADS)
    k4_hsb_grad_top(Sched s, int shared_tree, const TreeNode *__restrict__ nodes_all, int64_t n, int64_t N,
                    const float *__restrict__ y_logit, const double *__restrict__ us, double *__restrict__ gs,
                    float *__restrict__ y_logit_grad) {
    int tree;
    int64_t row;
    bin_row(s, shared_tree, tree, row);
    const TreeNode *nodes = nodes_all + (size_t)tree * N;
    const double *u = us + (size_t)row * N;
    double *g = gs + (size_t)row * N;
    const int l0 = s.bin_lvl_ptr[blockIdx.x], l1 = s.bin_lvl_ptr[blockIdx.x + 1] - 1;
    for (int l = l1 - 1; l >= l0; --l) {
        for (int q = s.lvl_off[l] + threadIdx.x; q < s.lvl_off[l + 1]; q += HSB_THREADS) {
            const int node = s.sch_node[q];
            const TreeNode nd = nodes[node];  // top nodes are internal: their subtrees exceed a bin
            const size_t i = (size_t)row * (n - 1) + nd.k;
            g[node] = hsb_grad_node(hsb_y(y_logit[i]), node == 0 ? 1.0 : u[node], g[nd.left], g[nd.right], &y_logit_grad[i]);
        }
        __syncthreads();
    }
}

// bottom bins: one CTA per (bin, row) runs the bin's forward and then its backward with u and G in shared memory, so no
// per-node value goes through global memory; in: u of the bin's roots (k4_hsb_fwd over the top bins), out: their G.
// Shared memory: u[nb] and, per internal node, y from the forward until the backward replaces it with G.
constexpr int HSB_GRAD_THREADS = 256;
__global__ void __launch_bounds__(HSB_GRAD_THREADS)
    k4_hsb_grad_bin(Sched s, int shared_tree, const TreeNode *__restrict__ nodes_all, const int32_t *__restrict__ bin_pos_all,
                    int64_t n, int64_t N, const float *__restrict__ x_grad, const float *__restrict__ y_logit,
                    const double *__restrict__ us, double *__restrict__ gs, float *__restrict__ y_logit_grad) {
    extern __shared__ double hsb_smem[];
    int tree;
    int64_t row;
    bin_row(s, shared_tree, tree, row);
    const TreeNode *nodes = nodes_all + (size_t)tree * N;
    const int32_t *pos = bin_pos_all + (size_t)tree * N;
    const int l0 = s.bin_lvl_ptr[blockIdx.x], l1 = s.bin_lvl_ptr[blockIdx.x + 1] - 1;
    const int q0 = s.lvl_off[l0];
    double *su = hsb_smem, *sg = hsb_smem + (s.lvl_off[l1] - q0);
    for (int l = l0; l < l1; ++l) {
        for (int q = s.lvl_off[l] + threadIdx.x; q < s.lvl_off[l + 1]; q += HSB_GRAD_THREADS) {
            const int node = s.sch_node[q];
            const TreeNode nd = nodes[node];
            double ui;
            if (l == l0) {
                ui = node == 0 ? 1.0 : us[(size_t)row * N + node];
                su[q - q0] = ui;
            } else {
                ui = su[q - q0];
            }
            if (nd.leaf < 0) {
                const double y = hsb_y(y_logit[(size_t)row * (n - 1) + nd.k]);
                sg[q - q0] = y;
                su[pos[nd.left]] = __dmul_rn(y, ui);
                su[pos[nd.right]] = __dmul_rn(__dsub_rn(1.0, y), ui);
            }
        }
        __syncthreads();
    }
    for (int l = l1 - 1; l >= l0; --l) {
        for (int q = s.lvl_off[l] + threadIdx.x; q < s.lvl_off[l + 1]; q += HSB_GRAD_THREADS) {
            const int node = s.sch_node[q];
            const TreeNode nd = nodes[node];
            double gj;
            if (nd.leaf >= 0) {
                gj = (double)x_grad[(size_t)row * n + nd.leaf];
            } else {
                const size_t i = (size_t)row * (n - 1) + nd.k;
                gj = hsb_grad_node(sg[q - q0], su[q - q0], sg[pos[nd.left]], sg[pos[nd.right]], &y_logit_grad[i]);
            }
            sg[q - q0] = gj;
            if (l == l0) gs[(size_t)row * N + node] = gj;
        }
        __syncthreads();
    }
}

// K5: log q(x) of the LogitSkewNormalPTT approximation (definition: DESIGN.md K5) from the y and log u that k4_inv_hsb
// wrote.  One thread per (internal node k, row); a row's terms are summed in Float64 in a fixed order (warp shuffles,
// then the block's warps, then k5_row_sum over the blocks), so results are run-to-run identical without atomics.
constexpr int K5_THREADS = 256;

// the block's sum, valid in thread 0; fixed association
__device__ __forceinline__ double k5_block_sum(double v) {
    __shared__ double warp_sum[K5_THREADS / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = v;
    __syncthreads();
    v = threadIdx.x < K5_THREADS / 32 ? warp_sum[threadIdx.x] : 0.0;
    if (threadIdx.x < 32) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    }
    return v;
}

// node k of row `row`: term = the LSN log density of y_k - log u_k (u_k = the node's subtree sum), y_grad = d term / d y_k
// (the log u part of the gradient is InvHSBGrad's ladj path).  partial[row][blockIdx.x] = the block's sum of terms.
__global__ void __launch_bounds__(K5_THREADS)
    k5_lsn_log_density(int64_t nm1, int per_row_params, const double *__restrict__ yv, const double *__restrict__ logu,
                       const float *__restrict__ mu, const float *__restrict__ omega, const float *__restrict__ alpha,
                       double *__restrict__ y_grad, double *__restrict__ partial) {
    const int64_t row = blockIdx.y, k = (int64_t)blockIdx.x * K5_THREADS + threadIdx.x;
    double term = 0.0;
    if (k < nm1) {
        const size_t i = (size_t)row * nm1 + k, ip = (per_row_params ? (size_t)row * nm1 : 0) + k;
        const double y = yv[i];
        // the fit's Float32 sigma = expf(omega) (likelihood-approximation.jl:505-507), correctly rounded: CUDA's expf may be
        // 2 ulp off, which moves lp by ~1e-9 relative; glibc's expf agrees with this value in all but ~0.1 % of cases
        const double sigma = (double)(float)exp((double)omega[ip]);
        const double ly = log(y), l1my = log1p(-y);
        const double s = (ly - l1my - (double)mu[ip]) / sigma;
        const double w = asinh(s) - (double)alpha[ip];
        const double z0 = sinh(w), r = hypot(1.0, s), aw = fabs(w);
        if (y > 0.0 && y < 1.0) {
            const double log_cosh_w = aw + log1p(exp(-2.0 * aw)) - 0.69314718055994530942;
            term = -0.5 * z0 * z0 - 0.91893853320467274178 + log_cosh_w - 0.5 * log1p(s * s) - log(sigma) - ly - l1my - logu[i];
        } else {
            term = -INFINITY;  // x is on the boundary of the support (a zero leaf under a non-zero subtree)
        }
        const double g_s = (tanh(w) - z0 * cosh(w)) / r - s / (r * r);
        y_grad[i] = g_s / (sigma * y * (1.0 - y)) + 1.0 / (1.0 - y) - 1.0 / y;
    }
    term = k5_block_sum(term);
    if (threadIdx.x == 0) partial[(size_t)row * gridDim.x + blockIdx.x] = term;
}

// lp[row] = the sum of the row's block partials; also the ladj_grad = 1 that k4_inv_hsb_grad reads for the gradient
__global__ void __launch_bounds__(K5_THREADS)
    k5_row_sum(int nblk, const double *__restrict__ partial, double *__restrict__ lp, float *__restrict__ ladj_grad) {
    const int64_t row = blockIdx.x;
    double v = 0.0;
    for (int b = threadIdx.x; b < nblk; b += K5_THREADS) v += partial[(size_t)row * nblk + b];
    v = k5_block_sum(v);
    if (threadIdx.x == 0) {
        lp[row] = v;
        ladj_grad[row] = 1.0f;
    }
}

template <typename T>
cudaError_t up_vec(const std::vector<T> &v, T **d) {
    *d = nullptr;
    cudaError_t e = polee::dmalloc((void **)d, std::max<size_t>(v.size(), 1) * sizeof(T));
    if (e == cudaSuccess && !v.empty()) e = cudaMemcpy(*d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
    return e;
}

struct DevBuf {
    std::vector<void *> ptrs;
    ~DevBuf() {
        for (void *p : ptrs) polee::dfree(p);
    }
    template <typename T>
    cudaError_t alloc(T **p, size_t count) {
        cudaError_t e = polee::dmalloc((void **)p, std::max<size_t>(count, 1) * sizeof(T));
        if (e == cudaSuccess) ptrs.push_back(*p);
        return e;
    }
    template <typename T>
    cudaError_t upload(T **p, const T *host, size_t count) {
        cudaError_t e = alloc(p, count);
        if (e == cudaSuccess && count) e = cudaMemcpy(*p, host, count * sizeof(T), cudaMemcpyHostToDevice);
        return e;
    }
};

}  // namespace

extern "C" {

typedef struct polee_hsb_plan polee_hsb_plan;

const char *polee_hsb_last_error(void) {
    std::lock_guard<std::mutex> lk(g_hsb_mu);
    return g_hsb_error.c_str();
}

int polee_hsb_plan_destroy(polee_hsb_plan *p) {
    if (!p) return POLEE_OK;
    cudaSetDevice(p->device);
    polee::dfree(p->nodes);
    polee::dfree(p->desc_order);
    polee::dfree(p->bin_pos);
    polee::dfree(p->scr[0]); polee::dfree(p->scr[1]); polee::dfree(p->scr[2]);
    for (int s = 0; s < 2; ++s) {
        polee::dfree(p->bin_lvl_ptr[s]); polee::dfree(p->lvl_off[s]); polee::dfree(p->sch_node[s]); polee::dfree(p->bin_tree[s]);
    }
    delete p;
    return POLEE_OK;
}

int polee_hsb_plan_create(polee_hsb_plan **out, int32_t device, int64_t n, int64_t idx_batch, const int32_t *left,
                          const int32_t *right, const int32_t *leaf) {
    if (!out || !left || !right || !leaf || n < 1 || idx_batch < 1) return hsb_fail(POLEE_EINVAL, "hsb plan: bad arguments");
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0)
        return hsb_fail(POLEE_ECUDA, "no CUDA device (libpolee_b200 has no CPU fallback)");
    if (device < 0 || device >= count || cudaSetDevice(device) != cudaSuccess) return hsb_fail(POLEE_ECUDA, "cudaSetDevice failed");
    const int64_t N = 2 * n - 1;
    std::vector<TreeNode> nodes((size_t)idx_batch * N);
    std::vector<int32_t> blp[2] = {{0}, {0}}, lo[2], sn[2], bt[2];
    std::vector<int32_t> bin_pos((size_t)idx_batch * N, -1);
    int max_bin_nodes = 0;
    for (int64_t t = 0; t < idx_batch; ++t) {
        TreeHost th;
        std::string e = th.build_from_lrf(n, left + t * N, right + t * N, leaf + t * N, HSB_BIN_NODES);
        if (!e.empty()) return hsb_fail(POLEE_EBADTREE, "tree " + std::to_string(t) + ": " + e);
        std::copy(th.nodes.begin(), th.nodes.end(), nodes.begin() + (size_t)t * N);
        for (int b = 0; b < th.bottom.nbins(); ++b) {
            const int32_t q0 = th.bottom.lvl_off[th.bottom.bin_lvl_ptr[b]], q1 = th.bottom.lvl_off[th.bottom.bin_lvl_ptr[b + 1] - 1];
            for (int32_t q = q0; q < q1; ++q) bin_pos[(size_t)t * N + th.bottom.sch_node[q]] = q - q0;
            max_bin_nodes = std::max(max_bin_nodes, (int)(q1 - q0));
        }
        const TreeSchedHost *hs[2] = {&th.top, &th.bottom};
        for (int s = 0; s < 2; ++s) {
            const int32_t node_base = (int32_t)sn[s].size(), lvl_base = (int32_t)lo[s].size();
            sn[s].insert(sn[s].end(), hs[s]->sch_node.begin(), hs[s]->sch_node.end());
            for (int32_t v : hs[s]->lvl_off) lo[s].push_back(v + node_base);
            for (int b = 0; b < hs[s]->nbins(); ++b) {
                blp[s].push_back(hs[s]->bin_lvl_ptr[b + 1] + lvl_base);
                bt[s].push_back((int32_t)t);
            }
        }
    }
    polee_hsb_plan *p = new polee_hsb_plan();
    p->device = device; p->n = n; p->N = N; p->ntrees = idx_batch; p->max_bin_nodes = max_bin_nodes;
    cudaError_t e = up_vec(nodes, &p->nodes);
    if (e == cudaSuccess) e = up_vec(bin_pos, &p->bin_pos);
    for (int s = 0; s < 2 && e == cudaSuccess; ++s) {
        p->nbins[s] = (int)bt[s].size();
        e = up_vec(blp[s], &p->bin_lvl_ptr[s]);
        if (e == cudaSuccess) e = up_vec(lo[s], &p->lvl_off[s]);
        if (e == cudaSuccess) e = up_vec(sn[s], &p->sch_node[s]);
        if (e == cudaSuccess) e = up_vec(bt[s], &p->bin_tree[s]);
    }
    if (e != cudaSuccess) {
        polee_hsb_plan_destroy(p);
        return hsb_fail(POLEE_ECUDA, std::string("hsb plan upload: ") + cudaGetErrorString(e));
    }
    *out = p;
    return POLEE_OK;
}

#define HCK(expr)                                                                                        \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess) return hsb_fail(POLEE_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
    } while (0)

static int check_plan(const polee_hsb_plan *p, int64_t B) {
    if (!p || B < 1) return hsb_fail(POLEE_EINVAL, "hsb: bad plan / batch");
    if (p->ntrees != 1 && p->ntrees != B) return hsb_fail(POLEE_EINVAL, "hsb: idx_batch must be 1 or B");
    if (cudaSetDevice(p->device) != cudaSuccess) return hsb_fail(POLEE_ECUDA, "cudaSetDevice failed");
    return POLEE_OK;
}

static Sched sched_of(const polee_hsb_plan *p, int s) {
    return Sched{p->bin_lvl_ptr[s], p->lvl_off[s], p->sch_node[s], p->bin_tree[s]};
}

static int plan_scratch(const polee_hsb_plan *p, int which, size_t count, double **out) {
    if (p->scr_count[which] < count) {
        HCK(cudaDeviceSynchronize());  // an earlier call on another stream may still use the old block
        polee::dfree(p->scr[which]);
        p->scr[which] = nullptr;
        p->scr_count[which] = 0;
        HCK(polee::dmalloc((void **)&p->scr[which], count * sizeof(double)));
        p->scr_count[which] = count;
    }
    *out = p->scr[which];
    return POLEE_OK;
}

// ---- device-resident forms: tensors already in device memory, work enqueued on the caller's stream (what a TF
// DEVICE_GPU kernel has: hsb_ops.cpp:120, 249, 402 register the ops for DEVICE_CPU only)
int polee_hsb_device(const polee_hsb_plan *p, int64_t B, const float *d_y_logit, float *d_x, void *stream) {
    int rc = check_plan(p, B);
    if (rc) return rc;
    if (!d_y_logit || !d_x) return hsb_fail(POLEE_EINVAL, "hsb: null pointer");
    std::lock_guard<std::mutex> lk(p->mu);
    cudaStream_t st = (cudaStream_t)stream;
    const int shared = p->ntrees == 1;
    double *d_us;
    if ((rc = plan_scratch(p, 0, (size_t)B * p->N, &d_us))) return rc;
    for (int s = 0; s < 2; ++s)
        if (p->nbins[s] > 0) {
            dim3 grid(p->nbins[s], shared ? (unsigned)B : 1u);
            k4_hsb_fwd<<<grid, HSB_THREADS, 0, st>>>(sched_of(p, s), shared, p->nodes, p->n, p->N, d_y_logit, d_us, d_x);
        }
    HCK(cudaGetLastError());
    return POLEE_OK;
}

int polee_inv_hsb_device(const polee_hsb_plan *p, int64_t B, const float *d_x, double *d_y, float *d_ladj, void *stream) {
    int rc = check_plan(p, B);
    if (rc) return rc;
    if (!d_x || !d_y || !d_ladj) return hsb_fail(POLEE_EINVAL, "inv_hsb: null pointer");
    std::lock_guard<std::mutex> lk(p->mu);
    cudaStream_t st = (cudaStream_t)stream;
    const int shared = p->ntrees == 1;
    const int64_t nm1 = p->n - 1;
    double *d_us, *d_logu;
    if ((rc = plan_scratch(p, 0, (size_t)B * p->N, &d_us))) return rc;
    if ((rc = plan_scratch(p, 1, (size_t)B * p->N, &d_logu))) return rc;
    for (int s = 1; s >= 0; --s)  // bottom bins first, then the top
        if (p->nbins[s] > 0) {
            dim3 grid(p->nbins[s], shared ? (unsigned)B : 1u);
            k4_inv_hsb<<<grid, HSB_THREADS, 0, st>>>(sched_of(p, s), shared, p->nodes, p->n, p->N, d_x, d_us, d_y, d_logu);
        }
    k4_ladj_chain<<<(unsigned)((B + 3) / 4), 128, 0, st>>>(B, nm1, d_logu, d_ladj);  // one warp per row
    HCK(cudaGetLastError());
    return POLEE_OK;
}

int polee_inv_hsb_grad_device(const polee_hsb_plan *p, int64_t B, const double *d_y_grad, const float *d_ladj_grad,
                              const double *d_y, float *d_backprops, void *stream) {
    int rc = check_plan(p, B);
    if (rc) return rc;
    if (!d_y_grad || !d_ladj_grad || !d_y || !d_backprops) return hsb_fail(POLEE_EINVAL, "inv_hsb_grad: null pointer");
    std::lock_guard<std::mutex> lk(p->mu);
    cudaStream_t st = (cudaStream_t)stream;
    const int shared = p->ntrees == 1;
    double *d_us, *d_vs;
    if ((rc = plan_scratch(p, 0, (size_t)B * p->N, &d_us))) return rc;
    if ((rc = plan_scratch(p, 1, (size_t)B * p->N, &d_vs))) return rc;
    for (int s = 0; s < 2; ++s)
        if (p->nbins[s] > 0) {
            dim3 grid(p->nbins[s], shared ? (unsigned)B : 1u);
            k4_inv_hsb_grad<<<grid, HSB_THREADS, 0, st>>>(sched_of(p, s), shared, p->nodes, p->n, p->N, d_y_grad, d_ladj_grad, d_y,
                                                          d_us, d_vs, d_backprops);
        }
    HCK(cudaGetLastError());
    return POLEE_OK;
}

// HSBGrad: k4_hsb_fwd over the top bins (u of the top nodes and of the bottom-bin roots) -> k4_hsb_grad_bin over the
// bottom bins (forward and backward in shared memory; G of the bin roots) -> k4_hsb_grad_top over the top bins.
int polee_hsb_grad_device(const polee_hsb_plan *p, int64_t B, const float *d_x_grad, const float *d_y_logit,
                          float *d_y_logit_grad, void *stream) {
    int rc = check_plan(p, B);
    if (rc) return rc;
    if (!d_x_grad || !d_y_logit || !d_y_logit_grad) return hsb_fail(POLEE_EINVAL, "hsb_grad: null pointer");
    if (p->n == 1) return POLEE_OK;  // no internal node: the output is empty
    std::lock_guard<std::mutex> lk(p->mu);
    cudaStream_t st = (cudaStream_t)stream;
    const int shared = p->ntrees == 1;
    const unsigned rows = shared ? (unsigned)B : 1u;
    double *d_us, *d_gs;
    if ((rc = plan_scratch(p, 0, (size_t)B * p->N, &d_us))) return rc;
    if ((rc = plan_scratch(p, 1, (size_t)B * p->N, &d_gs))) return rc;
    if (p->nbins[0] > 0)  // top bins hold internal nodes only: x is not written
        k4_hsb_fwd<<<dim3(p->nbins[0], rows), HSB_THREADS, 0, st>>>(sched_of(p, 0), shared, p->nodes, p->n, p->N, d_y_logit, d_us,
                                                                   nullptr);
    HCK(allow_max_smem(k4_hsb_grad_bin));
    k4_hsb_grad_bin<<<dim3(p->nbins[1], rows), HSB_GRAD_THREADS, (size_t)p->max_bin_nodes * 2 * sizeof(double), st>>>(
        sched_of(p, 1), shared, p->nodes, p->bin_pos, p->n, p->N, d_x_grad, d_y_logit, d_us, d_gs, d_y_logit_grad);
    if (p->nbins[0] > 0)
        k4_hsb_grad_top<<<dim3(p->nbins[0], rows), HSB_THREADS, 0, st>>>(sched_of(p, 0), shared, p->nodes, p->n, p->N, d_y_logit,
                                                                        d_us, d_gs, d_y_logit_grad);
    HCK(cudaGetLastError());
    return POLEE_OK;
}

// k4_inv_hsb -> k5_lsn_log_density -> k5_row_sum [-> k4_inv_hsb_grad with ladj_grad = 1].  The Float32 ladj replay
// (k4_ladj_chain) is not needed: the density sums -log u_j in Float64 with the other terms.
int polee_approx_log_prob_device(const polee_hsb_plan *p, int64_t B, int64_t param_batch, const float *d_x,
                                 const float *d_mu, const float *d_omega, const float *d_alpha, double *d_lp,
                                 float *d_x_grad, void *stream) {
    int rc = check_plan(p, B);
    if (rc) return rc;
    if (param_batch != 1 && param_batch != B) return hsb_fail(POLEE_EINVAL, "approx_log_prob: param_batch must be 1 or B");
    if (!d_x || !d_mu || !d_omega || !d_alpha || !d_lp) return hsb_fail(POLEE_EINVAL, "approx_log_prob: null pointer");
    std::lock_guard<std::mutex> lk(p->mu);
    cudaStream_t st = (cudaStream_t)stream;
    const int shared = p->ntrees == 1;
    const int64_t nm1 = p->n - 1;
    const int nblk = (int)((nm1 + K5_THREADS - 1) / K5_THREADS);
    double *d_us, *d_logu, *d_k5;
    if ((rc = plan_scratch(p, 0, (size_t)B * p->N, &d_us))) return rc;
    if ((rc = plan_scratch(p, 1, (size_t)B * p->N, &d_logu))) return rc;  // log u, then v of the gradient
    if ((rc = plan_scratch(p, 2, (size_t)B * (2 * nm1 + nblk + 1), &d_k5))) return rc;
    double *d_y = d_k5, *d_y_grad = d_y + (size_t)B * nm1, *d_part = d_y_grad + (size_t)B * nm1;
    float *d_ladj_grad = (float *)(d_part + (size_t)B * nblk);
    for (int s = 1; s >= 0; --s)
        if (p->nbins[s] > 0) {
            dim3 grid(p->nbins[s], shared ? (unsigned)B : 1u);
            k4_inv_hsb<<<grid, HSB_THREADS, 0, st>>>(sched_of(p, s), shared, p->nodes, p->n, p->N, d_x, d_us, d_y, d_logu);
        }
    if (nblk > 0)
        k5_lsn_log_density<<<dim3((unsigned)nblk, (unsigned)B), K5_THREADS, 0, st>>>(nm1, param_batch != 1, d_y, d_logu, d_mu,
                                                                                     d_omega, d_alpha, d_y_grad, d_part);
    k5_row_sum<<<(unsigned)B, K5_THREADS, 0, st>>>(nblk, d_part, d_lp, d_ladj_grad);
    if (d_x_grad)
        for (int s = 0; s < 2; ++s)
            if (p->nbins[s] > 0) {
                dim3 grid(p->nbins[s], shared ? (unsigned)B : 1u);
                k4_inv_hsb_grad<<<grid, HSB_THREADS, 0, st>>>(sched_of(p, s), shared, p->nodes, p->n, p->N, d_y_grad, d_ladj_grad,
                                                              d_y, d_us, d_logu, d_x_grad);
            }
    HCK(cudaGetLastError());
    return POLEE_OK;
}

// ---- host-tensor forms (the DEVICE_CPU registration of the shim): upload, the device form on the legacy stream, download
int polee_hsb_with_plan(const polee_hsb_plan *p, int64_t B, const float *y_logit, float *x) {
    int rc = check_plan(p, B);
    if (rc) return rc;
    DevBuf db;
    float *d_yl, *d_x;
    HCK(db.upload(&d_yl, y_logit, (size_t)B * (p->n - 1)));
    HCK(db.alloc(&d_x, (size_t)B * p->n));
    if ((rc = polee_hsb_device(p, B, d_yl, d_x, nullptr))) return rc;
    HCK(cudaMemcpy(x, d_x, sizeof(float) * (size_t)B * p->n, cudaMemcpyDeviceToHost));
    return POLEE_OK;
}

int polee_inv_hsb_with_plan(const polee_hsb_plan *p, int64_t B, const float *x, double *y, float *ladj) {
    int rc = check_plan(p, B);
    if (rc) return rc;
    const int64_t nm1 = p->n - 1;
    DevBuf db;
    float *d_x, *d_ladj;
    double *d_y;
    HCK(db.upload(&d_x, x, (size_t)B * p->n));
    HCK(db.alloc(&d_y, (size_t)B * nm1));
    HCK(db.alloc(&d_ladj, (size_t)B));
    if ((rc = polee_inv_hsb_device(p, B, d_x, d_y, d_ladj, nullptr))) return rc;
    if (nm1 > 0) HCK(cudaMemcpy(y, d_y, sizeof(double) * (size_t)B * nm1, cudaMemcpyDeviceToHost));
    HCK(cudaMemcpy(ladj, d_ladj, sizeof(float) * (size_t)B, cudaMemcpyDeviceToHost));
    return POLEE_OK;
}

int polee_inv_hsb_grad_with_plan(const polee_hsb_plan *p, int64_t B, const double *y_grad, const float *ladj_grad,
                                 const double *y, float *backprops) {
    int rc = check_plan(p, B);
    if (rc) return rc;
    const int64_t nm1 = p->n - 1;
    DevBuf db;
    double *d_yg, *d_y;
    float *d_lg, *d_bp;
    HCK(db.upload(&d_yg, y_grad, (size_t)B * nm1));
    HCK(db.upload(&d_y, y, (size_t)B * nm1));
    HCK(db.upload(&d_lg, ladj_grad, (size_t)B));
    HCK(db.alloc(&d_bp, (size_t)B * p->n));
    if ((rc = polee_inv_hsb_grad_device(p, B, d_yg, d_lg, d_y, d_bp, nullptr))) return rc;
    HCK(cudaMemcpy(backprops, d_bp, sizeof(float) * (size_t)B * p->n, cudaMemcpyDeviceToHost));
    return POLEE_OK;
}

int polee_hsb_grad_with_plan(const polee_hsb_plan *p, int64_t B, const float *x_grad, const float *y_logit, float *y_logit_grad) {
    int rc = check_plan(p, B);
    if (rc) return rc;
    if (!x_grad || !y_logit || !y_logit_grad) return hsb_fail(POLEE_EINVAL, "hsb_grad: null pointer");
    const int64_t nm1 = p->n - 1;
    if (nm1 == 0) return POLEE_OK;
    DevBuf db;
    float *d_xg, *d_yl, *d_ylg;
    HCK(db.upload(&d_xg, x_grad, (size_t)B * p->n));
    HCK(db.upload(&d_yl, y_logit, (size_t)B * nm1));
    HCK(db.alloc(&d_ylg, (size_t)B * nm1));
    if ((rc = polee_hsb_grad_device(p, B, d_xg, d_yl, d_ylg, nullptr))) return rc;
    HCK(cudaMemcpy(y_logit_grad, d_ylg, sizeof(float) * (size_t)B * nm1, cudaMemcpyDeviceToHost));
    return POLEE_OK;
}

int polee_approx_log_prob_with_plan(const polee_hsb_plan *p, int64_t B, int64_t param_batch, const float *x,
                                    const float *mu, const float *omega, const float *alpha, double *lp, float *x_grad) {
    int rc = check_plan(p, B);
    if (rc) return rc;
    if (param_batch != 1 && param_batch != B) return hsb_fail(POLEE_EINVAL, "approx_log_prob: param_batch must be 1 or B");
    if (!x || !mu || !omega || !alpha || !lp) return hsb_fail(POLEE_EINVAL, "approx_log_prob: null pointer");
    const size_t np = (size_t)param_batch * (p->n - 1);
    DevBuf db;
    float *d_x, *d_mu, *d_om, *d_al, *d_xg = nullptr;
    double *d_lp;
    HCK(db.upload(&d_x, x, (size_t)B * p->n));
    HCK(db.upload(&d_mu, mu, np));
    HCK(db.upload(&d_om, omega, np));
    HCK(db.upload(&d_al, alpha, np));
    HCK(db.alloc(&d_lp, (size_t)B));
    if (x_grad) HCK(db.alloc(&d_xg, (size_t)B * p->n));
    if ((rc = polee_approx_log_prob_device(p, B, param_batch, d_x, d_mu, d_om, d_al, d_lp, d_xg, nullptr))) return rc;
    HCK(cudaMemcpy(lp, d_lp, sizeof(double) * (size_t)B, cudaMemcpyDeviceToHost));
    if (x_grad) HCK(cudaMemcpy(x_grad, d_xg, sizeof(float) * (size_t)B * p->n, cudaMemcpyDeviceToHost));
    return POLEE_OK;
}

// ---- plan-less forms declared in include/polee_b200.h
int polee_hsb(int32_t device, int64_t B, int64_t n, const float *y_logit, const int32_t *left, const int32_t *right,
              const int32_t *leaf, int64_t idx_batch, float *x) {
    if (idx_batch != 1 && idx_batch != B) return hsb_fail(POLEE_EINVAL, "hsb: idx_batch must be 1 or B");
    polee_hsb_plan *p = nullptr;
    int rc = polee_hsb_plan_create(&p, device, n, idx_batch, left, right, leaf);
    if (!rc) rc = polee_hsb_with_plan(p, B, y_logit, x);
    polee_hsb_plan_destroy(p);
    return rc;
}

int polee_hsb_grad(int32_t device, int64_t B, int64_t n, const float *x_grad, const float *y_logit, const int32_t *left,
                   const int32_t *right, const int32_t *leaf, int64_t idx_batch, float *y_logit_grad) {
    if (idx_batch != 1 && idx_batch != B) return hsb_fail(POLEE_EINVAL, "hsb_grad: idx_batch must be 1 or B");
    polee_hsb_plan *p = nullptr;
    int rc = polee_hsb_plan_create(&p, device, n, idx_batch, left, right, leaf);
    if (!rc) rc = polee_hsb_grad_with_plan(p, B, x_grad, y_logit, y_logit_grad);
    polee_hsb_plan_destroy(p);
    return rc;
}

int polee_inv_hsb(int32_t device, int64_t B, int64_t n, const float *x, const int32_t *left, const int32_t *right,
                  const int32_t *leaf, int64_t idx_batch, double *y, float *ladj) {
    if (idx_batch != 1 && idx_batch != B) return hsb_fail(POLEE_EINVAL, "inv_hsb: idx_batch must be 1 or B");
    polee_hsb_plan *p = nullptr;
    int rc = polee_hsb_plan_create(&p, device, n, idx_batch, left, right, leaf);
    if (!rc) rc = polee_inv_hsb_with_plan(p, B, x, y, ladj);
    polee_hsb_plan_destroy(p);
    return rc;
}

int polee_inv_hsb_grad(int32_t device, int64_t B, int64_t n, const double *y_grad, const float *ladj_grad,
                       const double *y, const int32_t *left, const int32_t *right, const int32_t *leaf,
                       int64_t idx_batch, float *backprops) {
    if (idx_batch != 1 && idx_batch != B) return hsb_fail(POLEE_EINVAL, "inv_hsb_grad: idx_batch must be 1 or B");
    polee_hsb_plan *p = nullptr;
    int rc = polee_hsb_plan_create(&p, device, n, idx_batch, left, right, leaf);
    if (!rc) rc = polee_inv_hsb_grad_with_plan(p, B, y_grad, ladj_grad, y, backprops);
    polee_hsb_plan_destroy(p);
    return rc;
}

// make_inverse_ptt_params  src/ptt.jl:293-309 (pure integer host helper)
int polee_make_inverse_ptt_params(int64_t num_nodes, const int32_t *node_parent_idxs, const int32_t *node_js,
                                  int32_t *left_index, int32_t *right_index, int32_t *leaf_index) {
    if (!node_parent_idxs || !node_js || !left_index || !right_index || !leaf_index || num_nodes < 1) return POLEE_EINVAL;
    for (int64_t i = 0; i < num_nodes; ++i) left_index[i] = right_index[i] = -1;
    for (int64_t i = 1; i < num_nodes; ++i) {
        const int32_t p = node_parent_idxs[i];
        if (p < 1 || p > num_nodes) return POLEE_EBADTREE;
        if (right_index[p - 1] == -1)
            right_index[p - 1] = (int32_t)i;
        else
            left_index[p - 1] = (int32_t)i;
    }
    for (int64_t i = 0; i < num_nodes; ++i) leaf_index[i] = node_js[i] - 1;
    return POLEE_OK;
}

}  // extern "C"
