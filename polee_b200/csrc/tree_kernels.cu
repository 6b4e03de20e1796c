// tree_kernels.cu -- K3: reparameterisation, Polya-tree (hierarchical stick breaking) transform,
// its backward pass with the log-Jacobian term, and the ADAM update, for KP draws at once.
//
//   k3_reparam_fwd   zs0 -> zs -> ys          sinh_asinh_transform! + logit_normal_transform! + clamp!
//                                             (src/sinh_arcsinh.jl:10-23, src/logitnormal.jl:8-20,
//                                              src/likelihood-approximation.jl:517-523)
//   k3_tree_fwd      ys -> us -> xs           transform! + clamp!   (src/ptt.jl:125-160, l-a.jl:525-526)
//   k3_mid           S_k = sum_j x_jk/efflen_j, step bookkeeping    (src/likelihood.jl:96-100)
//   k3_tree_bwd      x_grad -> y_grad         effective_length_jacobian_adjustment! (likelihood.jl:104-106)
//                                             + transform_gradients! (src/ptt.jl:167-209 / :217-251)
//   k3_update        y_grad -> mu/omega/alpha grads (logitnormal.jl:38-55, sinh_arcsinh.jl:29-38,
//                    l-a.jl:547-558) + adam_update_mv!/adam_update_params! (l-a.jl:116-146)
//
// The tree passes are level-synchronous inside one CTA per schedule bin (tree_host.cu): a node's
// value depends only on its parent (forward) or its two children (backward), so the results are
// bit-identical to the reference's serial sweeps -- the same IEEE operations in the same association,
// with explicit _rn intrinsics so that nothing is contracted into an FMA the reference does not have.
#include <math_constants.h>

#include <climits>

#include "common.cuh"
#include "device_utils.cuh"

namespace polee {

namespace {

constexpr int TREE_THREADS = 256;
constexpr int ELEM_THREADS = 128;  // k3_elem: one thread per internal node; small CTAs keep the tail wave short
constexpr int TOP_THREADS = 1024;

// ---------------------------------------------------------------- noise ("polee-philox-v1")
__device__ __forceinline__ void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
        c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
}
// one standard normal for (node i, draw d, step s): counter (i, d, s, 0), key = seed, Box-Muller cos branch
__device__ __forceinline__ float philox_normal(uint64_t seed, uint32_t i, uint32_t d, uint32_t s, int fast) {
    uint32_t c[4] = {i, d, s, 0u};
    philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    float u1 = ((float)(c[0] >> 8) + 0.5f) * (1.0f / 16777216.0f);
    float u2 = ((float)(c[1] >> 8) + 0.5f) * (1.0f / 16777216.0f);
    if (fast)  // hardware log2 / cos: ~1e-6 absolute on a noise sample, no parity contract (tests inject noise)
        return sqrtf(-2.0f * __logf(u1)) * __cosf(6.28318530717958647692f * u2);
    float r = sqrtf(-2.0f * logf(u1));
    return r * cosf(6.28318530717958647692f * u2);
}

// deterministic block reduction of one double per thread laid out [slot][KP] (k fastest)
template <int KP, int THREADS>
__device__ __forceinline__ void block_reduce_k(double v, double *sm, double *out /* [KP] */) {
    sm[threadIdx.x] = v;
    __syncthreads();
    for (int span = THREADS / KP / 2; span >= 1; span >>= 1) {
        if ((int)threadIdx.x < span * KP) sm[threadIdx.x] += sm[threadIdx.x + span * KP];
        __syncthreads();
    }
    if (threadIdx.x < KP) out[threadIdx.x] = sm[threadIdx.x];
    __syncthreads();
}

// ---------------------------------------------------------------- tree forward
template <int KP, int THREADS>
__global__ void __launch_bounds__(THREADS)
    k3_tree_fwd(const int32_t *__restrict__ bin_lvl_ptr, const int32_t *__restrict__ lvl_off,
                const int32_t *__restrict__ sch_node, const TreeNode *__restrict__ nodes,
                const double *__restrict__ ys, double *__restrict__ us, float *__restrict__ x, int clamp_x,
                const float *__restrict__ efflen, double *__restrict__ S_partial, int part_base, int want_ladj,
                double *__restrict__ ladj_partial) {
    __shared__ double sm[THREADS];
    const int k = threadIdx.x % KP, slot = threadIdx.x / KP;
    constexpr int NPP = THREADS / KP;
    const int l0 = bin_lvl_ptr[blockIdx.x], l1 = bin_lvl_ptr[blockIdx.x + 1] - 1;  // levels l0..l1-1
    double sacc = 0.0, lacc = 0.0;
    for (int l = l0; l < l1; ++l) {
        const int lo = lvl_off[l], hi = lvl_off[l + 1];
        for (int q = lo + slot; q < hi; q += NPP) {
            const int node = sch_node[q];
            const TreeNode nd = nodes[node];
            const double ui = node == 0 ? 1.0 : us[(size_t)node * KP + k];
            if (nd.leaf >= 0) {
                float xv = (float)ui;
                double d = (double)xv;
                xv = (float)(d > 1e-16 ? d : 1e-16);  // ptt.jl:136-137
                if (clamp_x) {                         // clamp!(xs, 1e-10, 1 - 1e-10) on a Float32 vector
                    d = (double)xv;
                    d = fmin(fmax(d, 1e-10), 1.0 - 1e-10);
                    xv = (float)d;
                }
                x[(size_t)nd.leaf * KP + k] = xv;
                if (efflen) sacc = __dadd_rn(sacc, (double)__fdiv_rn(xv, efflen[nd.leaf]));
            } else {
                const double y = ys[(size_t)nd.k * KP + k];
                if (node == 0) us[k] = 1.0;
                us[(size_t)nd.left * KP + k] = __dmul_rn(y, ui);
                us[(size_t)nd.right * KP + k] = __dmul_rn(__dsub_rn(1.0, y), ui);
                if (want_ladj) lacc += log(ui);
            }
        }
        __syncthreads();
    }
    if (S_partial) block_reduce_k<KP, THREADS>(sacc, sm, S_partial + (size_t)(part_base + blockIdx.x) * KP);
    if (want_ladj) block_reduce_k<KP, THREADS>(lacc, sm, ladj_partial + (size_t)(part_base + blockIdx.x) * KP);
}

// ---------------------------------------------------------------- mid-step: S reduction + step bookkeeping
__global__ void __launch_bounds__(1024)
    k3_mid(const double *__restrict__ S_partial, int count, int KP, double *__restrict__ S, StepCtl *ctl, int advance) {
    __shared__ double sm[1024];
    const int k = threadIdx.x % KP, lane_t = threadIdx.x / KP, per = 1024 / KP;
    double s = 0.0;
    for (int t = lane_t; t < count; t += per) s += S_partial[(size_t)t * KP + k];
    sm[threadIdx.x] = s;
    __syncthreads();
    for (int span = per / 2; span >= 1; span >>= 1) {
        if (lane_t < span) sm[threadIdx.x] += sm[threadIdx.x + span * KP];
        __syncthreads();
    }
    if (threadIdx.x < KP) S[threadIdx.x] = sm[threadIdx.x];
    if (advance && threadIdx.x == 0) {
        ctl->step_upd = ctl->step_fwd;
        ctl->step_fwd = ctl->step_fwd + 1;
    }
}

// ---------------------------------------------------------------- tree backward
// WITH_LADJ: transform_gradients! (y_grad rounded to Float32 as in the reference's Float32 vector);
// otherwise transform_gradients_no_ladj! with a Float64 y_grad (OptimizePTTApprox).
template <int KP, int THREADS, bool WITH_LADJ>
__global__ void __launch_bounds__(THREADS)
    k3_tree_bwd(const int32_t *__restrict__ bin_lvl_ptr, const int32_t *__restrict__ lvl_off,
                const int32_t *__restrict__ sch_node, const TreeNode *__restrict__ nodes,
                const double *__restrict__ ys, const double *__restrict__ us, const double *__restrict__ g,
                const float *__restrict__ efflen_adj, const double *__restrict__ S, float2 *__restrict__ G,
                double *__restrict__ ygrad, double *__restrict__ xgrad_out) {
    const int k = threadIdx.x % KP, slot = threadIdx.x / KP;
    constexpr int NPP = THREADS / KP;
    const int l0 = bin_lvl_ptr[blockIdx.x], l1 = bin_lvl_ptr[blockIdx.x + 1] - 1;
    for (int l = l1 - 1; l >= l0; --l) {
        const int lo = lvl_off[l], hi = lvl_off[l + 1];
        for (int q = lo + slot; q < hi; q += NPP) {
            const int node = sch_node[q];
            const TreeNode nd = nodes[node];
            if (nd.leaf >= 0) {
                double gv = g[(size_t)nd.leaf * KP + k];
                if (efflen_adj) gv = __dsub_rn(gv, __ddiv_rn((double)efflen_adj[nd.leaf], S[k]));  // likelihood.jl:105
                if (xgrad_out) xgrad_out[(size_t)nd.leaf * KP + k] = gv;
                G[(size_t)node * KP + k] = make_float2((float)gv, 0.0f);
            } else {
                const float2 gl = G[(size_t)nd.left * KP + k], gr = G[(size_t)nd.right * KP + k];
                const double y = ys[(size_t)nd.k * KP + k];
                const double ui = node == 0 ? 1.0 : us[(size_t)node * KP + k];
                const double omy = __dsub_rn(1.0, y);
                float2 out;
                out.x = (float)__dadd_rn(__dmul_rn(y, (double)gl.x), __dmul_rn(omy, (double)gr.x));
                if (WITH_LADJ) {
                    const float d = __fsub_rn(__fadd_rn(gl.x, gl.y), __fadd_rn(gr.x, gr.y));
                    ygrad[(size_t)nd.k * KP + k] = (double)(float)__dmul_rn(ui, (double)d);
                    out.y = (float)__dadd_rn(__dadd_rn(__ddiv_rn(1.0, ui), __dmul_rn(y, (double)gl.y)),
                                             __dmul_rn(omy, (double)gr.y));
                } else {
                    const float d = __fsub_rn(gl.x, gr.x);
                    ygrad[(size_t)nd.k * KP + k] = __dmul_rn(ui, (double)d);
                    out.y = 0.0f;
                }
                G[(size_t)node * KP + k] = out;
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------- inverse transform
// inverse_transform! (src/ptt.jl:257-285): u_i = x_leaf at a leaf, u_left + u_right at an internal node (one Float64
// add per node, the association the reference's descending-index sweep has, so the same bits), y_k = u_left / u_i and
// logu_k = log(Float32(u_i)).  Level-synchronous from the deepest level up, one CTA per schedule bin (bottom forests,
// then the top part).  us is indexed by node here.
template <int KP, int THREADS>
__global__ void __launch_bounds__(THREADS)
    k3_tree_inv(const int32_t *__restrict__ bin_lvl_ptr, const int32_t *__restrict__ lvl_off,
                const int32_t *__restrict__ sch_node, const TreeNode *__restrict__ nodes, const float *__restrict__ x,
                double *__restrict__ us, double *__restrict__ ys, float *__restrict__ logu) {
    const int k = threadIdx.x % KP, slot = threadIdx.x / KP;
    constexpr int NPP = THREADS / KP;
    const int l0 = bin_lvl_ptr[blockIdx.x], l1 = bin_lvl_ptr[blockIdx.x + 1] - 1;
    for (int l = l1 - 1; l >= l0; --l) {
        const int lo = lvl_off[l], hi = lvl_off[l + 1];
        for (int q = lo + slot; q < hi; q += NPP) {
            const int node = sch_node[q];
            const TreeNode nd = nodes[node];
            if (nd.leaf >= 0) {
                us[(size_t)node * KP + k] = (double)x[(size_t)nd.leaf * KP + k];
            } else {
                const double ul = us[(size_t)nd.left * KP + k], ur = us[(size_t)nd.right * KP + k];
                const double ui = __dadd_rn(ul, ur);
                us[(size_t)node * KP + k] = ui;
                ys[(size_t)nd.k * KP + k] = __ddiv_rn(ul, ui);
                if (logu) logu[(size_t)nd.k * KP + k] = logf((float)ui);
            }
        }
        __syncthreads();
    }
}

// The same sweep for caterpillar (:sequential) trees, whose depth is n: one thread per draw walks the nodes in the
// reference's own order (descending index), children before parents by construction of the node order.
__global__ void k3_tree_inv_serial(int64_t N, int KP, const TreeNode *__restrict__ nodes, const float *__restrict__ x,
                                   double *us, double *__restrict__ ys, float *__restrict__ logu) {
    const int k = threadIdx.x;
    if (k >= KP) return;
    for (int64_t i = N - 1; i >= 0; --i) {
        const TreeNode nd = nodes[i];
        if (nd.leaf >= 0) {
            us[(size_t)i * KP + k] = (double)x[(size_t)nd.leaf * KP + k];
        } else {
            const double ul = us[(size_t)nd.left * KP + k], ur = us[(size_t)nd.right * KP + k];
            const double ui = __dadd_rn(ul, ur);
            us[(size_t)i * KP + k] = ui;
            ys[(size_t)nd.k * KP + k] = __ddiv_rn(ul, ui);
            if (logu) logu[(size_t)nd.k * KP + k] = logf((float)ui);
        }
    }
}

// ladj = - sum_k log(Float32(u_k)), a Float64 accumulator fed in the reference's order (descending node index =
// descending k, ptt.jl:265-281): one thread per draw, the loads do not depend on the chain of adds
__global__ void k3_inv_ladj(int64_t nm1, int KP, const float *__restrict__ logu, double *__restrict__ ladj) {
    const int k = threadIdx.x;
    if (k >= KP) return;
    double l = 0.0;
#pragma unroll 8
    for (int64_t i = nm1 - 1; i >= 0; --i) l = __dsub_rn(l, (double)logu[(size_t)i * KP + k]);
    ladj[k] = l;
}

__global__ void k3_fill_f32(float *__restrict__ p, int64_t count, float v) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < count) p[i] = v;
}

// mu = Float32(logit(y)) in Float64 (map!(logit, mu, ys), likelihood-approximation.jl:453), omega = log(0.1f0), alpha = 0
__global__ void k3_init_params(int64_t nm1, int KP, const double *__restrict__ ys, float omega0, float *__restrict__ mu0,
                               float *__restrict__ mu, float *__restrict__ omega, float *__restrict__ alpha) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= nm1) return;
    float v;
    if (ys) {
        const double y = ys[(size_t)i * KP];
        v = (float)log(__ddiv_rn(y, __dsub_rn(1.0, y)));
        mu0[i] = v;
    } else {
        v = mu0[i];
    }
    mu[i] = v;
    omega[i] = omega0;
    alpha[i] = 0.0f;
}

// ================================================================ shared-memory tree kernels
// Same arithmetic as k3_tree_fwd / k3_tree_bwd above, but a CTA first pulls everything its bin needs into shared
// memory with coalesced loads (schedule-order records, ys, the u of its subtree roots / the G of its leaves), runs
// the level loops entirely out of shared memory (one __syncthreads per level, no global load on the critical path)
// and writes its results back at the end.  grid = (bins, KP / KPC): KPC draws per CTA (8 for the bottom forests,
// 1 for the top part so that a few thousand nodes fit).  Bottom subtree roots exchange u (top -> bottom) and G
// (bottom -> top) through [slot][KP] arrays.  The forward kernel also leaves u of every internal node by k in us_k,
// where the backward kernel reads it, as it does after the DFS-run and path-product forward kernels.
template <int KPC, int THREADS>
__device__ __forceinline__ void block_reduce_kc(double v, double *red, double *out /* [KPC] */) {
    red[threadIdx.x] = v;
    __syncthreads();
    for (int span = THREADS / KPC / 2; span >= 1; span >>= 1) {
        if ((int)threadIdx.x < span * KPC) red[threadIdx.x] += red[threadIdx.x + span * KPC];
        __syncthreads();
    }
    if (threadIdx.x < KPC) out[threadIdx.x] = red[threadIdx.x];
    __syncthreads();
}

template <int KP, int KPC, int THREADS, int MINB>
__global__ void __launch_bounds__(THREADS, MINB)
    k3s_tree_fwd(const int32_t *__restrict__ bin_off, const int32_t *__restrict__ bin_lvl_ptr,
                 const int32_t *__restrict__ lvl_off, const SNode *__restrict__ recs, const double *__restrict__ ys,
                 double *__restrict__ root_us, double *__restrict__ us_k, float *__restrict__ x, int clamp_x,
                 const float *__restrict__ efflen, double *__restrict__ S_partial, int part_base, int want_ladj,
                 double *__restrict__ ladj_partial) {
    extern __shared__ __align__(16) unsigned char smraw[];
    __shared__ double red[THREADS];
    const int q0 = bin_off[blockIdx.x], nb = bin_off[blockIdx.x + 1] - q0;
    SNode *rec_s = reinterpret_cast<SNode *>(smraw);
    double *us_s = reinterpret_cast<double *>(smraw + (size_t)nb * sizeof(SNode));
    double *ys_s = us_s + (size_t)nb * KPC;
    int *lvl_s = reinterpret_cast<int *>(ys_s + (size_t)nb * KPC);
    const int kk = threadIdx.x % KPC, slot_t = threadIdx.x / KPC, k = blockIdx.y * KPC + kk;
    constexpr int NPP = THREADS / KPC;
    const int l0 = bin_lvl_ptr[blockIdx.x], nlev = bin_lvl_ptr[blockIdx.x + 1] - 1 - l0;

    for (int p = threadIdx.x; p < nb; p += THREADS) rec_s[p] = recs[q0 + p];
    for (int l = threadIdx.x; l <= nlev; l += THREADS) lvl_s[l] = lvl_off[l0 + l] - q0;
    __syncthreads();
    // gather phase, 4 positions per thread in flight (the loads are independent: batch them for MLP)
    for (int base = slot_t; base < nb; base += 4 * NPP) {
        SNode r[4];
        double yv[4], uv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int p = base + u * NPP;
            r[u] = p < nb ? rec_s[p] : SNode{-1, -1, -1, -2};
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            yv[u] = 0.0;
            uv[u] = 1.0;
            if (r[u].k_or_leaf >= 0) yv[u] = ys[(size_t)r[u].k_or_leaf * KP + k];
            if (r[u].slot >= 0 && r[u].k_or_leaf != INT32_MIN) uv[u] = root_us[(size_t)r[u].slot * KP + k];
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int p = base + u * NPP;
            if (p < nb) {
                if (r[u].k_or_leaf >= 0) ys_s[p * KPC + kk] = yv[u];
                if (r[u].slot >= -1 && r[u].k_or_leaf != INT32_MIN) us_s[p * KPC + kk] = uv[u];
            }
        }
    }
    __syncthreads();

    double sacc = 0.0, lacc = 0.0;
    for (int l = 0; l < nlev; ++l) {
        const int lo = lvl_s[l], hi = lvl_s[l + 1];
        for (int p = lo + slot_t; p < hi; p += NPP) {
            const SNode r = rec_s[p];
            const double ui = us_s[p * KPC + kk];
            if (r.k_or_leaf >= 0) {
                const double y = ys_s[p * KPC + kk];
                us_s[r.left * KPC + kk] = __dmul_rn(y, ui);
                us_s[r.right * KPC + kk] = __dmul_rn(__dsub_rn(1.0, y), ui);
                us_k[(size_t)r.k_or_leaf * KP + k] = ui;
                if (want_ladj) lacc += log(ui);
            } else if (r.k_or_leaf == INT32_MIN) {
                root_us[(size_t)r.slot * KP + k] = ui;  // a bottom subtree root: hand u over
            } else {
                const int leaf = -1 - r.k_or_leaf;
                float xv = (float)ui;
                double d = (double)xv;
                xv = (float)(d > 1e-16 ? d : 1e-16);  // ptt.jl:136-137
                if (clamp_x) {                         // clamp!(xs, 1e-10, 1 - 1e-10) on a Float32 vector
                    d = (double)xv;
                    d = fmin(fmax(d, 1e-10), 1.0 - 1e-10);
                    xv = (float)d;
                }
                x[(size_t)leaf * KP + k] = xv;
                if (efflen) sacc = __dadd_rn(sacc, (double)__fdiv_rn(xv, __int_as_float(r.left)));
            }
        }
        __syncthreads();
    }
    if (S_partial)
        block_reduce_kc<KPC, THREADS>(sacc, red, S_partial + (size_t)(part_base + blockIdx.x) * KP + blockIdx.y * KPC);
    if (want_ladj)
        block_reduce_kc<KPC, THREADS>(lacc, red, ladj_partial + (size_t)(part_base + blockIdx.x) * KP + blockIdx.y * KPC);
}

template <int KP, int KPC, int THREADS, int MINB, bool WITH_LADJ>
__global__ void __launch_bounds__(THREADS, MINB)
    k3s_tree_bwd(const int32_t *__restrict__ bin_off, const int32_t *__restrict__ bin_lvl_ptr,
                 const int32_t *__restrict__ lvl_off, const SNode *__restrict__ recs, const double *__restrict__ ys,
                 const double *__restrict__ us_k, float2 *__restrict__ root_G, const double *__restrict__ g,
                 const float *__restrict__ efflen_adj, const double *__restrict__ S, double *__restrict__ ygrad,
                 double *__restrict__ xgrad_out) {
    // us_k: u of every internal node by k, as the forward kernel left it
    extern __shared__ __align__(16) unsigned char smraw[];
    const int q0 = bin_off[blockIdx.x], nb = bin_off[blockIdx.x + 1] - q0;
    SNode *rec_s = reinterpret_cast<SNode *>(smraw);
    double *us_s = reinterpret_cast<double *>(smraw + (size_t)nb * sizeof(SNode));
    double *ys_s = us_s + (size_t)nb * KPC;
    float2 *G_s = reinterpret_cast<float2 *>(ys_s + (size_t)nb * KPC);
    int *lvl_s = reinterpret_cast<int *>(G_s + (size_t)nb * KPC);
    const int kk = threadIdx.x % KPC, slot_t = threadIdx.x / KPC, k = blockIdx.y * KPC + kk;
    constexpr int NPP = THREADS / KPC;
    const int l0 = bin_lvl_ptr[blockIdx.x], nlev = bin_lvl_ptr[blockIdx.x + 1] - 1 - l0;

    pdl_trigger();
    for (int p = threadIdx.x; p < nb; p += THREADS) rec_s[p] = recs[q0 + p];
    for (int l = threadIdx.x; l <= nlev; l += THREADS) lvl_s[l] = lvl_off[l0 + l] - q0;
    pdl_wait();  // the schedule above is constant; ys, us_k, g, root_G and S come from this step's kernels
    __syncthreads();
    const double Sk = efflen_adj ? S[k] : 1.0;
    for (int base = slot_t; base < nb; base += 4 * NPP) {
        SNode r[4];
        double v0[4], uv[4];
        float adj[4];
        float2 gx[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int p = base + u * NPP;
            r[u] = p < nb ? rec_s[p] : SNode{-1, -1, -1, -2};
            if (p >= nb) r[u].k_or_leaf = INT32_MIN + 1;  // nothing to load
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            v0[u] = 0.0; uv[u] = 1.0; adj[u] = 0.0f; gx[u] = make_float2(0.f, 0.f);
            if (r[u].k_or_leaf >= 0) {
                v0[u] = ys[(size_t)r[u].k_or_leaf * KP + k];
                uv[u] = us_k[(size_t)r[u].k_or_leaf * KP + k];
            } else if (r[u].k_or_leaf == INT32_MIN) {
                gx[u] = root_G[(size_t)r[u].slot * KP + k];
            } else if (r[u].k_or_leaf != INT32_MIN + 1) {
                const int leaf = -1 - r[u].k_or_leaf;
                v0[u] = g[(size_t)leaf * KP + k];
                if (efflen_adj) adj[u] = __int_as_float(r[u].right);
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int p = base + u * NPP;
            if (p >= nb) continue;
            if (r[u].k_or_leaf >= 0) {
                ys_s[p * KPC + kk] = v0[u];
                us_s[p * KPC + kk] = uv[u];
            } else if (r[u].k_or_leaf == INT32_MIN) {
                G_s[p * KPC + kk] = gx[u];
            } else {
                const int leaf = -1 - r[u].k_or_leaf;
                double gv = v0[u];
                if (efflen_adj) gv = __dsub_rn(gv, __ddiv_rn((double)adj[u], Sk));  // likelihood.jl:105
                if (xgrad_out) xgrad_out[(size_t)leaf * KP + k] = gv;
                G_s[p * KPC + kk] = make_float2((float)gv, 0.0f);
            }
        }
    }
    __syncthreads();

    // backward sweep
    for (int l = nlev - 1; l >= 0; --l) {
        const int lo = lvl_s[l], hi = lvl_s[l + 1];
        for (int p = lo + slot_t; p < hi; p += NPP) {
            const SNode r = rec_s[p];
            if (r.k_or_leaf >= 0) {
                const float2 gl = G_s[r.left * KPC + kk], gr = G_s[r.right * KPC + kk];
                const double y = ys_s[p * KPC + kk], ui = us_s[p * KPC + kk];
                const double omy = __dsub_rn(1.0, y);
                float2 out;
                out.x = (float)__dadd_rn(__dmul_rn(y, (double)gl.x), __dmul_rn(omy, (double)gr.x));
                if (WITH_LADJ) {
                    const float d = __fsub_rn(__fadd_rn(gl.x, gl.y), __fadd_rn(gr.x, gr.y));
                    ygrad[(size_t)r.k_or_leaf * KP + k] = (double)(float)__dmul_rn(ui, (double)d);
                    out.y = (float)__dadd_rn(__dadd_rn(__ddiv_rn(1.0, ui), __dmul_rn(y, (double)gl.y)),
                                             __dmul_rn(omy, (double)gr.y));
                } else {
                    const float d = __fsub_rn(gl.x, gr.x);
                    ygrad[(size_t)r.k_or_leaf * KP + k] = __dmul_rn(ui, (double)d);
                    out.y = 0.0f;
                }
                G_s[p * KPC + kk] = out;
            }
            if (r.slot >= 0 && r.k_or_leaf != INT32_MIN && l == 0)
                root_G[(size_t)r.slot * KP + k] = G_s[p * KPC + kk];  // bottom subtree root: hand G to the top part
        }
        __syncthreads();
    }
}

// transform! (src/ptt.jl:125-158) as path products: u_i is the product, from the root down, of y (into a left child) or
// 1 - y (into a right child) -- the very multiplications the reference's index-order sweep performs on the way to node
// i, in the same order, so every u (and x) has the reference's bits; but no node waits for another, so there are no
// levels and no exchange between kernels.  One CTA = one group of PATH_GROUP consecutive nodes x KP draws: the y of the
// group's distinct ancestors are gathered into shared memory once (neighbours in DFS order share nearly all of them),
// then a thread = (PATH_GROUP / PATH_SLOTS nodes, one draw) multiplies along the group's common path prefix once and
// along each of its nodes' own suffixes.  Internal nodes store u by k for the backward kernels, leaves produce x.
template <int KP>
__global__ void __launch_bounds__(PATH_SLOTS *KP, 2048 / (PATH_SLOTS * KP) > 16 ? 16 : 2048 / (PATH_SLOTS * KP))
    k3p_tree_fwd(int64_t N, const TreeNode *__restrict__ nodes, const uint32_t *__restrict__ ganc_ptr,
                 const uint32_t *__restrict__ ganc, const uint32_t *__restrict__ gcp, const uint32_t *__restrict__ nsuf_ptr,
                 const uint16_t *__restrict__ nsuf, const double *__restrict__ ys, double *__restrict__ us_k,
                 float *__restrict__ x, int clamp_x, const float *__restrict__ efflen,
                 double *__restrict__ S_partial, int want_ladj, double *__restrict__ ladj_partial) {
    constexpr int THREADS = PATH_SLOTS * KP, NPT = PATH_GROUP / PATH_SLOTS;
    extern __shared__ __align__(16) unsigned char smraw[];
    __shared__ double red[THREADS];
    const int k = threadIdx.x % KP, t = threadIdx.x / KP;
    // everything that does not depend on another load first
    const uint32_t a0 = ganc_ptr[blockIdx.x], na = ganc_ptr[blockIdx.x + 1] - a0, cp = gcp[blockIdx.x];
    const int64_t g0 = (int64_t)blockIdx.x * PATH_GROUP, i0 = g0 + t;
    const int64_t g1 = g0 + PATH_GROUP < N ? g0 + PATH_GROUP : N;
    const uint32_t s0 = nsuf_ptr[g0], ns = nsuf_ptr[g1] - s0;  // the group's suffix entries are contiguous
    TreeNode nd[NPT];
    uint32_t sb[NPT], se[NPT];
#pragma unroll
    for (int j = 0; j < NPT; ++j) {
        const int64_t i = i0 + j * PATH_SLOTS;
        nd[j] = TreeNode{-1, -1, -1, -1};
        sb[j] = se[j] = 0;
        if (i < N) {
            nd[j] = nodes[i];
            sb[j] = nsuf_ptr[i] - s0;
            se[j] = nsuf_ptr[i + 1] - s0;
        }
    }
    // shared memory: yy[2 a + side][KP] = y of ancestor a (side 1: the path goes left) or 1 - y (side 0: right), so a
    // path step is one load and one multiply; pre[a] = 2 a + side of the common prefix; suf[] = the group's suffixes
    double *yy_s = reinterpret_cast<double *>(smraw);                          // [2 na][KP]
    uint16_t *pre_s = reinterpret_cast<uint16_t *>(yy_s + (size_t)2 * na * KP);  // [cp]
    uint16_t *suf_s = pre_s + ((cp + 7u) & ~7u);                                 // [ns]
    for (uint32_t a = t; a < na; a += PATH_SLOTS) {
        const uint32_t en = ganc[a0 + a];
        if (k == 0 && a < cp) pre_s[a] = (uint16_t)((a << 1) | (en & 1u));
        const double y = ys[(size_t)(en >> 1) * KP + k];
        yy_s[(2 * a + 1) * KP + k] = y;
        yy_s[(2 * a) * KP + k] = __dsub_rn(1.0, y);
    }
    for (uint32_t e = threadIdx.x; e < ns; e += THREADS) suf_s[e] = nsuf[s0 + e];
    float ef[NPT];
#pragma unroll
    for (int j = 0; j < NPT; ++j) ef[j] = (efflen && nd[j].leaf >= 0) ? efflen[nd[j].leaf] : 1.0f;
    __syncthreads();
    const double *yk = yy_s + k;
    double up = 1.0;  // the group's common prefix
#pragma unroll 4
    for (uint32_t a = 0; a < cp; ++a) up = __dmul_rn(yk[(uint32_t)pre_s[a] * KP], up);
    double sacc = 0.0, lacc = 0.0;
#pragma unroll
    for (int j = 0; j < NPT; ++j) {
        if (i0 + j * PATH_SLOTS >= N) continue;
        double u = up;
#pragma unroll 4
        for (uint32_t e = sb[j]; e < se[j]; ++e) u = __dmul_rn(yk[(uint32_t)suf_s[e] * KP], u);
        if (nd[j].leaf >= 0) {
            float xv = (float)u;
            double d = (double)xv;
            xv = (float)(d > 1e-16 ? d : 1e-16);  // ptt.jl:136-137
            if (clamp_x) {                         // clamp!(xs, 1e-10, 1 - 1e-10) on a Float32 vector
                d = (double)xv;
                d = fmin(fmax(d, 1e-10), 1.0 - 1e-10);
                xv = (float)d;
            }
            x[(size_t)nd[j].leaf * KP + k] = xv;
            if (efflen) sacc = __dadd_rn(sacc, (double)__fdiv_rn(xv, ef[j]));
        } else {
            us_k[(size_t)nd[j].k * KP + k] = u;
            if (want_ladj) lacc += log(u);
        }
    }
    if (S_partial) block_reduce_kc<KP, THREADS>(sacc, red, S_partial + (size_t)blockIdx.x * KP);
    if (want_ladj) block_reduce_kc<KP, THREADS>(lacc, red, ladj_partial + (size_t)blockIdx.x * KP);
}

// transform! (src/ptt.jl:125-158) for trees stored in DFS pre-order (what order_nodes emits: a node, its right subtree,
// its left subtree): a thread = (run of DFS_RUN consecutive nodes, one draw) walks its nodes in index order exactly as
// the reference's sweep does.  At an internal node it forms both children's u (the reference's two multiplications): the
// right child is the next node and takes its value from a register, the left child's value waits in a per-thread stack
// indexed by depth (shared memory, [depth][thread]: conflict-free) until the walk comes back to it.  The stack a run
// starts with is what the serial sweep would hold there: the thread multiplies down the root path of its first node
// (ancestor list prepared on the host) and parks the left values of the ancestors it passes on the right.  Every u is
// therefore the reference's product chain from the root -- the same bits -- at ~20 instructions per node instead of a
// path product per node, with no levels, no barriers between levels and no exchange between kernels.  The CTA's nodes and
// the y of its internal nodes (consecutive k: one contiguous slice of ys) are staged in shared memory by coalesced loads.
template <int KP>
__global__ void __launch_bounds__(DFS_RUNS_PER_CTA *KP)
    k3d_tree_fwd(int64_t N, const DNode *__restrict__ dnodes, const uint32_t *__restrict__ run_anc_ptr,
                 const uint32_t *__restrict__ run_anc, const int32_t *__restrict__ cta_k0, const double *__restrict__ ys,
                 double *__restrict__ us_k, float *__restrict__ x, int clamp_x, int want_ladj,
                 double *__restrict__ ladj_partial, int stack_levels, int max_nk) {
    constexpr int THREADS = DFS_RUNS_PER_CTA * KP, RS = DFS_RUN + 2;  // record stride of a run: 16-byte aligned, 4 banks apart
    extern __shared__ __align__(16) unsigned char smraw[];
    __shared__ double red[THREADS];
    double *stack = reinterpret_cast<double *>(smraw);                      // [stack_levels][THREADS]
    double *ys_s = stack + (size_t)stack_levels * THREADS;                  // [max_nk][KP]
    DNode *rec_s = reinterpret_cast<DNode *>(ys_s + (size_t)max_nk * KP);   // [DFS_RUNS_PER_CTA][RS]
    const int k = threadIdx.x % KP, rl = threadIdx.x / KP;
    const int64_t c0 = (int64_t)blockIdx.x * DFS_CTA_NODES;
    const int nn = (int)(N - c0 < DFS_CTA_NODES ? N - c0 : DFS_CTA_NODES);
    const int k0 = cta_k0[blockIdx.x], nk = cta_k0[blockIdx.x + 1] - k0;
    pdl_trigger();
    // ---- stage the CTA's node records and y slice (one contiguous piece of ys) with 1-D bulk copies (TMA) completing
    // on an mbarrier; they are in flight while the threads walk the root paths.  The records (and the first batch of
    // each run's ancestor list below) are constant and requested before pdl_wait(); ys is the previous step's output.
    __shared__ uint64_t bar;
    const bool bulk = KP >= 2;  // 16-byte granularity: k0 KP and nk KP doubles are even then
    if (bulk) {
        if (threadIdx.x == 0) {
            mbar_init(&bar, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            // 8-byte records, 16-byte copies: an odd tail takes the padding record the host appended
            const int nn2 = (nn + 1) & ~1;
            mbar_expect_tx(&bar, (uint32_t)(nk * KP * 8 + nn2 * (int)sizeof(DNode)));
            for (int q = 0; q * DFS_RUN < nn2; ++q) {
                const int len = nn2 - q * DFS_RUN < DFS_RUN ? nn2 - q * DFS_RUN : DFS_RUN;
                bulk_g2s(rec_s + q * RS, dnodes + c0 + (int64_t)q * DFS_RUN, (uint32_t)(len * sizeof(DNode)), &bar);
            }
        }
    } else {
        for (int idx = threadIdx.x; idx < nn; idx += THREADS) rec_s[(idx / DFS_RUN) * RS + idx % DFS_RUN] = dnodes[c0 + idx];
    }
    // ---- the run's starting state: down the root path of its first node
    constexpr int AB = 16;  // ancestors per batch: their y are all requested before the first product
    const int64_t i0 = c0 + (int64_t)rl * DFS_RUN;
    const int cnt = i0 < N ? (int)(N - i0 < DFS_RUN ? N - i0 : DFS_RUN) : 0;
    uint32_t a0 = 0, na = 0, en[AB];
    if (cnt > 0) {
        const int64_t run = i0 / DFS_RUN;
        a0 = run_anc_ptr[run];
        na = run_anc_ptr[run + 1] - a0;
    }
#pragma unroll
    for (int j = 0; j < AB; ++j) en[j] = j < (int)na ? run_anc[a0 + j] : 0u;
    pdl_wait();
    if (bulk) {
        if (threadIdx.x == 0 && nk > 0) bulk_g2s(ys_s, ys + (size_t)k0 * KP, (uint32_t)(nk * KP * 8), &bar);
    } else {
        for (int idx = threadIdx.x; idx < nk * KP; idx += THREADS) ys_s[idx] = ys[(size_t)k0 * KP + idx];
    }
    double *st = stack + threadIdx.x;
    double u = 1.0;
    if (cnt > 0) {
        for (uint32_t a = 0; a < na; a += AB) {
            double yv[AB];
            if (a > 0) {
#pragma unroll
                for (int j = 0; j < AB; ++j) en[j] = a + j < na ? run_anc[a0 + a + j] : 0u;
            }
#pragma unroll
            for (int j = 0; j < AB; ++j) yv[j] = a + j < na ? ys[(size_t)(en[j] >> 1) * KP + k] : 0.0;
#pragma unroll
            for (int j = 0; j < AB; ++j) {
                if (a + j < na) {
                    const double ul = __dmul_rn(yv[j], u), ur = __dmul_rn(__dsub_rn(1.0, yv[j]), u);
                    if (en[j] & 1u) {
                        u = ul;  // into the left child: its right sibling's subtree lies before this run
                    } else {
                        st[(size_t)(a + j + 1) * THREADS] = ul;  // the left child (depth a + j + 1) comes later
                        u = ur;
                    }
                }
            }
        }
    }
    if (bulk) mbar_wait(&bar, 0);
    else __syncthreads();
    // ---- the run, in node order.  The record and the y of the NEXT node are fetched before the current node is
    // worked on, so that only the products (and the stack read of a left child) are on the thread's critical path
    double lacc = 0.0, carry = 0.0;
    const DNode *rr = rec_s + rl * RS;
    DNode rn = cnt > 0 ? rr[0] : DNode{-1, 0u};
    double yn = (cnt > 0 && rn.k_or_leaf >= 0) ? ys_s[(rn.k_or_leaf - k0) * KP + k] : 0.0;
    for (int j = 0; j < cnt; ++j) {
        const DNode r = rn;
        const double y = yn, omy = __dsub_rn(1.0, yn);
        if (j + 1 < cnt) {
            rn = rr[j + 1];
            yn = rn.k_or_leaf >= 0 ? ys_s[(rn.k_or_leaf - k0) * KP + k] : 0.0;
        }
        const uint32_t d = r.meta & 0x7fffffffu;
        if (j > 0) u = (r.meta >> 31) ? st[(size_t)d * THREADS] : carry;
        if (r.k_or_leaf >= 0) {
            st[(size_t)(d + 1) * THREADS] = __dmul_rn(y, u);
            carry = __dmul_rn(omy, u);
            us_k[(size_t)r.k_or_leaf * KP + k] = u;
            if (want_ladj) lacc += log(u);
        } else {
            const int leaf = -1 - r.k_or_leaf;
            // xs[j] = max(us[i], 1e-16) stored as Float32 (ptt.jl:136-137), then clamp!(xs, 1e-10, 1 - 1e-10) on the Float32
            // vector (l-a.jl:526).  In Float32 alone: a Float32 lies below the Float64 bound exactly when it lies below the
            // bound rounded to Float32, and Float32(1 - 1e-10) is 1, so these are the reference's values bit for bit
            float xv = fmaxf((float)u, (float)1e-16);
            if (clamp_x) xv = fminf(fmaxf(xv, (float)1e-10), 1.0f);
            x[(size_t)leaf * KP + k] = xv;
        }
    }
    if (want_ladj) block_reduce_kc<KP, THREADS>(lacc, red, ladj_partial + (size_t)blockIdx.x * KP);
}

// S_k = sum_j x_jk / efflen_j (effective_length_jacobian_adjustment!, likelihood.jl:96-100: Float32 quotients, Float64
// sum) and the step bookkeeping of k3_mid, for the forward kernels that leave S out of their node loop.  A warp adds
// LEAF_S_PER_WARP transcripts (all loads of a batch in flight, fixed order) and writes one partial row; the CTA that
// finishes last adds the partial rows, again in a fixed order.  Small on purpose (128 threads, ~1 KB of shared memory):
// it runs on the side stream in the registers and shared memory the likelihood kernel leaves free on every SM.
constexpr int LEAF_S_THREADS = 128, LEAF_S_PER_WARP = 256;
template <int KP>
__global__ void __launch_bounds__(LEAF_S_THREADS)
    k3_leaf_S(int64_t n, const float *__restrict__ x, const float *__restrict__ efflen, double *__restrict__ S_partial,
              int nwarps, double *__restrict__ S, StepCtl *ctl, int advance, unsigned int *counter) {
    constexpr int LPW = 32 / KP;  // transcripts per warp-wide step
    constexpr int UN = 8;
    __shared__ double red[LEAF_S_THREADS];
    __shared__ bool last;
    const int lane = threadIdx.x & 31, k = lane % KP, slot = lane / KP;
    const int w = (int)((blockIdx.x * (size_t)LEAF_S_THREADS + threadIdx.x) >> 5);
    if (w < nwarps) {
        const int64_t j0 = (int64_t)w * LEAF_S_PER_WARP, j1 = j0 + LEAF_S_PER_WARP < n ? j0 + LEAF_S_PER_WARP : n;
        double sacc = 0.0;
        for (int64_t jb = j0 + slot; jb < j1; jb += (int64_t)UN * LPW) {
            float xv[UN], ev[UN];
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                const int64_t j = jb + (int64_t)u * LPW;
                xv[u] = j < j1 ? x[(size_t)j * KP + k] : 0.0f;
                ev[u] = j < j1 ? efflen[j] : 1.0f;
            }
#pragma unroll
            for (int u = 0; u < UN; ++u) sacc = __dadd_rn(sacc, (double)__fdiv_rn(xv[u], ev[u]));
        }
#pragma unroll
        for (int o = KP; o < 32; o <<= 1) sacc = __dadd_rn(sacc, __shfl_xor_sync(0xffffffffu, sacc, o));
        if (lane < KP) S_partial[(size_t)w * KP + k] = sacc;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(counter, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    // the last CTA: S[k] = sum over the warps' partial rows
    constexpr int SLOTS = LEAF_S_THREADS / KP;
    const int kk = threadIdx.x % KP, ss = threadIdx.x / KP;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    int t = ss;
    for (; t + 3 * SLOTS < nwarps; t += 4 * SLOTS) {
        a0 += __ldcg(S_partial + (size_t)t * KP + kk);
        a1 += __ldcg(S_partial + (size_t)(t + SLOTS) * KP + kk);
        a2 += __ldcg(S_partial + (size_t)(t + 2 * SLOTS) * KP + kk);
        a3 += __ldcg(S_partial + (size_t)(t + 3 * SLOTS) * KP + kk);
    }
    for (; t < nwarps; t += SLOTS) a0 += __ldcg(S_partial + (size_t)t * KP + kk);
    red[threadIdx.x] = (a0 + a1) + (a2 + a3);
    __syncthreads();
    for (int span = SLOTS / 2; span >= 1; span >>= 1) {
        if (ss < span) red[threadIdx.x] += red[threadIdx.x + span * KP];
        __syncthreads();
    }
    if (threadIdx.x < KP) S[threadIdx.x] = red[threadIdx.x];
    if (threadIdx.x == 0) {
        *counter = 0u;
        if (advance) {
            ctl->step_upd = ctl->step_fwd;
            ctl->step_fwd = ctl->step_fwd + 1;
        }
    }
}

// Leaf records carry the leaf's effective length (left) and Float32(n / efflen) (right) as raw Float32 bits, so the
// level loops never touch global memory for them.
__global__ void k_patch_leaf_recs(SNode *recs, int count, const float *__restrict__ efflen, const float *__restrict__ adj) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= count) return;
    SNode r = recs[q];
    if (r.k_or_leaf < 0 && r.k_or_leaf != INT32_MIN) {
        const int leaf = -1 - r.k_or_leaf;
        r.left = __float_as_int(efflen[leaf]);
        r.right = __float_as_int(adj[leaf]);
        recs[q] = r;
    }
}

// ---------------------------------------------------------------- reparameterisation backward + ADAM
struct AdamCfg {
    double max_step_mu, max_step_omega, max_step_alpha, max_step_z;
};

__device__ __forceinline__ void adam_one(float &param, float &m, float &v, double grad, float grad_sq_f32,
                                         bool grad_is_f32, int step, double lr, double m_denom, double v_denom,
                                         double max_step) {
    // adam_update_mv!  l-a.jl:116-130
    if (step == 1) {
        m = (float)grad;
        v = grad_is_f32 ? grad_sq_f32 : (float)__dmul_rn(grad, grad);
    } else {
        const double g2 = grad_is_f32 ? (double)grad_sq_f32 : __dmul_rn(grad, grad);
        m = (float)__dadd_rn(__dmul_rn(0.7, (double)m), __dmul_rn(1.0 - 0.7, grad));
        v = (float)__dadd_rn(__dmul_rn(0.9, (double)v), __dmul_rn(1.0 - 0.9, g2));
    }
    // adam_update_params!  l-a.jl:136-146  (ascent)
    const double pm = __ddiv_rn((double)m, m_denom);
    const double pv = __ddiv_rn((double)v, v_denom);
    double delta = __ddiv_rn(__dmul_rn(lr, pm), __dadd_rn(sqrt(pv), 1e-8));
    delta = fmin(fmax(delta, -max_step), max_step);
    param = (float)__dadd_rn((double)param, delta);
}

// One thread per internal node; both halves of the step boundary in one pass over the parameters:
//   UPDATE  (step s):   logit-normal + sinh-arcsinh backward accumulated over the K draws in draw order, /K, finite
//                       check, ADAM ascent with step clamp
//   REPARAM (step s+1): noise -> zs -> ys for the next step's tree forward
// sinh(alpha + asinh z0) is evaluated as z0 cosh(alpha) + sqrt(1 + z0^2) sinh(alpha) (and cosh(c), tanh(c)
// likewise from cosh/sinh(alpha)): the same real function as the reference's Float32 expression with two
// transcendentals per NODE instead of four per DRAW; the difference is a few Float32 ulp.
template <int KP>
__global__ void __launch_bounds__(ELEM_THREADS)
    k3_elem(int64_t nm1, int K, int mode, int do_update, int do_adam, int do_reparam, float *__restrict__ mu,
            float *__restrict__ omega, float *__restrict__ alpha, float *__restrict__ m_mu, float *__restrict__ m_omega,
            float *__restrict__ m_alpha, float *__restrict__ v_mu, float *__restrict__ v_omega, float *__restrict__ v_alpha,
            float *__restrict__ zs0, double *__restrict__ ys, const double *__restrict__ ygrad,
            const StepCtl *__restrict__ ctl, AdamCfg cfg, int *__restrict__ bad_step, float *__restrict__ grad_out,
            const float *__restrict__ noise, int64_t noise_steps, uint64_t seed, int fast_noise, int want_ladj,
            double *__restrict__ ladj_partial /* [2][gridDim.x][KP] */, int step0_fixed, int clamp_y) {
    __shared__ double sm[ELEM_THREADS];
    pdl_trigger();
    pdl_wait();  // everything this kernel reads, the step counters included, is written inside the step loop
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const bool live = i < nm1;
    float p_mu = 0.f, p_om = 0.f, p_al = 0.f;
    if (live) {
        p_mu = mu[i];
        if (mode == 0) { p_om = omega[i]; p_al = alpha[i]; }
    }

    if (do_update && live) {
        const int step = ctl->step_upd;
        // adam_learning_rate(step_num - 1)  l-a.jl:107-110, 497
        const double lr = fmax(1e-3, 1.0 * exp(-2e-2 * (double)(step - 1)));
        const double m_denom = 1.0 - pow(0.7, (double)step), v_denom = 1.0 - pow(0.9, (double)step);
        if (mode == 1) {  // OptimizePTTApprox: z_grad = y (1 - y) y_grad, Float64 (l-a.jl:211-213)
            const double y = ys[(size_t)i * KP];
            const double zg = __dmul_rn(__dmul_rn(y, __dsub_rn(1.0, y)), ygrad[(size_t)i * KP]);
            if (grad_out) grad_out[i] = (float)zg;
            if (!isfinite(zg)) atomicCAS(bad_step, 0, step);
            if (do_adam) {
                float mm = m_mu[i], vv = v_mu[i];
                adam_one(p_mu, mm, vv, zg, 0.0f, false, step, lr, m_denom, v_denom, cfg.max_step_z);
                m_mu[i] = mm; v_mu[i] = vv; mu[i] = p_mu;
            }
        } else {
            const float sigma = expf(p_om);
            const float sa = sinhf(p_al), ca = coshf(p_al);
            const float inv_sigma = __fdiv_rn(1.0f, sigma);
            float mu_g = 0.0f, om_g = 0.0f, al_g = 0.0f;
#pragma unroll 4
            for (int k = 0; k < K; ++k) {
                const double y = ys[(size_t)i * KP + k];
                const double yg = ygrad[(size_t)i * KP + k];  // already rounded to Float32
                const float z0 = zs0[(size_t)i * KP + k];
                const float r = sqrtf(fmaf(z0, z0, 1.0f));     // cosh(asinh z0)
                const float zf = fmaf(z0, ca, r * sa);         // sinh(alpha + asinh z0)
                const float ch = fmaf(ca, r, sa * z0);         // cosh(alpha + asinh z0)
                const double z = (double)zf;
                const double d = __dmul_rn(y, __dsub_rn(1.0, y));
                const double omy2 = __dsub_rn(1.0, __dmul_rn(2.0, y));
                // logit_normal_transform_gradients! (8-arg)  logitnormal.jl:38-55; sigma_grad / z_grad restart per draw
                mu_g = (float)__dadd_rn((double)mu_g, __dmul_rn(d, yg));
                float sg = (float)__dmul_rn(__dmul_rn(d, z), yg);
                float zg = (float)__dmul_rn(__dmul_rn(d, (double)sigma), yg);
                mu_g = (float)__dadd_rn((double)mu_g, omy2);
                sg = (float)__dadd_rn((double)sg, __dadd_rn((double)inv_sigma, __dmul_rn(z, omy2)));
                zg = (float)__dadd_rn((double)zg, __dmul_rn((double)sigma, omy2));
                // sinh_asinh_transform_gradients!  sinh_arcsinh.jl:29-38: cosh(c) z_grad + tanh(c)
                al_g = __fadd_rn(al_g, __fmul_rn(ch, zg));
                al_g = __fadd_rn(al_g, __fdiv_rn(zf, ch));
                // omega chain rule  l-a.jl:547-549
                om_g = __fadd_rn(om_g, __fmul_rn(sigma, sg));
            }
            const float Kf = (float)K;
            mu_g = __fdiv_rn(mu_g, Kf);  // l-a.jl:552-556
            om_g = __fdiv_rn(om_g, Kf);
            al_g = __fdiv_rn(al_g, Kf);
            if (!(isfinite(mu_g) && isfinite(om_g) && isfinite(al_g))) atomicCAS(bad_step, 0, step);
            if (grad_out) {
                grad_out[i] = mu_g;
                grad_out[nm1 + i] = om_g;
                grad_out[2 * nm1 + i] = al_g;
            }
            if (do_adam) {
                float mm = m_mu[i], vv = v_mu[i];
                adam_one(p_mu, mm, vv, (double)mu_g, __fmul_rn(mu_g, mu_g), true, step, lr, m_denom, v_denom, cfg.max_step_mu);
                m_mu[i] = mm; v_mu[i] = vv; mu[i] = p_mu;
                mm = m_omega[i]; vv = v_omega[i];
                adam_one(p_om, mm, vv, (double)om_g, __fmul_rn(om_g, om_g), true, step, lr, m_denom, v_denom, cfg.max_step_omega);
                m_omega[i] = mm; v_omega[i] = vv; omega[i] = p_om;
                mm = m_alpha[i]; vv = v_alpha[i];
                adam_one(p_al, mm, vv, (double)al_g, __fmul_rn(al_g, al_g), true, step, lr, m_denom, v_denom, cfg.max_step_alpha);
                m_alpha[i] = mm; v_alpha[i] = vv; alpha[i] = p_al;
            }
        }
    }

    if (!do_reparam) return;
    double l_skew[KP], l_ln[KP];
#pragma unroll
    for (int k = 0; k < KP; ++k) { l_skew[k] = 0.0; l_ln[k] = 0.0; }
    if (live) {
        if (mode == 1) {
            const float e = expf(-p_mu);
            ys[(size_t)i * KP] = (double)__fdiv_rn(1.0f, __fadd_rn(1.0f, e));  // ys = logistic(zs), no clamp (l-a.jl:196)
            zs0[(size_t)i * KP] = 0.0f;
        } else {
            const int step0 = step0_fixed >= 0 ? step0_fixed : ctl->step_fwd - 1;  // 0-based index of the step of these draws
            const float sigma = expf(p_om);
            const float sa = sinhf(p_al), ca = coshf(p_al);
#pragma unroll
            for (int k = 0; k < KP; ++k) {
                float z0 = 0.0f;
                if (k < K) {
                    if (noise) z0 = noise[((size_t)(step0 % noise_steps) * K + k) * (size_t)nm1 + i];
                    else z0 = philox_normal(seed, (uint32_t)i, (uint32_t)k, (uint32_t)step0, fast_noise);
                }
                const float r = sqrtf(fmaf(z0, z0, 1.0f));
                const float zf = fmaf(z0, ca, r * sa);
                const float xx = __fadd_rn(p_mu, __fmul_rn(zf, sigma));
                const float e = expf(-xx);
                const float y32 = __fdiv_rn(1.0f, __fadd_rn(1.0f, e));
                double y = (double)y32;
                if (want_ladj && k < K) {
                    const float ch = fmaf(ca, r, sa * z0);
                    l_skew[k] = (double)logf(ch) - (double)logf(r);  // log cosh(c) - 0.5 log1p(z0^2)
                    l_ln[k] = log(__dmul_rn(__dmul_rn((double)sigma, y), __dsub_rn(1.0, y)));
                }
                if (clamp_y) y = fmin(fmax(y, 1e-10), 1.0 - 1e-10);
                zs0[(size_t)i * KP + k] = z0;
                ys[(size_t)i * KP + k] = y;
            }
        }
    }
    if (want_ladj) {
        // per-draw block sums, fixed order
        for (int k = 0; k < KP; ++k) {
            sm[threadIdx.x] = l_skew[k];
            __syncthreads();
            for (int span = ELEM_THREADS / 2; span >= 1; span >>= 1) {
                if ((int)threadIdx.x < span) sm[threadIdx.x] += sm[threadIdx.x + span];
                __syncthreads();
            }
            if (threadIdx.x == 0) ladj_partial[(size_t)blockIdx.x * KP + k] = sm[0];
            __syncthreads();
            sm[threadIdx.x] = l_ln[k];
            __syncthreads();
            for (int span = ELEM_THREADS / 2; span >= 1; span >>= 1) {
                if ((int)threadIdx.x < span) sm[threadIdx.x] += sm[threadIdx.x + span];
                __syncthreads();
            }
            if (threadIdx.x == 0) ladj_partial[((size_t)gridDim.x + blockIdx.x) * KP + k] = sm[0];
            __syncthreads();
        }
    }
}

// ELBO of the step being updated: mean over the K draws of lp + the three log-Jacobians
// (the reference ASSIGNS per draw and divides by K, l-a.jl:540,561 -- a quirk; this is the mean).
__global__ void __launch_bounds__(256) k3_elbo(int K, int KP, const double *__restrict__ lp, const double *__restrict__ ladj_partial,
                                               int n_elem_ctas, int n_tree_parts, const StepCtl *__restrict__ ctl,
                                               double *__restrict__ elbo, int max_steps) {
    // one CTA; the partial sums of a draw (two per k3_elem CTA, one per tree CTA: contiguous rows of ladj_partial) are
    // added thread-strided and then by a shared-memory tree: a fixed order
    __shared__ double sm[256];
    const int total = 2 * n_elem_ctas + n_tree_parts;
    double tot = 0.0;
    for (int k = 0; k < K; ++k) {
        double s = 0.0;
        for (int t = threadIdx.x; t < total; t += 256) s += ladj_partial[(size_t)t * KP + k];
        sm[threadIdx.x] = s;
        __syncthreads();
        for (int span = 128; span >= 1; span >>= 1) {
            if ((int)threadIdx.x < span) sm[threadIdx.x] += sm[threadIdx.x + span];
            __syncthreads();
        }
        if (threadIdx.x == 0) tot += (lp ? lp[k] : 0.0) + sm[0];
        __syncthreads();
    }
    const int step = ctl->step_upd;
    if (threadIdx.x == 0 && step >= 1 && step <= max_steps) elbo[step - 1] = tot / (double)K;
}

}  // namespace

// ================================================================== host side
#define CK(expr) POLEE_CUDA_CHECK(h, expr)

void release_work_buffers(polee_handle *h) {
    void *ptrs[] = {h->zs0, h->zs, h->ys, h->ygrad, h->us, h->G, h->root_us, h->root_G, h->x, h->w, h->g, h->seg_partial, h->S_partial,
                    h->S, h->lp_partial, h->ladj_partial, h->grad_out, h->ft_partial, h->ft_lvl2, h->g32,
                    h->ec_partial, h->ec_lvl2, h->ec_lp_partial};
    for (void *p : ptrs) polee::dfree(p);
    h->ft_partial = nullptr; h->ft_lvl2 = nullptr; h->g32 = nullptr;
    h->ec_partial = h->ec_lvl2 = h->ec_lp_partial = nullptr;
    h->zs0 = h->zs = nullptr; h->ys = h->ygrad = h->us = nullptr; h->G = nullptr; h->x = h->w = nullptr; h->root_us = nullptr; h->root_G = nullptr;
    h->g = h->seg_partial = h->S_partial = h->S = h->lp_partial = h->ladj_partial = nullptr;
    h->grad_out = nullptr;
    h->work_KP = 0;
}

int elem_ctas(polee_handle *h, int KP) {
    (void)KP;
    return (int)std::max<int64_t>(1, (h->n - 1 + ELEM_THREADS - 1) / ELEM_THREADS);
}

int ensure_work_buffers(polee_handle *h, int KP) {
    if (h->work_KP == KP) return POLEE_OK;
    release_work_buffers(h);
    const int64_t n = h->n, nm1 = std::max<int64_t>(n - 1, 1), N = 2 * n - 1;
    // rows of the per-CTA partial sums (S_partial and the tree part of ladj_partial): those the route's forward kernels
    // write, or one per warp of k3_leaf_S.  k3_mid, k3_elbo and polee_ptt_transform add them all in a fixed order; the
    // rows a route does not write stay 0
    const TreeDev &td = h->td;
    int rows = 1;  // k3c_chain_fwd: one
    switch (tree_route(td, KP)) {
        case TreeRoute::Chain: break;
        case TreeRoute::DfsRun: rows = td.dfs_ctas; break;
        case TreeRoute::PathProduct: rows = td.n_groups; break;
        case TreeRoute::SmemLevels: rows = 1 + td.s_bottom.nbins; break;  // the top part, then the bottom bins
        case TreeRoute::GlobalLevels: rows = 1 + td.bottom.nbins; break;
    }
    h->n_tree_ctas = std::max(rows, (int)((n + LEAF_S_PER_WARP - 1) / LEAF_S_PER_WARP));
    CK(polee::dmalloc((void **)&h->zs0, sizeof(float) * nm1 * KP));
    CK(polee::dmalloc((void **)&h->zs, sizeof(float) * nm1 * KP));
    CK(polee::dmalloc((void **)&h->ys, sizeof(double) * nm1 * KP));
    CK(polee::dmalloc((void **)&h->ygrad, sizeof(double) * nm1 * KP));
    CK(polee::dmalloc((void **)&h->us, sizeof(double) * N * KP));
    CK(polee::dmalloc((void **)&h->G, sizeof(float2) * N * KP));
    CK(polee::dmalloc((void **)&h->root_us, sizeof(double) * std::max(h->td.n_slots, 1) * KP));
    CK(polee::dmalloc((void **)&h->root_G, sizeof(float2) * std::max(h->td.n_slots, 1) * KP));
    CK(polee::dmalloc((void **)&h->x, sizeof(float) * n * KP));
    CK(polee::dmalloc((void **)&h->g, sizeof(double) * (n + 1) * KP));
    CK(polee::dmalloc((void **)&h->S_partial, sizeof(double) * h->n_tree_ctas * KP));
    CK(polee::dmalloc((void **)&h->S, sizeof(double) * KP));
    CK(polee::dmalloc((void **)&h->ladj_partial, sizeof(double) * (2 * (size_t)elem_ctas(h, KP) + h->n_tree_ctas) * KP));
    CK(polee::dmalloc((void **)&h->grad_out, sizeof(float) * 3 * nm1));
    CK(cudaMemsetAsync(h->S_partial, 0, sizeof(double) * h->n_tree_ctas * KP, h->stream));
    CK(cudaMemsetAsync(h->ladj_partial, 0, sizeof(double) * (2 * (size_t)elem_ctas(h, KP) + h->n_tree_ctas) * KP, h->stream));
    CK(cudaMemsetAsync(h->g, 0, sizeof(double) * (n + 1) * KP, h->stream));
    if (h->nranks > 1) CK(polee::dmalloc((void **)&h->g32, sizeof(float) * (n + 1) * KP));
    if (h->have_matrix) {
        CK(polee::dmalloc((void **)&h->w, sizeof(float) * std::max<int64_t>(h->m_pad, 1) * KP));
        CK(cudaMemsetAsync(h->w, 0, sizeof(float) * std::max<int64_t>(h->m_pad, 1) * KP, h->stream));
        CK(polee::dmalloc((void **)&h->seg_partial, sizeof(double) * std::max(h->n_slots, 1) * KP));
        CK(polee::dmalloc((void **)&h->lp_partial, sizeof(double) * std::max(std::max(h->n_row_tiles, h->ft_tiles), 1) * KP));
        if (h->fused) {
            CK(polee::dmalloc((void **)&h->ft_partial, sizeof(float) * std::max<int64_t>(h->ft_parts, 1) * KP));
            CK(polee::dmalloc((void **)&h->ft_lvl2, sizeof(double) * std::max(h->ft_nlvl2, 1) * KP));
            h->ft_grid = fused_grid(h, KP);
        }
        if (h->ec_tasks > 0) {
            CK(polee::dmalloc((void **)&h->ec_partial, sizeof(double) * std::max<int64_t>(h->ec_parts, 1) * KP));
            CK(polee::dmalloc((void **)&h->ec_lvl2, sizeof(double) * std::max(h->ec_nlvl2, 1) * KP));
            CK(polee::dmalloc((void **)&h->ec_lp_partial, sizeof(double) * (size_t)h->ec_tasks * KP));
            h->ec_grid = ec_grid(h, KP);
        }
    }
    h->work_KP = KP;
    return POLEE_OK;
}

int patch_leaf_records(polee_handle *h) {
    if (!h->have_efflen || !h->have_tree) return POLEE_OK;
    for (SSchedDev *sd : {&h->td.s_top, &h->td.s_bottom}) {
        const int count = (int)(sd == &h->td.s_top ? h->th.s_top.recs.size() : h->th.s_bottom.recs.size());
        if (count > 0)
            k_patch_leaf_recs<<<(count + 255) / 256, 256, 0, h->stream>>>(sd->recs, count, h->efflen, h->efflen_adj);
    }
    CK(cudaGetLastError());
    return POLEE_OK;
}

int launch_elem(polee_handle *h, int KP, int K, bool do_update, bool do_adam, bool do_reparam, const float *noise,
                int64_t noise_steps, int want_ladj, float *grad_out, int step0_fixed, uint64_t seed_override, int clamp_y) {
    const int64_t nm1 = h->n - 1;
    if (nm1 <= 0) return POLEE_OK;
    const int mode = h->o.approx == POLEE_APPROX_OPTIMIZE_PTT ? 1 : 0;
    AdamCfg cfg{h->o.max_step_mu, h->o.max_step_omega, h->o.max_step_alpha, h->o.max_step_z};
    const int ctas = elem_ctas(h, KP);
    DISPATCH_KP(KP, launch_pdl(h, k3_elem<KPC>, ctas, ELEM_THREADS, 0, h->stream,
                        nm1, K, mode, do_update ? 1 : 0, do_adam ? 1 : 0, do_reparam ? 1 : 0, h->mu, h->omega, h->alpha, h->m_mu,
                        h->m_omega, h->m_alpha, h->v_mu, h->v_omega, h->v_alpha, h->zs0, h->ys, h->ygrad, h->d_step, cfg,
                        h->d_bad_step, grad_out, noise, std::max<int64_t>(noise_steps, 1),
                        step0_fixed >= 0 ? seed_override : h->o.seed, 1, want_ladj, h->ladj_partial, step0_fixed, clamp_y));
    return POLEE_OK;
}

int launch_reparam_fwd(polee_handle *h, int KP, int K, const float *noise, int64_t noise_steps, int want_ladj) {
    return launch_elem(h, KP, K, false, false, true, noise, noise_steps, want_ladj, nullptr, -1, 0, 1);
}

constexpr int S_TOP_THREADS = 1024;
// bottom forests: draws per CTA and min CTAs per SM of the TREE_THREADS-thread CTAs (KP = 8: the shape that measured
// fastest, profiles/r02_k3_sweep.log)
constexpr int bottom_kpc(int KP) { return KP == 8 ? 4 : (KP < 8 ? KP : 8); }
constexpr int bottom_minb(int KP) { return KP == 8 ? 3 : 2; }

// dynamic shared memory of k3d_tree_fwd: the walks' stacks, the CTA's y slice and its node records
static size_t dfs_fwd_smem(const TreeDev &td, int KP) {
    const size_t threads = (size_t)DFS_RUNS_PER_CTA * KP;
    return (size_t)(td.max_depth + 2) * threads * 8 + (size_t)((std::max(td.dfs_max_nk, 1) + 1) & ~1) * KP * 8 +
           (size_t)DFS_RUNS_PER_CTA * (DFS_RUN + 2) * sizeof(DNode);
}

// dynamic shared memory of k3p_tree_fwd: y and 1 - y of the group's ancestors by draw, the common prefix, the suffixes
static size_t path_fwd_smem(const TreeDev &td, int KP) {
    return (size_t)td.max_ganc * (16 * KP + 2) + 16 + 2 * (size_t)td.max_gsuf;
}

// The kernels that serve a tree at KP draws: the first route whose condition holds.
//
//   route         condition                                       forward        backward       inverse
//   Chain         caterpillar, N >= chain_min_nodes               k3c_chain_fwd  k3c_chain_bwd  k3_tree_inv_serial
//   DfsRun        bins fit, DFS-run inputs built (pre-order,      k3d_tree_fwd   k3s_tree_bwd   k3_tree_inv
//                 depth <= DFS_MAX_DEPTH), KP <= 16,
//                 dfs_fwd_smem <= 200 KB
//   PathProduct   bins fit, root-path tables built,               k3p_tree_fwd   k3s_tree_bwd   k3_tree_inv
//                 path_fwd_smem <= 200 KB
//   SmemLevels    bins fit                                        k3s_tree_fwd   k3s_tree_bwd   k3_tree_inv
//   GlobalLevels  everything else                                 k3_tree_fwd    k3_tree_bwd    k3_tree_inv
//
// "Bins fit": the largest bottom bin (min(KP, 8) draws) and the top part (one draw) each fit in 200 KB of shared memory
// with the records, u, y and G the shared-memory kernels hold per node.  The forward kernels of the three routes that
// share k3s_tree_bwd all leave u of every internal node by k in h->us, where it reads it; the chain and global-level
// kernels keep u by node there.
TreeRoute tree_route(const TreeDev &td, int KP) {
    if (td.caterpillar && td.N >= td.chain_min_nodes) return TreeRoute::Chain;
    const size_t limit = 200 * 1024;
    const int KPC = KP < 8 ? KP : 8;
    const bool bins_fit =
        (size_t)td.s_bottom.max_bin_nodes * (sizeof(SNode) + 24 * KPC) + 4 * (td.s_bottom.max_bin_levels + 2) <= limit &&
        (size_t)td.s_top.max_bin_nodes * (sizeof(SNode) + 24) + 4 * (td.s_top.max_bin_levels + 2) <= limit;
    if (!bins_fit) return TreeRoute::GlobalLevels;
    if (td.dnodes && KP <= 16 && dfs_fwd_smem(td, KP) <= limit) return TreeRoute::DfsRun;
    if (td.ganc_ptr && path_fwd_smem(td, KP) <= limit) return TreeRoute::PathProduct;
    return TreeRoute::SmemLevels;
}

template <int KP>
static int launch_tree_fwd_smem(polee_handle *h, int clamp_x, const float *eff, double *Sp, int want_ladj, double *ladj_tree) {
    const TreeDev &td = h->td;
    if (td.s_top.nbins > 0) {
        const size_t smem = (size_t)td.s_top.max_bin_nodes * (sizeof(SNode) + 16) + 4 * (td.s_top.max_bin_levels + 2);
        auto fn = k3s_tree_fwd<KP, 1, S_TOP_THREADS, 1>;
        allow_max_smem(fn);  // per-function, process-wide: see common.cuh
        fn<<<dim3(td.s_top.nbins, KP), S_TOP_THREADS, smem, h->stream>>>(
            td.s_top.bin_off, td.s_top.bin_lvl_ptr, td.s_top.lvl_off, td.s_top.recs, h->ys, h->root_us, h->us, h->x,
            clamp_x, eff, Sp, 0, want_ladj, ladj_tree);
    }
    if (td.s_bottom.nbins > 0) {
        constexpr int KPC = bottom_kpc(KP);
        const size_t smem = (size_t)td.s_bottom.max_bin_nodes * (sizeof(SNode) + 16 * KPC) + 4 * (td.s_bottom.max_bin_levels + 2);
        auto fn = k3s_tree_fwd<KP, KPC, TREE_THREADS, bottom_minb(KP)>;
        allow_max_smem(fn);
        fn<<<dim3(td.s_bottom.nbins, KP / KPC), TREE_THREADS, smem, h->stream>>>(
            td.s_bottom.bin_off, td.s_bottom.bin_lvl_ptr, td.s_bottom.lvl_off, td.s_bottom.recs, h->ys, h->root_us, h->us,
            h->x, clamp_x, eff, Sp, 1, want_ladj, ladj_tree);
    }
    return POLEE_OK;
}

template <int KP, bool WITH_LADJ>
static int launch_tree_bwd_smem(polee_handle *h, const float *adj, double *xgrad_out) {
    const TreeDev &td = h->td;
    if (td.s_bottom.nbins > 0) {
        constexpr int KPC = bottom_kpc(KP);
        const size_t smem = (size_t)td.s_bottom.max_bin_nodes * (sizeof(SNode) + 24 * KPC) + 4 * (td.s_bottom.max_bin_levels + 2);
        auto fn = k3s_tree_bwd<KP, KPC, TREE_THREADS, bottom_minb(KP), WITH_LADJ>;
        allow_max_smem(fn);
        launch_pdl(h, fn, dim3(td.s_bottom.nbins, KP / KPC), TREE_THREADS, smem, h->stream, td.s_bottom.bin_off,
                   td.s_bottom.bin_lvl_ptr, td.s_bottom.lvl_off, td.s_bottom.recs, h->ys, h->us, h->root_G, h->g, adj, h->S,
                   h->ygrad, xgrad_out);
    }
    if (td.s_top.nbins > 0) {
        const size_t smem = (size_t)td.s_top.max_bin_nodes * (sizeof(SNode) + 24) + 4 * (td.s_top.max_bin_levels + 2);
        auto fn = k3s_tree_bwd<KP, 1, S_TOP_THREADS, 1, WITH_LADJ>;
        allow_max_smem(fn);
        launch_pdl(h, fn, dim3(td.s_top.nbins, KP), S_TOP_THREADS, smem, h->stream, td.s_top.bin_off, td.s_top.bin_lvl_ptr,
                   td.s_top.lvl_off, td.s_top.recs, h->ys, h->us, h->root_G, h->g, adj, h->S, h->ygrad, xgrad_out);
    }
    return POLEE_OK;
}

int launch_tree_fwd(polee_handle *h, int KP, int clamp_x, int want_S, int want_ladj) {
    const TreeDev &td = h->td;
    double *ladj_tree = h->ladj_partial + (size_t)2 * elem_ctas(h, KP) * KP;
    const float *eff = want_S ? h->efflen : nullptr;
    double *Sp = want_S ? h->S_partial : nullptr;
    int rc = POLEE_OK;
    switch (tree_route(td, KP)) {
        case TreeRoute::Chain:
            return launch_chain_fwd(h, KP, clamp_x, eff, Sp, want_ladj, ladj_tree);
        case TreeRoute::DfsRun: {
            const size_t smem = dfs_fwd_smem(td, KP);
            if (smem > 40 * 1024) DISPATCH_KP(KP, allow_max_smem(k3d_tree_fwd<KPC>));
            DISPATCH_KP(KP, launch_pdl(h, k3d_tree_fwd<KPC>, td.dfs_ctas, DFS_RUNS_PER_CTA * KPC, smem, h->stream, td.N,
                                       td.dnodes, td.drun_anc_ptr, td.drun_anc, td.dcta_k0, h->ys, h->us, h->x, clamp_x,
                                       want_ladj, ladj_tree, td.max_depth + 2, (std::max(td.dfs_max_nk, 1) + 1) & ~1));
            h->S_deferred = want_S != 0;  // launch_mid adds S = sum_j x_j / efflen_j (k3_leaf_S) beside the likelihood pass
            break;
        }
        case TreeRoute::PathProduct: {
            const size_t smem = path_fwd_smem(td, KP);
            if (smem > 40 * 1024) DISPATCH_KP(KP, allow_max_smem(k3p_tree_fwd<KPC>));
            DISPATCH_KP(KP, (k3p_tree_fwd<KPC><<<td.n_groups, PATH_SLOTS * KPC, smem, h->stream>>>(
                                td.N, td.nodes, td.ganc_ptr, td.ganc, td.gcp, td.nsuf_ptr, td.nsuf, h->ys, h->us, h->x, clamp_x,
                                eff, Sp, want_ladj, ladj_tree)));
            break;
        }
        case TreeRoute::SmemLevels:
            DISPATCH_KP(KP, rc = launch_tree_fwd_smem<KPC>(h, clamp_x, eff, Sp, want_ladj, ladj_tree));
            break;
        case TreeRoute::GlobalLevels:
            if (td.top.nbins > 0) {
                DISPATCH_KP(KP, (k3_tree_fwd<KPC, TOP_THREADS><<<td.top.nbins, TOP_THREADS, 0, h->stream>>>(
                                    td.top.bin_lvl_ptr, td.top.lvl_off, td.top.sch_node, td.nodes, h->ys, h->us, h->x, clamp_x,
                                    eff, Sp, 0, want_ladj, ladj_tree)));
            }
            if (td.bottom.nbins > 0) {
                DISPATCH_KP(KP, (k3_tree_fwd<KPC, TREE_THREADS><<<td.bottom.nbins, TREE_THREADS, 0, h->stream>>>(
                                    td.bottom.bin_lvl_ptr, td.bottom.lvl_off, td.bottom.sch_node, td.nodes, h->ys, h->us, h->x,
                                    clamp_x, eff, Sp, 1, want_ladj, ladj_tree)));
            }
            break;
    }
    return rc;
}

int launch_mid(polee_handle *h, int KP, int advance, cudaStream_t st) {
    if (h->S_deferred) {  // S and the bookkeeping in one small kernel (k3_leaf_S)
        h->S_deferred = false;
        const int nwarps = (int)((h->n + LEAF_S_PER_WARP - 1) / LEAF_S_PER_WARP);
        if (nwarps > h->n_tree_ctas) return h->fail(POLEE_EINVAL, "internal: S partial buffer too small");
        const int ctas = (nwarps * 32 + LEAF_S_THREADS - 1) / LEAF_S_THREADS;
        DISPATCH_KP(KP, (k3_leaf_S<KPC><<<ctas, LEAF_S_THREADS, 0, st ? st : h->stream>>>(
                            h->n, h->x, h->efflen, h->S_partial, nwarps, h->S, h->d_step, advance, h->d_leafS_counter)));
        return POLEE_OK;
    }
    k3_mid<<<1, 1024, 0, st ? st : h->stream>>>(h->S_partial, h->n_tree_ctas, KP, h->S, h->d_step, advance);
    return POLEE_OK;
}

int launch_tree_bwd(polee_handle *h, int KP, bool with_ladj, bool apply_efflen, double *xgrad_out) {
    const TreeDev &td = h->td;
    const float *adj = apply_efflen ? h->efflen_adj : nullptr;
    int rc = POLEE_OK;
#define BWD(SCHED, THREADS)                                                                                          \
    if (with_ladj) {                                                                                                 \
        DISPATCH_KP(KP, (k3_tree_bwd<KPC, THREADS, true><<<SCHED.nbins, THREADS, 0, h->stream>>>(                    \
                            SCHED.bin_lvl_ptr, SCHED.lvl_off, SCHED.sch_node, td.nodes, h->ys, h->us, h->g, adj, h->S, \
                            h->G, h->ygrad, xgrad_out)));                                                            \
    } else {                                                                                                         \
        DISPATCH_KP(KP, (k3_tree_bwd<KPC, THREADS, false><<<SCHED.nbins, THREADS, 0, h->stream>>>(                   \
                            SCHED.bin_lvl_ptr, SCHED.lvl_off, SCHED.sch_node, td.nodes, h->ys, h->us, h->g, adj, h->S, \
                            h->G, h->ygrad, xgrad_out)));                                                            \
    }
    switch (tree_route(td, KP)) {
        case TreeRoute::Chain:
            return launch_chain_bwd(h, KP, with_ladj, adj, xgrad_out);
        case TreeRoute::DfsRun:
        case TreeRoute::PathProduct:
        case TreeRoute::SmemLevels:
            if (with_ladj) {
                DISPATCH_KP(KP, (rc = launch_tree_bwd_smem<KPC, true>(h, adj, xgrad_out)));
            } else {
                DISPATCH_KP(KP, (rc = launch_tree_bwd_smem<KPC, false>(h, adj, xgrad_out)));
            }
            break;
        case TreeRoute::GlobalLevels:
            if (td.bottom.nbins > 0) { BWD(td.bottom, TREE_THREADS) }
            if (td.top.nbins > 0) { BWD(td.top, TOP_THREADS) }
            break;
    }
#undef BWD
    return rc;
}

// Under CUDA's lazy module loading a kernel's code is loaded at its first launch (a few hundred microseconds to
// milliseconds each, the device idle meanwhile).  polee_set_sample calls this from a helper thread while the matrix is on
// its way to the device, so that the first ADAM step finds the kernels of the default step (balanced trees in
// pre-order, logit-skew-normal fit) resident.  Asking for a kernel's attributes loads it; nothing else happens here.
template <int KP>
static void preload_tree_kernels_kp() {
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, k3_elem<KP>);
    cudaFuncGetAttributes(&a, k3d_tree_fwd<KP>);
    cudaFuncGetAttributes(&a, k3_leaf_S<KP>);
    cudaFuncGetAttributes(&a, k3s_tree_bwd<KP, bottom_kpc(KP), TREE_THREADS, bottom_minb(KP), true>);
    cudaFuncGetAttributes(&a, k3s_tree_bwd<KP, 1, S_TOP_THREADS, 1, true>);
    cudaGetLastError();
}
void preload_tree_kernels(int KP) {
    switch (KP) {
        case 1: preload_tree_kernels_kp<1>(); break;
        case 2: preload_tree_kernels_kp<2>(); break;
        case 4: preload_tree_kernels_kp<4>(); break;
        case 8: preload_tree_kernels_kp<8>(); break;
        case 16: preload_tree_kernels_kp<16>(); break;
        default: break;
    }
}

int launch_update(polee_handle *h, int KP, int K, bool do_adam, float *grad_out) {
    return launch_elem(h, KP, K, true, do_adam, false, nullptr, 1, 0, grad_out, -1, 0, 1);
}

int launch_elbo(polee_handle *h, int KP, int K, bool have_lp) {
    k3_elbo<<<1, 256, 0, h->stream>>>(K, KP, have_lp ? h->g + (size_t)h->n * KP : nullptr, h->ladj_partial,
                                     elem_ctas(h, KP), h->n_tree_ctas, h->d_step, h->elbo,
                                     h->o.num_steps);
    return POLEE_OK;
}


// inverse_transform! of the KP draws in x_dev ([n][KP] Float32) -> ys_out ([n-1][KP] Float64) and, when ladj_out is
// given, ladj[KP].  us_tmp: [2n-1][KP] Float64 scratch (indexed by node); logu_tmp: [n-1][KP] Float32 scratch (needed
// only with ladj_out).
int launch_tree_inv(polee_handle *h, int KP, const float *x_dev, double *us_tmp, double *ys_out, float *logu_tmp, double *ladj_out) {
    const TreeDev &td = h->td;
    float *logu = ladj_out ? logu_tmp : nullptr;
    if (td.n < 2) return POLEE_OK;
    if (tree_route(td, KP) == TreeRoute::Chain) {
        k3_tree_inv_serial<<<1, 32, 0, h->stream>>>(td.N, KP, td.nodes, x_dev, us_tmp, ys_out, logu);
    } else {
        if (td.bottom.nbins > 0) {
            DISPATCH_KP(KP, (k3_tree_inv<KPC, TREE_THREADS><<<td.bottom.nbins, TREE_THREADS, 0, h->stream>>>(
                                td.bottom.bin_lvl_ptr, td.bottom.lvl_off, td.bottom.sch_node, td.nodes, x_dev, us_tmp, ys_out, logu)));
        }
        if (td.top.nbins > 0) {
            DISPATCH_KP(KP, (k3_tree_inv<KPC, TOP_THREADS><<<td.top.nbins, TOP_THREADS, 0, h->stream>>>(
                                td.top.bin_lvl_ptr, td.top.lvl_off, td.top.sch_node, td.nodes, x_dev, us_tmp, ys_out, logu)));
        }
    }
    if (ladj_out) k3_inv_ladj<<<1, 32, 0, h->stream>>>(td.n - 1, KP, logu, ladj_out);
    return POLEE_OK;
}

int launch_fill_f32(polee_handle *h, float *p, int64_t count, float v) {
    if (count > 0) k3_fill_f32<<<(unsigned)((count + 255) / 256), 256, 0, h->stream>>>(p, count, v);
    return POLEE_OK;
}

// the starting point of the fit (likelihood-approximation.jl:451-456) from ys0 = inverse_transform!(fill(1f0/n)) when
// given (it also fills mu0), else from the stored mu0
int launch_init_params(polee_handle *h, const double *ys0, int KP) {
    const int64_t nm1 = h->td.n - 1;
    if (nm1 < 1) return POLEE_OK;
    k3_init_params<<<(unsigned)((nm1 + 255) / 256), 256, 0, h->stream>>>(nm1, KP, ys0, logf(0.1f), h->mu0_dev, h->mu, h->omega, h->alpha);
    return POLEE_OK;
}

}  // namespace polee
