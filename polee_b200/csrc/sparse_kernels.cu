// sparse_kernels.cu -- the two HBM-bound sparse passes of one ADAM step, for KP (= K padded to a
// power of two) Monte-Carlo draws at once, so the matrix is streamed once per step instead of once
// per draw as in the reference.
//
//  K1  fragment likelihood   p[i][k] = sum_j X[i][j] * x[j][k]       pAt_mul_B!(frag_probs, Xt, xs)
//      fused with w = 1/p (or ks/p) and, optionally, sum_i log p      src/sparse.jl:6-21, likelihood.jl:21-25,46-51,78-80
//  K2  transposed gradient   g[j][k] = sum_i X[i][j] * w[i][k]       pAt_mulinv_B!(x_grad, X, frag_probs)
//      deterministic: no atomics, fixed reduction trees              src/sparse.jl:25-40
//
// Arithmetic contract (SURVEY App. A steps 5-7), two modes selected by opts.exact_accumulation:
//   exact (1): each product x*v is rounded to Float32 and summed in Float64 in ascending-transcript order,
//              exactly as the reference does -> p is bit-identical to the reference's frag_probs; g is a
//              Float64 FMA per entry.  (v1 K1 kernel: direct global loads.)
//   fast  (0, default): K1 sums a row's products in Float32 batches of four (rows of <= 4 entries entirely in
//              Float32, one MUFU.RCP per draw) and the batches in Float64; K2 accumulates a lane's <= 8 products of a
//              segment in Float32 and everything above that in Float64.  Both stay <= 3e-7 relative of the oracle,
//              30x inside the 1e-5 gate.
// w is stored as Float32 (one rounding, <= 2^-24 relative).  Deterministic either way: no atomics, fixed
// reduction trees.  Tensor cores are not used: nothing here is a dense contraction.
#include <algorithm>
#include <cstdlib>

#include "common.cuh"
#include "device_utils.cuh"

namespace polee {

namespace {


// ---------------------------------------------------------------- K1
// One thread = one row (fragment) of one row-length class; KP Float64 accumulators in registers.
template <int KP, bool LP, bool WEIGHTED>
__global__ void __launch_bounds__(ROW_TILE)
    k1_sell_fwd(const RowTile *__restrict__ tiles, const uint32_t *__restrict__ idx, const float *__restrict__ val,
                const float *__restrict__ x, float *__restrict__ w, const float *__restrict__ row_weight,
                double *__restrict__ lp_partial) {
    const RowTile t = tiles[blockIdx.x];
    const uint32_t r = threadIdx.x;
    double lpv[KP];
#pragma unroll
    for (int k = 0; k < KP; ++k) lpv[k] = 0.0;

    if (r < t.nrows) {
        const uint32_t *ip = idx + t.slab_off + r;
        const float *vp = val + t.slab_off + r;
        const size_t stride = t.stride;
        const uint32_t L = t.len;
        double acc[KP];
#pragma unroll
        for (int k = 0; k < KP; ++k) acc[k] = 0.0;
        uint32_t tt = 0;
        constexpr int U = (KP >= 16) ? 2 : 4;
        for (; tt + U <= L; tt += U) {
            uint32_t c[U];
            float v[U];
            float xv[U][KP];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                c[u] = ld_stream_u32(ip + (size_t)(tt + u) * stride);
                v[u] = ld_stream_f32(vp + (size_t)(tt + u) * stride);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) Vec<KP>::ld(x + (size_t)c[u] * KP, xv[u]);
#pragma unroll
            for (int u = 0; u < U; ++u)
#pragma unroll
                for (int k = 0; k < KP; ++k) acc[k] = __dadd_rn(acc[k], (double)__fmul_rn(xv[u][k], v[u]));
        }
        for (; tt < L; ++tt) {
            uint32_t c = ld_stream_u32(ip + (size_t)tt * stride);
            float v = ld_stream_f32(vp + (size_t)tt * stride);
            float xv[KP];
            Vec<KP>::ld(x + (size_t)c * KP, xv);
#pragma unroll
            for (int k = 0; k < KP; ++k) acc[k] = __dadd_rn(acc[k], (double)__fmul_rn(xv[k], v));
        }
        float wt = 1.0f;
        if (WEIGHTED) wt = row_weight[t.row0 + r];
        float wv[KP];
#pragma unroll
        for (int k = 0; k < KP; ++k) {
            float rc = __frcp_rn((float)acc[k]);
            wv[k] = WEIGHTED ? rc * wt : rc;
        }
        Vec<KP>::st(w + (size_t)(t.row0 + r) * KP, wv);
        if (LP) {
#pragma unroll
            for (int k = 0; k < KP; ++k) lpv[k] = WEIGHTED ? log(acc[k]) * (double)wt : log(acc[k]);
        }
    }
    if (LP) {
        // fixed-order block reduction: shuffle tree inside each warp, then warp 0 adds the 8 warp sums
        __shared__ double sm[ROW_TILE / 32][KP];
#pragma unroll
        for (int k = 0; k < KP; ++k) {
            double v = lpv[k];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5][k] = v;
        }
        __syncthreads();
        if (threadIdx.x < KP) {
            double s = 0.0;
            for (int wi = 0; wi < ROW_TILE / 32; ++wi) s += sm[wi][threadIdx.x];
            lp_partial[(size_t)blockIdx.x * KP + threadIdx.x] = s;
        }
    }
}

// ---------------------------------------------------------------- K2
// Fixed butterfly: after it, the lane holds in acc[0] the warp total of draw k = draw_of_lane<KP>(lane).
template <int KP>
__device__ __forceinline__ void warp_reduce_scatter(double (&acc)[KP], int lane) {
    int mask = 16;
#pragma unroll
    for (int half = KP / 2; half >= 1; half >>= 1, mask >>= 1) {
        const bool up = (lane & mask) != 0;
#pragma unroll
        for (int i = 0; i < half; ++i) {
            double keep = up ? acc[i + half] : acc[i];
            double send = up ? acc[i] : acc[i + half];
            acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, mask);
        }
    }
    for (; mask >= 1; mask >>= 1) acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], mask);
}
template <int KP>
__device__ __forceinline__ int draw_of_lane(int lane) {
    // bits consumed from the top: lane bit 4 is the most significant bit of k
    int k = 0, mask = 16;
    for (int half = KP / 2; half >= 1; half >>= 1, mask >>= 1) k = (k << 1) | ((lane & mask) ? 1 : 0);
    return k;
}
template <int KP>
__device__ __forceinline__ bool lane_writes(int lane) {
    // one writer per draw: the lanes whose unconsumed low bits are zero
    int consumed = 0;
    for (int half = KP / 2; half >= 1; half >>= 1) ++consumed;
    int low_mask = (1 << (5 - consumed)) - 1;
    return (lane & low_mask) == 0;
}

constexpr int K2_WARPS = 8;

// single CTA, fixed order: out[k] = sum_t partial[t][k]
__global__ void __launch_bounds__(1024) k_reduce_partials(const double *__restrict__ partial, int count, int KP,
                                                          double *__restrict__ out) {
    __shared__ double sm[1024];
    const int k = threadIdx.x % KP, lane_t = threadIdx.x / KP, per = 1024 / KP;
    double s = 0.0;
    for (int t = lane_t; t < count; t += per) s += partial[(size_t)t * KP + k];
    sm[threadIdx.x] = s;
    __syncthreads();
    for (int span = per / 2; span >= 1; span >>= 1) {
        if (lane_t < span) sm[threadIdx.x] += sm[threadIdx.x + span * KP];
        __syncthreads();
    }
    if (threadIdx.x < KP) out[threadIdx.x] = sm[threadIdx.x];
}


// =====================================================================================================
// v2 kernels: warp-specialised, TMA-fed.  One producer warp streams the matrix tiles into a shared-memory
// ring with 1-D bulk async copies (cp.async.bulk -> SASS UBLKCP) completing on mbarriers; eight consumer
// warps do the gathers and the arithmetic.  The stream never touches registers or L1, tens of KB per SM
// are in flight without any occupancy cost, and the only latency left on a consumer's critical path is
// the gather itself.
// =====================================================================================================

// one short row (L <= 4 entries, the common case): everything in Float32 -- L gathers in flight, L FFMAs per draw,
// one MUFU reciprocal per draw; no Float64 and no conversions at all
template <int KP, int L, bool WEIGHTED>
__device__ __forceinline__ void k1_short_row(const uint32_t (*sidx)[ROW_TILE], const float (*sval)[ROW_TILE], uint32_t r,
                                             const float *__restrict__ xf, float *__restrict__ wout, float wt,
                                             float *pout) {
    float xv[L][KP], v[L];
    const char *xb = reinterpret_cast<const char *>(xf);
#pragma unroll
    for (int u = 0; u < L; ++u) {
        const uint32_t c = sidx[u][r];
        v[u] = sval[u][r];
        Vec<KP>::ld(reinterpret_cast<const float *>(xb + (size_t)c * (KP * 4)), xv[u]);
    }
    float facc[KP];
#pragma unroll
    for (int k = 0; k < KP; ++k) facc[k] = v[0] * xv[0][k];
#pragma unroll
    for (int u = 1; u < L; ++u)
#pragma unroll
        for (int k = 0; k < KP; ++k) facc[k] = fmaf(v[u], xv[u][k], facc[k]);
#pragma unroll
    for (int k = 0; k < KP; ++k) {
        if (pout) pout[k] = facc[k];
        const float rc = rcp_approx(facc[k]);
        facc[k] = WEIGHTED ? rc * wt : rc;
    }
    Vec<KP>::st(wout, facc);
}

constexpr int V2_CONSUMER_WARPS = 8;
constexpr int V2_THREADS = (V2_CONSUMER_WARPS + 1) * 32;
constexpr int K1_TC = 8;      // entries of a row per ring stage
constexpr int K1_STAGES = 3;

struct K1Smem {
    uint32_t idx[K1_STAGES][K1_TC][ROW_TILE];
    float val[K1_STAGES][K1_TC][ROW_TILE];
    double lpsm[V2_CONSUMER_WARPS][16];
    uint64_t full[K1_STAGES], empty[K1_STAGES];
};

// K1 v2.  Rows of <= 4 entries: k1_short_row, all Float32.  Longer rows: batches of <= 4 products summed in Float32,
// each batch widened once and added to a Float64 row sum.
// (EXACT builds keep the v1 kernel, whose products are rounded to Float32 first as in the reference.)
template <int KP, bool LP, bool WEIGHTED>
__global__ void __launch_bounds__(V2_THREADS, 3)
    k1_sell_fwd_tma(const RowTile *__restrict__ tiles, int n_tiles, const uint32_t *__restrict__ idx,
                    const float *__restrict__ val, const float *__restrict__ xf, float *__restrict__ w,
                    const float *__restrict__ row_weight, double *__restrict__ lp_partial) {
    extern __shared__ __align__(128) unsigned char smraw[];
    K1Smem &sm = *reinterpret_cast<K1Smem *>(smraw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < K1_STAGES; ++s) {
            mbar_init(&sm.full[s], 1);
            mbar_init(&sm.empty[s], V2_CONSUMER_WARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp == V2_CONSUMER_WARPS) {
        // ------------------------------ producer warp (one lane)
        if (lane == 0) {
            int item = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                const RowTile t = tiles[tile];
                const uint32_t bytes_row = ((t.nrows + 31u) & ~31u) * 4u;
                for (uint32_t t0 = 0; t0 < t.len; t0 += K1_TC, ++item) {
                    const int stage = item % K1_STAGES;
                    mbar_wait(&sm.empty[stage], ((item / K1_STAGES) & 1) ^ 1);
                    const uint32_t tc = min((uint32_t)K1_TC, t.len - t0);
                    mbar_expect_tx(&sm.full[stage], tc * 2u * bytes_row);
                    for (uint32_t tt = 0; tt < tc; ++tt) {
                        const size_t off = t.slab_off + (size_t)(t0 + tt) * t.stride;
                        bulk_g2s(&sm.idx[stage][tt][0], idx + off, bytes_row, &sm.full[stage]);
                        bulk_g2s(&sm.val[stage][tt][0], val + off, bytes_row, &sm.full[stage]);
                    }
                }
            }
        }
        return;
    }

    // ------------------------------ consumer warps: thread = one row of the tile
    const uint32_t r = threadIdx.x;  // 0..255
    int item = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const RowTile t = tiles[tile];
        const bool active = r < t.nrows;
        if (t.len <= 4) {  // warp-uniform: the whole tile is one ring item
            const int stage = item % K1_STAGES;
            mbar_wait(&sm.full[stage], (item / K1_STAGES) & 1);
            float pv[KP];
#pragma unroll
            for (int k = 0; k < KP; ++k) pv[k] = 1.0f;
            float wt = 1.0f;
            if (active) {
                if (WEIGHTED) wt = row_weight[t.row0 + r];
                float *wout = w + (size_t)(t.row0 + r) * KP;
                float *pp = LP ? pv : nullptr;
                switch (t.len) {
                    case 1: k1_short_row<KP, 1, WEIGHTED>(sm.idx[stage], sm.val[stage], r, xf, wout, wt, pp); break;
                    case 2: k1_short_row<KP, 2, WEIGHTED>(sm.idx[stage], sm.val[stage], r, xf, wout, wt, pp); break;
                    case 3: k1_short_row<KP, 3, WEIGHTED>(sm.idx[stage], sm.val[stage], r, xf, wout, wt, pp); break;
                    default: k1_short_row<KP, 4, WEIGHTED>(sm.idx[stage], sm.val[stage], r, xf, wout, wt, pp); break;
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&sm.empty[stage]);
            ++item;
            if constexpr (LP) {
#pragma unroll
                for (int k = 0; k < KP; ++k) {
                    double v = active ? (WEIGHTED ? log((double)pv[k]) * (double)wt : log((double)pv[k])) : 0.0;
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                    if (lane == 0) sm.lpsm[warp][k] = v;
                }
                consumer_bar_sync();
                if (threadIdx.x < KP) {
                    double sacc = 0.0;
                    for (int wi = 0; wi < V2_CONSUMER_WARPS; ++wi) sacc += sm.lpsm[wi][threadIdx.x];
                    lp_partial[(size_t)tile * KP + threadIdx.x] = sacc;
                }
                consumer_bar_sync();
            }
            continue;
        }
        double acc[KP];
#pragma unroll
        for (int k = 0; k < KP; ++k) acc[k] = 0.0;
        for (uint32_t t0 = 0; t0 < t.len; t0 += K1_TC, ++item) {
            const int stage = item % K1_STAGES;
            mbar_wait(&sm.full[stage], (item / K1_STAGES) & 1);
            const uint32_t tc = min((uint32_t)K1_TC, t.len - t0);
            if (active) {
                constexpr int U = 4;
                for (uint32_t tt = 0; tt < tc; tt += U) {
                    float xv[U][KP];
                    float v[U];
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const bool ok = tt + u < tc;
                        const uint32_t c = ok ? sm.idx[stage][tt + u][r] : 0u;
                        v[u] = ok ? sm.val[stage][tt + u][r] : 0.0f;
                        Vec<KP>::ld(xf + (size_t)c * KP, xv[u]);
                    }
                    float facc[KP];
#pragma unroll
                    for (int k = 0; k < KP; ++k) facc[k] = v[0] * xv[0][k];
#pragma unroll
                    for (int u = 1; u < U; ++u)
#pragma unroll
                        for (int k = 0; k < KP; ++k) facc[k] = fmaf(v[u], xv[u][k], facc[k]);
#pragma unroll
                    for (int k = 0; k < KP; ++k) acc[k] += (double)facc[k];
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&sm.empty[stage]);
        }
        double lpv[KP];
#pragma unroll
        for (int k = 0; k < KP; ++k) lpv[k] = 0.0;
        if (active) {
            float wt = 1.0f;
            if (WEIGHTED) wt = row_weight[t.row0 + r];
            float wv[KP];
#pragma unroll
            for (int k = 0; k < KP; ++k) {
                float rc = __frcp_rn((float)acc[k]);
                wv[k] = WEIGHTED ? rc * wt : rc;
            }
            Vec<KP>::st(w + (size_t)(t.row0 + r) * KP, wv);
            if (LP) {
#pragma unroll
                for (int k = 0; k < KP; ++k) lpv[k] = WEIGHTED ? log(acc[k]) * (double)wt : log(acc[k]);
            }
        }
        if (LP) {
#pragma unroll
            for (int k = 0; k < KP; ++k) {
                double v = lpv[k];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                if (lane == 0) sm.lpsm[warp][k] = v;
            }
            consumer_bar_sync();
            if (threadIdx.x < KP) {
                double s = 0.0;
                for (int wi = 0; wi < V2_CONSUMER_WARPS; ++wi) s += sm.lpsm[wi][threadIdx.x];
                lp_partial[(size_t)tile * KP + threadIdx.x] = s;
            }
            consumer_bar_sync();
        }
    }
}

// ---------------------------------------------------------------- K2 v2
constexpr int K2_STAGES = 2;
constexpr int K2_ITEM_ENTRIES = K2_WARPS * COL_SEG;  // 2048

constexpr int K2_PART_BUFS = 2 * K2_STAGES;  // consumers can run at most K2_STAGES items ahead of a combine
struct K2Smem {
    uint32_t row[K2_STAGES][K2_ITEM_ENTRIES + 8];
    float val[K2_STAGES][K2_ITEM_ENTRIES + 8];
    ColSeg seg[K2_STAGES][K2_WARPS];  // the item's segment descriptors travel through the ring too
    double part[K2_PART_BUFS][K2_WARPS][16];
    uint64_t full[K2_STAGES], empty[K2_STAGES], part_full[K2_PART_BUFS];
};

// One item = K2_WARPS consecutive segments = one contiguous range of CSC entries.  Consumer warp wi owns
// segment wi of the item.  FAST: the lane's <= COL_SEG/32 products are accumulated in Float32, then widened
// and reduced in Float64 (lane -> warp butterfly -> segments of a column inside the CTA -> k2_combine);
// EXACT: every product is a Float64 FMA.  Fixed order everywhere: deterministic, no atomics.
template <int KP, bool EXACT>
__global__ void __launch_bounds__(V2_THREADS, 3)
    k2_csc_grad_tma(const ColSeg *__restrict__ segs, int n_segs, const uint32_t *__restrict__ csc_row,
                    const float *__restrict__ csc_val, const float *__restrict__ w, double *__restrict__ g,
                    double *__restrict__ seg_partial) {
    extern __shared__ __align__(128) unsigned char smraw[];
    K2Smem &sm = *reinterpret_cast<K2Smem *>(smraw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < K2_STAGES; ++s) {
            mbar_init(&sm.full[s], 1);
            mbar_init(&sm.empty[s], K2_WARPS);
        }
        for (int s = 0; s < K2_PART_BUFS; ++s) mbar_init(&sm.part_full[s], K2_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int n_items = (n_segs + K2_WARPS - 1) / K2_WARPS;

    if (warp == K2_WARPS) {
        // ------------------------------ producer warp (one lane)
        if (lane == 0) {
            int j = 0;
            for (int it = blockIdx.x; it < n_items; it += gridDim.x, ++j) {
                const int stage = j % K2_STAGES;
                const ColSeg first = segs[it * K2_WARPS];
                const ColSeg last = segs[min(it * K2_WARPS + K2_WARPS - 1, n_segs - 1)];
                const uint32_t a0 = first.start & ~3u;
                const uint32_t cnt = last.start + (last.len & 0xffffu) - a0;
                const uint32_t bytes = (cnt * 4u + 15u) & ~15u;
                const uint32_t nseg = (uint32_t)min(K2_WARPS, n_segs - it * K2_WARPS);
                mbar_wait(&sm.empty[stage], ((j / K2_STAGES) & 1) ^ 1);
                mbar_expect_tx(&sm.full[stage], 2u * bytes + nseg * (uint32_t)sizeof(ColSeg));
                bulk_g2s(&sm.seg[stage][0], segs + (size_t)it * K2_WARPS, nseg * (uint32_t)sizeof(ColSeg), &sm.full[stage]);
                if (bytes) {
                    bulk_g2s(&sm.row[stage][0], csc_row + a0, bytes, &sm.full[stage]);
                    bulk_g2s(&sm.val[stage][0], csc_val + a0, bytes, &sm.full[stage]);
                }
            }
        }
        return;
    }

    int j = 0;
    for (int it = blockIdx.x; it < n_items; it += gridDim.x, ++j) {
        const int stage = j % K2_STAGES;
        const int sidx = it * K2_WARPS + warp;
        const bool have = sidx < n_segs;
        mbar_wait(&sm.full[stage], (j / K2_STAGES) & 1);
        ColSeg sg;
        sg.start = sm.seg[stage][0].start; sg.len = 0; sg.col = 0; sg.slot = -1;
        if (have) sg = sm.seg[stage][warp];
        const uint32_t a0 = sm.seg[stage][0].start & ~3u;
        const uint32_t len = sg.len & 0xffffu, run = sg.len >> 16;  // run > 0: head of a run of `run` segments
        double acc[KP];
        {
            const uint32_t *rp = &sm.row[stage][sg.start - a0];
            const float *vp = &sm.val[stage][sg.start - a0];
            float facc[KP];
#pragma unroll
            for (int k = 0; k < KP; ++k) { acc[k] = 0.0; facc[k] = 0.0f; }
            constexpr int U = (KP >= 16) ? 2 : 4;
            uint32_t off = lane;
            for (; off + 32 * (U - 1) < len; off += 32 * U) {
                float wv[U][KP];
                float v[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const uint32_t r = rp[off + 32 * u];
                    v[u] = vp[off + 32 * u];
                    Vec<KP>::ld(w + (size_t)r * KP, wv[u]);
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
#pragma unroll
                    for (int k = 0; k < KP; ++k) {
                        if (EXACT) acc[k] = fma((double)v[u], (double)wv[u][k], acc[k]);
                        else facc[k] = fmaf(v[u], wv[u][k], facc[k]);
                    }
                }
            }
            for (; off < len; off += 32) {
                const uint32_t r = rp[off];
                const float v = vp[off];
                float wv[KP];
                Vec<KP>::ld(w + (size_t)r * KP, wv);
#pragma unroll
                for (int k = 0; k < KP; ++k) {
                    if (EXACT) acc[k] = fma((double)v, (double)wv[k], acc[k]);
                    else facc[k] = fmaf(v, wv[k], facc[k]);
                }
            }
            if (!EXACT) {
#pragma unroll
                for (int k = 0; k < KP; ++k) acc[k] = (double)facc[k];
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&sm.empty[stage]);
        warp_reduce_scatter<KP>(acc, lane);
        // in-CTA combine without a block-wide stall: every warp publishes its partial and arrives on an mbarrier;
        // only the warps that head a run wait for it, everyone else moves on to the next item
        const int buf = j % K2_PART_BUFS;
        if (lane_writes<KP>(lane)) sm.part[buf][warp][draw_of_lane<KP>(lane)] = acc[0];
        __syncwarp();
        if (lane == 0) mbar_arrive(&sm.part_full[buf]);
        if (have && run > 0) mbar_wait(&sm.part_full[buf], (j / K2_PART_BUFS) & 1);
        if (have && run > 0 && lane < KP) {
            double s = 0.0;
            for (uint32_t q = 0; q < run; ++q) s += sm.part[buf][warp + q][lane];
            if (sg.slot < 0)
                g[(size_t)sg.col * KP + lane] = s;
            else
                seg_partial[(size_t)sg.slot * KP + lane] = s;
        }
    }
}

// columns that span several CTA items: one warp per column adds the partials in slot order
template <int KP>
__global__ void __launch_bounds__(256) k2_combine_warp(const MultiCol *__restrict__ multi, int n_multi,
                                                       const double *__restrict__ seg_partial, double *__restrict__ g) {
    const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (wid >= n_multi) return;
    const MultiCol mc = multi[wid];
    constexpr int SUB = 32 / KP;  // slots per warp iteration
    const int k = lane % KP, sub = lane / KP;
    double s = 0.0;
    for (uint32_t q = sub; q < mc.nslots; q += SUB) s += seg_partial[(size_t)(mc.first_slot + q) * KP + k];
#pragma unroll
    for (int o = 16; o >= KP; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (sub == 0) g[(size_t)mc.col * KP + k] = s;
}

__global__ void k_widen_f32(const float *__restrict__ in, double *__restrict__ out, size_t count) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x)
        out[i] = (double)in[i];
}

__global__ void k_narrow_f64(const double *__restrict__ in, float *__restrict__ out, size_t count) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x)
        out[i] = (float)in[i];
}

template <int KP>
int launch_k1_t(polee_handle *h, const float *x, float *w, bool want_lp, double *lp_partial) {
    if (h->n_row_tiles == 0) return POLEE_OK;
    const bool wt = h->row_weight != nullptr;
    if (h->o.exact_accumulation) {
        dim3 grid(h->n_row_tiles), block(ROW_TILE);
#define K1_LAUNCH(LPF, WF)                                                                                      \
    k1_sell_fwd<KP, LPF, WF><<<grid, block, 0, h->stream>>>(h->row_tiles, h->sell_idx, h->sell_val, x, w,       \
                                                            h->row_weight, lp_partial)
        if (want_lp) {
            if (wt) K1_LAUNCH(true, true); else K1_LAUNCH(true, false);
        } else {
            if (wt) K1_LAUNCH(false, true); else K1_LAUNCH(false, false);
        }
#undef K1_LAUNCH
        return POLEE_OK;
    }
    const int grid = std::min(h->n_row_tiles, h->num_sms * 3);
    const size_t smem = sizeof(K1Smem);
#define K1_LAUNCH2(LPF, WF)                                                                                 \
    do {                                                                                                    \
        allow_max_smem(k1_sell_fwd_tma<KP, LPF, WF>);                                                       \
        k1_sell_fwd_tma<KP, LPF, WF><<<grid, V2_THREADS, smem, h->stream>>>(                                \
            h->row_tiles, h->n_row_tiles, h->sell_idx, h->sell_val, x, w, h->row_weight, lp_partial);       \
    } while (0)
    if (want_lp) {
        if (wt) K1_LAUNCH2(true, true); else K1_LAUNCH2(true, false);
    } else {
        if (wt) K1_LAUNCH2(false, true); else K1_LAUNCH2(false, false);
    }
#undef K1_LAUNCH2
    return POLEE_OK;
}

template <int KP>
int launch_k2_t(polee_handle *h, const float *w, double *g) {
    if (h->n_segs > 0) {
        const int n_items = (h->n_segs + K2_WARPS - 1) / K2_WARPS;
        static const int k2_ctas = getenv("POLEE_K2_CTAS") ? atoi(getenv("POLEE_K2_CTAS")) : 3;
        const int grid = std::min(n_items, h->num_sms * k2_ctas);
        const size_t smem = sizeof(K2Smem);
#define K2_LAUNCH(EX)                                                                                           \
    do {                                                                                                        \
        allow_max_smem(k2_csc_grad_tma<KP, EX>);                                                                \
        k2_csc_grad_tma<KP, EX><<<grid, V2_THREADS, smem, h->stream>>>(h->segs, h->n_segs, h->csc_row, h->csc_val, \
                                                                       w, g, h->seg_partial);                  \
    } while (0)
        if (h->o.exact_accumulation) K2_LAUNCH(true);
        else K2_LAUNCH(false);
#undef K2_LAUNCH
    }
    if (h->n_multi > 0) {
        const int warps_per_block = 8;
        k2_combine_warp<KP><<<(h->n_multi + warps_per_block - 1) / warps_per_block, 256, 0, h->stream>>>(
            h->multi, h->n_multi, h->seg_partial, g);
    }
    return POLEE_OK;
}

}  // namespace

int launch_k1(polee_handle *h, const float *x, float *w, bool want_lp, double *lp_partial, int KP) {
    int rc = POLEE_OK;
    DISPATCH_KP(KP, rc = launch_k1_t<KPC>(h, x, w, want_lp, lp_partial));
    return rc;
}

int launch_k2(polee_handle *h, const float *w, double *g, int KP) {
    int rc = POLEE_OK;
    DISPATCH_KP(KP, rc = launch_k2_t<KPC>(h, w, g));
    return rc;
}

// the gradient crosses NVLink as Float32 (half the bytes of the all-reduce): narrow before, widen after
int launch_narrow(polee_handle *h, const double *in, float *out, size_t count) {
    k_narrow_f64<<<(unsigned)std::min<size_t>((count + 255) / 256, 4096), 256, 0, h->stream>>>(in, out, count);
    return POLEE_OK;
}
int launch_widen(polee_handle *h, const float *in, double *out, size_t count) {
    k_widen_f32<<<(unsigned)std::min<size_t>((count + 255) / 256, 4096), 256, 0, h->stream>>>(in, out, count);
    return POLEE_OK;
}

int launch_reduce_lp(polee_handle *h, const double *lp_partial, double *lp, int KP) {
    k_reduce_partials<<<1, 1024, 0, h->stream>>>(lp_partial, h->fused ? h->ft_tiles : h->n_row_tiles, KP, lp);
    return POLEE_OK;
}

}  // namespace polee
