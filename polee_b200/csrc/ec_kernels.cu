// ec_kernels.cu -- the likelihood pass of one ADAM step on the equivalence-class layout (common.cuh, "ec"):
// pAt_mul_B! (src/sparse.jl:6-21), 1 ./ frag_probs, log! + sum (src/likelihood.jl:21-25,43-51) and pAt_mulinv_B!
// (src/sparse.jl:25-40) in ONE pass over the matrix, for the K Monte-Carlo draws of the step at once.
//
// A task = <= ec_nbt(L) blocks of one class (L transcripts).  One warp works on one task at a time; a block is 32
// lanes = 32 / q fragments (rows) x q column slices of LH = ceil(L / q) <= 8 transcripts (q = 1 for L <= 8).  A lane
// holds its row's LH values and, for the whole task, the LH x K gradient sums of its slice in registers:
//     p[k]     = sum_j v[j] * x[col_j][k]   (own slice, then summed over the q lanes of the row by butterflies)
//     w[k]     = 1 / p[k]
//     a[j][k] += v[j] * w[k]
// so the matrix is read ONCE from shared memory (one conflict-free 128-byte read per 32 entries), w never leaves the
// registers, and nothing is exchanged between lanes per row when L <= 8.  At the end of the task the 32 / q lanes of
// a slice add their sums (reduce-scatter by shuffles, fixed order) and write one partial per (task, transcript) to
// its slot of the transcript-ordered partial array; k_ec_combine1/2 add each transcript's partials in Float64 in a
// fixed order (no atomics anywhere).
//
// Arithmetic, template parameter T (opts.exact_accumulation, see ec_math_f32):
//   double: values and x widened exactly, every product and every sum in Float64 -- at least the reference's
//           "Float32 product, Float64 accumulation" (SURVEY App. A); 1/p = MUFU.RCP64H + one Newton step (8.5e-13).
//   float : FFMA2 (two draws per instruction); a row's sum (<= 64 terms) and a lane's column sums over the task's
//           blocks (<= 32 terms) + the 5-level lane tree are Float32, everything across tasks is Float64.
//
// Every warp is its own pipeline: it owns EC_STAGES shared-memory stages fed by 1-D bulk copies
// (cp.async.bulk -> UBLKCP) completing on mbarriers, takes tasks gw, gw + G, gw + 2G, ... (static, so results do not
// depend on scheduling), and never synchronises with another warp.
#include <algorithm>
#include <cstdlib>

#include "common.cuh"
#include "device_utils.cuh"

namespace polee {

namespace {

#ifndef POLEE_EC_F32_WARPS
#define POLEE_EC_F32_WARPS 12
#endif
#ifndef POLEE_EC_F64_WARPS
#define POLEE_EC_F64_WARPS 8
#endif
constexpr int EC_STAGES = 2;
constexpr uint32_t EC_STAGE_STRIDE = (EC_STAGE_BYTES + 127u) & ~127u;
constexpr uint32_t EC_CTL_BYTES = 256;  // the mbarriers
constexpr uint32_t EC_FLAG_LP = 1u, EC_FLAG_WRITE_W = 2u;

template <typename T>
struct EcCfg {
    // x of the task's columns, staged per warp as T: slice h at h * XS, column j of the slice at j * 8, draw k at + k.
    // XS is an odd number of 16-byte units, so the q lanes of a row (which read q different slices with one
    // instruction) hit different banks.
    static constexpr uint32_t XS = (8u * 8u * sizeof(T) + 16u) / sizeof(T);
    static constexpr uint32_t XBUF = (8u * XS * (uint32_t)sizeof(T) + 127u) & ~127u;
    static constexpr uint32_t WARP_BYTES = EC_STAGES * EC_STAGE_STRIDE + XBUF;
    // float: as many warps as the shared memory holds (11, 168 registers each); double: 8, so that a lane's 64
    // Float64 sums + operands fit the 255 registers a thread may have
    static constexpr int SMEM_WARPS = (int)((MAX_SMEM_PER_CTA - EC_CTL_BYTES) / WARP_BYTES);
    static constexpr int CAP = sizeof(T) == 8 ? POLEE_EC_F64_WARPS : POLEE_EC_F32_WARPS;
    static constexpr int WARPS = SMEM_WARPS < CAP ? SMEM_WARPS : CAP;
    static constexpr uint32_t SMEM = WARPS * WARP_BYTES + EC_CTL_BYTES;
};
static_assert(EcCfg<float>::WARPS * EC_STAGES * 8 <= (int)EC_CTL_BYTES, "mbarrier block");
static_assert(EcCfg<float>::WARPS >= EcCfg<double>::WARPS, "mbarrier block");

// ---------------------------------------------------------------- scalar helpers
template <typename T>
__device__ __forceinline__ T ec_rcp(T p);
// 1 / p: MUFU.RCP64H seed (9e-7) + one Newton step (8.5e-13 measured, tools/ubench/fp64_rates.cu)
template <>
__device__ __forceinline__ double ec_rcp<double>(double p) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(p));
    const double e = fma(-p, r, 1.0);
    return fma(r, e, r);
}
// MUFU.RCP alone: 1 ulp, the same order as the Float32 rounding of the sums around it
template <>
__device__ __forceinline__ float ec_rcp<float>(float p) {
    return rcp_approx(p);
}

// a[k] += s * b[k]
template <int KD>
__device__ __forceinline__ void fma_vec(double (&a)[KD], double s, const double (&b)[KD]) {
#pragma unroll
    for (int k = 0; k < KD; ++k) a[k] = fma(s, b[k], a[k]);
}
template <int KD>
__device__ __forceinline__ void fma_vec(float (&a)[KD], float s, const float (&b)[KD]) {
#pragma unroll
    for (int k = 0; k + 1 < KD; k += 2)  // FFMA2: both halves are exactly fmaf
        asm("{\n\t.reg .b64 ra, rb, rc;\n\tmov.b64 ra, {%2, %2};\n\tmov.b64 rb, {%3, %4};\n\tmov.b64 rc, {%0, %1};\n\t"
            "fma.rn.f32x2 rc, ra, rb, rc;\n\tmov.b64 {%0, %1}, rc;\n\t}"
            : "+f"(a[k]), "+f"(a[k + 1])
            : "f"(s), "f"(b[k]), "f"(b[k + 1]));
    if constexpr (KD & 1) a[KD - 1] = fmaf(s, b[KD - 1], a[KD - 1]);
}

// KD consecutive elements from / to 16-byte aligned addresses
template <int KD>
__device__ __forceinline__ void ld_vec(const float *p, float (&v)[KD]) {
    if constexpr (KD >= 4) {
        const float4 t = *reinterpret_cast<const float4 *>(p);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    }
    if constexpr (KD == 8) {
        const float4 t = *reinterpret_cast<const float4 *>(p + 4);
        v[4] = t.x; v[5] = t.y; v[6] = t.z; v[7] = t.w;
    }
    if constexpr (KD == 6 || KD == 2) {
        const float2 t = *reinterpret_cast<const float2 *>(p + (KD - 2));
        v[KD - 2] = t.x; v[KD - 1] = t.y;
    }
    if constexpr (KD == 1) v[0] = p[0];
}
template <int KD>
__device__ __forceinline__ void ld_vec(const double *p, double (&v)[KD]) {
#pragma unroll
    for (int k = 0; k + 1 < KD; k += 2) {
        const double2 t = *reinterpret_cast<const double2 *>(p + k);
        v[k] = t.x; v[k + 1] = t.y;
    }
    if constexpr (KD & 1) v[KD - 1] = p[KD - 1];
}
// store KD values and zeros up to KPAD (the draws the padded layout carries but nobody asked for)
template <int KD>
__device__ __forceinline__ void st_vec(float *p, const float (&v)[KD], int kpad) {
    if constexpr (KD == 8) {
        *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4 *>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
    } else if constexpr (KD == 6) {
        *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4 *>(p + 4) = make_float4(v[4], v[5], 0.0f, 0.0f);
    } else if constexpr (KD == 4) {
        *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
#pragma unroll
        for (int k = 0; k < KD; ++k) p[k] = v[k];
        for (int k = KD; k < kpad; ++k) p[k] = 0.0f;
    }
}
template <int KD>
__device__ __forceinline__ void st_vec(double *p, const double (&v)[KD], int kpad) {
    if constexpr (KD >= 2) {
#pragma unroll
        for (int k = 0; k + 1 < KD; k += 2) *reinterpret_cast<double2 *>(p + k) = make_double2(v[k], v[k + 1]);
        if constexpr (KD == 6) *reinterpret_cast<double2 *>(p + 6) = make_double2(0.0, 0.0);
    } else {
        p[0] = v[0];
        for (int k = KD; k < kpad; ++k) p[k] = 0.0;
    }
}

// One level of the reduce-scatter over the lanes of a slice: lanes with (lane & MASK) == 0 keep columns [0, H) of
// their N = 2 H, the others keep [H, 2 H); each receives the partner's copy of what it keeps.
template <typename T, int KD, int H>
__device__ __forceinline__ void scatter_level(const T (&in)[2 * H][KD], T (&out)[H][KD], int lane, int mask) {
    const bool up = (lane & mask) != 0;
#pragma unroll
    for (int j = 0; j < H; ++j)
#pragma unroll
        for (int k = 0; k < KD; ++k) {
            const T send = up ? in[j][k] : in[j + H][k];
            const T keep = up ? in[j + H][k] : in[j][k];
            out[j][k] = keep + __shfl_xor_sync(0xffffffffu, send, mask);
        }
}

struct EcArgs {
    const float *xf;              // [n][KP]
    void *partial;                // [parts][KP] of T
    const float *slot_weight;     // nullable
    const uint32_t *row_of_slot;  // for WRITE_W
    double *lp_partial;           // [tasks][KP]
    float *w_out;                 // [m][KP]
    int KP;
    uint32_t flags;
};

// ---- shared-memory helpers on 32-bit shared-window addresses (no generic -> shared conversion per use)
__device__ __forceinline__ void mbar_wait_u32(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "EC_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra EC_DONE;\n"
        "bra EC_WAIT;\n"
        "EC_DONE:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_refill_u32(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}

// ---- x of a task's columns.  An "item" is one 16-byte piece (4 draws) of one column's row of x when KD >= 4, else one
// draw of one column; item idx of the task in `stage` -> registers (zero beyond the task's items) ...
template <int KD>
__device__ __forceinline__ float4 ec_xload(const unsigned char *__restrict__ stage, const EcArgs &A, int kb, uint32_t idx) {
    const uint32_t pk = reinterpret_cast<const EcHdr *>(stage)->pk, Lq = ec_pk_q(pk) * ec_pk_lh(pk);
    const uint32_t *cols = reinterpret_cast<const uint32_t *>(stage + 16);
    float4 t = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    if constexpr (KD >= 4) {
        constexpr uint32_t NV = (KD + 3) / 4;
        if (idx < Lq * NV) {
            const uint32_t c = idx / NV, part = idx - c * NV;
            t = __ldg(reinterpret_cast<const float4 *>(A.xf + (size_t)cols[c] * A.KP + kb + part * 4));
        }
    } else {
        if (idx < Lq * KD) {
            const uint32_t c = idx / KD, k = idx - c * KD;
            t.x = __ldg(A.xf + (size_t)cols[c] * A.KP + kb + k);
        }
    }
    return t;
}
// ... -> its place in xbuf, as T (LH compile-time; q = 1 when LH <= 4)
template <typename T, int KD, int LH>
__device__ __forceinline__ void ec_xstore(T *__restrict__ xbuf, uint32_t idx, uint32_t q, const float4 &t) {
    constexpr uint32_t NI = KD >= 4 ? (KD + 3) / 4 : KD;  // items per column
    if (idx >= q * LH * NI) return;
    const uint32_t c = idx / NI, r = idx - c * NI;
    uint32_t hs = 0, j = c;
    if constexpr (LH > 4) {
        hs = c / (uint32_t)LH;
        j = c - hs * LH;
    }
    T *d = xbuf + hs * EcCfg<T>::XS + j * 8u;
    if constexpr (KD >= 4) {
        d += r * 4u;
        d[0] = (T)t.x; d[1] = (T)t.y; d[2] = (T)t.z; d[3] = (T)t.w;
    } else {
        d[r] = (T)t.x;
    }
}

// UB rows of one lane at a time (UB blocks of the task): p, w = 1 / p, a += v w.  CHECK: the rows may be padding.
template <typename T, int KD, int LH, int UB, bool CHECK, bool FULL>
__device__ __forceinline__ void ec_rows(const float *__restrict__ vb, const T *__restrict__ xs, uint32_t q, uint32_t row0,
                                        uint32_t nr, uint32_t rows, uint32_t slot, uint32_t h, int kb, const EcArgs &A,
                                        T (&acc)[LH][KD], double (&lpv)[KD]) {
    T v[UB][LH];
#pragma unroll
    for (int u = 0; u < UB; ++u)
#pragma unroll
        for (int j = 0; j < LH; ++j) v[u][j] = (T)vb[(u * LH + j) * 32];
    T p[UB][KD];
#pragma unroll
    for (int u = 0; u < UB; ++u)
#pragma unroll
        for (int k = 0; k < KD; ++k) p[u][k] = (T)0;
#pragma unroll
    for (int j = 0; j < LH; ++j) {
        T xk[KD];
        ld_vec<KD>(xs + j * 8, xk);
#pragma unroll
        for (int u = 0; u < UB; ++u) fma_vec<KD>(p[u], v[u][j], xk);
    }
    if constexpr (LH > 4) {  // q > 1 only then: add the row's other slices
        if (q >= 2) {
#pragma unroll
            for (int u = 0; u < UB; ++u)
#pragma unroll
                for (int k = 0; k < KD; ++k) p[u][k] += __shfl_xor_sync(0xffffffffu, p[u][k], 1);
            if (q >= 4) {
#pragma unroll
                for (int u = 0; u < UB; ++u)
#pragma unroll
                    for (int k = 0; k < KD; ++k) p[u][k] += __shfl_xor_sync(0xffffffffu, p[u][k], 2);
                if (q >= 8) {
#pragma unroll
                    for (int u = 0; u < UB; ++u)
#pragma unroll
                        for (int k = 0; k < KD; ++k) p[u][k] += __shfl_xor_sync(0xffffffffu, p[u][k], 4);
                }
            }
        }
    }
#pragma unroll
    for (int u = 0; u < UB; ++u) {
        const bool valid = !CHECK || row0 + u * nr < rows;
        T w[KD];
#pragma unroll
        for (int k = 0; k < KD; ++k) w[k] = valid ? ec_rcp<T>(p[u][k]) : (T)0;  // padding rows: p = 0, w = 0
        if constexpr (FULL) {
            const uint32_t sl = slot + u * 32u;
            T wt = (T)1;
            if (A.slot_weight != nullptr) {
                wt = valid ? (T)A.slot_weight[sl] : (T)0;
#pragma unroll
                for (int k = 0; k < KD; ++k) w[k] *= wt;
            }
            if ((A.flags & EC_FLAG_LP) && valid && h == 0u) {
#pragma unroll 1
                for (int k = 0; k < KD; ++k) lpv[k] += (double)wt * log((double)p[u][k]);
            }
            if ((A.flags & EC_FLAG_WRITE_W) && valid && h == 0u) {
                float *o = A.w_out + (size_t)A.row_of_slot[sl] * A.KP + kb;
#pragma unroll
                for (int k = 0; k < KD; ++k) o[k] = (float)w[k];
            }
        }
#pragma unroll
        for (int j = 0; j < LH; ++j) fma_vec<KD>(acc[j], v[u][j], w);
    }
}

// Sum over the lanes of a slice of the LH column sums a lane holds, one partial per column out.
// LH <= 4 (q = 1, all five lane bits are row bits): columns are scattered over the top lane bits, the rest are
// butterflies, the lane with the low bits clear writes.  LH > 4 (q = 1, 2, 4, 8; the slice's rows are lane bits >= lq):
// the 8 columns are scattered over lane bits 4, 3 (, 2), butterflies below.
template <typename T, int KD, int LH>
__device__ __forceinline__ void ec_reduce(T (&acc)[LH][KD], int lane, uint32_t L, uint32_t q, uint32_t lq,
                                          const uint32_t *__restrict__ dest, T *__restrict__ partial, int KP, int kb, int kpad) {
    if constexpr (LH <= 4) {
        constexpr int NC = LH == 1 ? 1 : (LH == 2 ? 2 : 4);
        T r[KD];
        uint32_t j = 0;
        int low = 31;  // lane bits still to be reduced by butterflies
        if constexpr (NC == 4) {
            T a4[4][KD], a2[2][KD], a1[1][KD];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int k = 0; k < KD; ++k) a4[i][k] = i < LH ? acc[i < LH ? i : 0][k] : (T)0;
            scatter_level<T, KD, 2>(a4, a2, lane, 16);
            scatter_level<T, KD, 1>(a2, a1, lane, 8);
#pragma unroll
            for (int k = 0; k < KD; ++k) r[k] = a1[0][k];
            j = (uint32_t)lane >> 3;
            low = 7;
        } else if constexpr (NC == 2) {
            T a1[1][KD];
            scatter_level<T, KD, 1>(acc, a1, lane, 16);
#pragma unroll
            for (int k = 0; k < KD; ++k) r[k] = a1[0][k];
            j = (uint32_t)lane >> 4;
            low = 15;
        } else {
#pragma unroll
            for (int k = 0; k < KD; ++k) r[k] = acc[0][k];
        }
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1)
            if (o & low) {
#pragma unroll
                for (int k = 0; k < KD; ++k) r[k] += __shfl_xor_sync(0xffffffffu, r[k], o);
            }
        if ((lane & low) == 0 && j < L) st_vec<KD>(partial + (size_t)dest[j] * KP + kb, r, kpad);
    } else {
        const uint32_t h = (uint32_t)lane & (q - 1u);
        T a8[8][KD], a4[4][KD], a2[2][KD];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int k = 0; k < KD; ++k) a8[i][k] = i < LH ? acc[i < LH ? i : 0][k] : (T)0;
        scatter_level<T, KD, 4>(a8, a4, lane, 16);
        scatter_level<T, KD, 2>(a4, a2, lane, 8);
        if (q == 8u) {  // 4 rows per block: done, the lane holds columns 2 (lane >> 3) + {0, 1} of slice h
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const uint32_t j = 2u * ((uint32_t)lane >> 3) + i, l = h * LH + j;
                if (j < (uint32_t)LH && l < L) st_vec<KD>(partial + (size_t)dest[l] * KP + kb, a2[i], kpad);
            }
        } else {
            T a1[1][KD];
            scatter_level<T, KD, 1>(a2, a1, lane, 4);
            if (q <= 2u) {
#pragma unroll
                for (int k = 0; k < KD; ++k) a1[0][k] += __shfl_xor_sync(0xffffffffu, a1[0][k], 2);
                if (q == 1u) {
#pragma unroll
                    for (int k = 0; k < KD; ++k) a1[0][k] += __shfl_xor_sync(0xffffffffu, a1[0][k], 1);
                }
            }
            const uint32_t j = (uint32_t)lane >> 2, l = h * LH + j;
            const bool writer = (((uint32_t)lane & 3u) >> lq) == 0u;  // q = 1: lane & 3 == 0; q = 2: lane & 2 == 0; q = 4: all
            if (writer && j < (uint32_t)LH && l < L) st_vec<KD>(partial + (size_t)dest[l] * KP + kb, a1[0], kpad);
        }
    }
}

// A warp's position in its task sequence and in its two-stage pipeline
struct EcWarp {
    int tk, G, n_tasks;        // current task, stride, total
    uint32_t s, phase;         // current stage; parity bit per stage
    uint32_t mine_u32, bar_u32;  // shared-window addresses of the warp's first stage and first mbarrier
    float4 xpre;               // item `lane` of the current task's first draw batch
};

// All tasks of the warp below `end` (they all have LH columns per slice): for each, x -> xbuf, the blocks, the x items
// of the NEXT task requested (their latency is covered by the reduction), the reduction, the stage refilled.
template <typename T, int KD, int LH, bool FULL>
__device__ __forceinline__ void ec_run(EcWarp &W, int end, unsigned char *__restrict__ mine, T *__restrict__ xbuf,
                                       const EcTaskDesc *__restrict__ desc, const unsigned char *__restrict__ blob,
                                       const EcArgs &A, int lane) {
    constexpr uint32_t NI = KD >= 4 ? (KD + 3) / 4 : KD;
    constexpr int UB = sizeof(T) == 8 ? (LH <= 4 ? 2 : 1) : (LH <= 6 ? 2 : 1);  // rows of a lane in flight (registers permitting)
    const int KP = A.KP, kpad = KP < 8 ? KP : 8, nbatch = KP > 8 ? KP / 8 : 1;
    T *partial = reinterpret_cast<T *>(A.partial);
#pragma unroll 1
    while (W.tk < end) {
        const uint32_t s = W.s, s1 = s ^ 1u;
        const unsigned char *stage = mine + s * EC_STAGE_STRIDE;
        const EcHdr hd = *reinterpret_cast<const EcHdr *>(stage);
        const uint32_t L = ec_pk_l(hd.pk);
        uint32_t q = 1u, lq = 0u;
        if constexpr (LH > 4) {
            q = ec_pk_q(hd.pk);
            lq = ec_pk_lq(hd.pk);
        }
        const uint32_t h = (uint32_t)lane & (q - 1u), rho = (uint32_t)lane >> lq, nr = 32u >> lq;
        const uint32_t *dest = reinterpret_cast<const uint32_t *>(stage + 16) + q * LH;
        const float *V = reinterpret_cast<const float *>(stage + ((16u + 8u * q * LH + 15u) & ~15u)) + lane;
        const T *xs = xbuf + h * EcCfg<T>::XS;
        const bool has_next = W.tk + W.G < W.n_tasks;
        // descriptor of the task that will reuse this stage, fetched while the current one is processed
        const int nxt = W.tk + EC_STAGES * W.G;
        EcTaskDesc dn{0, 0, 0};
        if (lane == 0 && nxt < W.n_tasks) dn = desc[nxt];
#pragma unroll 1
        for (int bt = 0; bt < nbatch; ++bt) {
            const int kb = bt * 8;
            // ---- x of the task's columns -> xbuf (as T)
            __syncwarp();  // everybody is done with the previous contents of xbuf
            if (bt > 0) W.xpre = ec_xload<KD>(stage, A, kb, (uint32_t)lane);
            ec_xstore<T, KD, LH>(xbuf, (uint32_t)lane, q, W.xpre);
            if constexpr (LH > 4) {
                for (uint32_t idx = lane + 32u; idx < q * LH * NI; idx += 32u)
                    ec_xstore<T, KD, LH>(xbuf, idx, q, ec_xload<KD>(stage, A, kb, idx));
            } else if constexpr (LH * NI > 32) {
                ec_xstore<T, KD, LH>(xbuf, lane + 32u, q, ec_xload<KD>(stage, A, kb, lane + 32u));
            }
            __syncwarp();
            T acc[LH][KD];
#pragma unroll
            for (int j = 0; j < LH; ++j)
#pragma unroll
                for (int k = 0; k < KD; ++k) acc[j][k] = (T)0;
            double lpv[KD];
#pragma unroll
            for (int k = 0; k < KD; ++k) lpv[k] = 0.0;
            const uint32_t nb_full = hd.rows >> (5u - lq);  // blocks without padding rows
            uint32_t b = 0;
#pragma unroll 1
            for (; b + UB <= nb_full; b += UB)
                ec_rows<T, KD, LH, UB, false, FULL>(V + b * (LH * 32u), xs, q, b * nr + rho, nr, hd.rows, hd.slot0 + b * 32u + rho, h,
                                                    kb, A, acc, lpv);
#pragma unroll 1
            for (; b < hd.nb; ++b)
                ec_rows<T, KD, LH, 1, true, FULL>(V + b * (LH * 32u), xs, q, b * nr + rho, nr, hd.rows, hd.slot0 + b * 32u + rho, h,
                                                  kb, A, acc, lpv);
            if (bt + 1 == nbatch && has_next) {
                mbar_wait_u32(W.bar_u32 + s1 * 8u, (W.phase >> s1) & 1u);
                W.xpre = ec_xload<KD>(mine + s1 * EC_STAGE_STRIDE, A, 0, (uint32_t)lane);
            }
            ec_reduce<T, KD, LH>(acc, lane, L, q, lq, dest, partial, KP, kb, kpad);
            if constexpr (FULL) {
                if (A.flags & EC_FLAG_LP) {
#pragma unroll
                    for (int k = 0; k < KD; ++k) {
                        double sum = lpv[k];
#pragma unroll
                        for (int o = 16; o >= 1; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
                        if (lane == 0) A.lp_partial[(size_t)W.tk * KP + kb + k] = sum;
                    }
                    if (lane == 0)
                        for (int k = KD; k < kpad; ++k) A.lp_partial[(size_t)W.tk * KP + kb + k] = 0.0;
                }
            }
        }
        if (has_next) W.phase ^= 1u << s1;  // waited for above
        __syncwarp();                       // every lane is done reading the stage
        if (lane == 0 && nxt < W.n_tasks) bulk_refill_u32(W.mine_u32 + s * EC_STAGE_STRIDE, blob + dn.off, dn.bytes, W.bar_u32 + s * 8u);
        W.s = s1;
        W.tk += W.G;
    }
}

// tasks are ordered by LH, 8 first: tasks [kinds.end[i - 1], kinds.end[i]) have LH = 8 - i
struct EcKinds {
    int end[8];
};

template <typename T, int KD, bool FULL>
__global__ void __launch_bounds__(EcCfg<T>::WARPS * 32, 1)
    k_ec_lik(const EcTaskDesc *__restrict__ desc, int n_tasks, const unsigned char *__restrict__ blob, const EcArgs A,
             const EcKinds kinds) {
    using Cfg = EcCfg<T>;
    extern __shared__ __align__(128) unsigned char smraw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smraw) + warp * EC_STAGES;
    unsigned char *mine = smraw + EC_CTL_BYTES + (size_t)warp * Cfg::WARP_BYTES;
    T *xbuf = reinterpret_cast<T *>(mine + EC_STAGES * EC_STAGE_STRIDE);
    EcWarp W;
    W.G = gridDim.x * Cfg::WARPS;
    W.tk = blockIdx.x * Cfg::WARPS + warp;
    W.n_tasks = n_tasks;
    if (W.tk >= n_tasks) {
        pdl_wait();
        return;
    }
    W.mine_u32 = smem_u32(mine);
    W.bar_u32 = smem_u32(bars);
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < EC_STAGES; ++s) mbar_init(&bars[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#pragma unroll
        for (int s = 0; s < EC_STAGES; ++s) {  // prologue: the first EC_STAGES tasks of this warp
            const int tk = W.tk + s * W.G;
            if (tk < n_tasks) {
                const EcTaskDesc dd = desc[tk];
                bulk_refill_u32(W.mine_u32 + s * EC_STAGE_STRIDE, blob + dd.off, dd.bytes, W.bar_u32 + s * 8u);
            }
        }
    }
    __syncwarp();
    // the copies above read only the constant blob; x is the tree forward's output
    pdl_wait();
    W.s = 0;
    mbar_wait_u32(W.bar_u32, 0u);
    W.phase = 1u;
    W.xpre = ec_xload<KD>(mine, A, 0, (uint32_t)lane);
#define EC_KIND(i) \
    if (W.tk < kinds.end[i]) ec_run<T, KD, 8 - (i), FULL>(W, kinds.end[i], mine, xbuf, desc, blob, A, lane)
    EC_KIND(0); EC_KIND(1); EC_KIND(2); EC_KIND(3); EC_KIND(4); EC_KIND(5); EC_KIND(6); EC_KIND(7);
#undef EC_KIND
    // not at the start: the next kernel's waiting CTAs would take SM space k3_leaf_S uses beside this kernel
    pdl_trigger();
}

// g[col] (or a level-2 slot) = [g[col] +] sum of <= FT_UNIT partials of one column, in task order, in Float64
template <typename P, int KP>
__global__ void __launch_bounds__(256)
    k_ec_combine1(const FusedUnit *__restrict__ units, int n_units, const P *__restrict__ partial, double *__restrict__ g,
                  double *__restrict__ lvl2, int add_to_g) {
    constexpr int GP = 32 / KP;
    const int warp_global = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    const int unit = warp_global * GP + lane / KP, k = lane % KP;
    pdl_trigger();
    FusedUnit u{};
    if (unit < n_units) u = units[unit];
    pdl_wait();
    if (unit >= n_units) return;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    uint32_t i = u.begin;
    for (; i + 4 <= u.end; i += 4) {
        a0 += (double)partial[(size_t)i * KP + k];
        a1 += (double)partial[(size_t)(i + 1) * KP + k];
        a2 += (double)partial[(size_t)(i + 2) * KP + k];
        a3 += (double)partial[(size_t)(i + 3) * KP + k];
    }
    for (; i < u.end; ++i) a0 += (double)partial[(size_t)i * KP + k];
    const double a = (a0 + a1) + (a2 + a3);
    if (u.out < 0) {
        double *o = g + (size_t)u.col * KP + k;
        *o = add_to_g ? *o + a : a;
    } else {
        lvl2[(size_t)u.out * KP + k] = a;
    }
}

template <int KP>
__global__ void __launch_bounds__(256)
    k_ec_combine2(const FusedMulti *__restrict__ multi, int n_multi, const double *__restrict__ lvl2, double *__restrict__ g,
                  int add_to_g) {
    const int idx = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    pdl_trigger();
    FusedMulti mc{};
    if (idx < n_multi) mc = multi[idx];
    pdl_wait();
    if (idx >= n_multi) return;
    const int lane = threadIdx.x & 31;
    constexpr int GP = 32 / KP;
    const int grp = lane / KP, k = lane % KP;
    double a = 0.0;
    for (uint32_t i = grp; i < mc.count; i += GP) a += lvl2[(size_t)(mc.first + i) * KP + k];
#pragma unroll
    for (int o = 16; o >= KP; o >>= 1) a += __shfl_down_sync(0xffffffffu, a, o);
    if (grp == 0) {
        double *o = g + (size_t)mc.col * KP + k;
        *o = add_to_g ? *o + a : a;
    }
}

// single CTA, fixed order: out[k] = [out[k] +] sum_t partial[t][k]
__global__ void __launch_bounds__(1024) k_ec_reduce_lp(const double *__restrict__ partial, int count, int KP, double *__restrict__ out,
                                                       int add) {
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
    if (threadIdx.x < KP) out[threadIdx.x] = add ? out[threadIdx.x] + sm[threadIdx.x] : sm[threadIdx.x];
}

template <typename T, int KD, bool FULL>
int launch_lik_full(polee_handle *h, const EcArgs &A) {
    auto kern = k_ec_lik<T, KD, FULL>;
    cudaError_t e = allow_max_smem(kern);
    if (e != cudaSuccess) return h->fail(POLEE_ECUDA, std::string("ec kernel smem: ") + cudaGetErrorString(e));
    const int grid = std::max(1, std::min(h->ec_grid, (h->ec_tasks + EcCfg<T>::WARPS - 1) / EcCfg<T>::WARPS));
    EcKinds kinds;
    for (int i = 0; i < 8; ++i) kinds.end[i] = h->ec_kind_end[i];
    launch_pdl(h, kern, grid, EcCfg<T>::WARPS * 32, EcCfg<T>::SMEM, h->stream, h->ec_desc, h->ec_tasks, h->ec_blob, A, kinds);
    return POLEE_OK;
}

template <typename T, int KD>
int launch_lik(polee_handle *h, const EcArgs &A) {
    const bool full = A.flags != 0u || A.slot_weight != nullptr;
    return full ? launch_lik_full<T, KD, true>(h, A) : launch_lik_full<T, KD, false>(h, A);
}

template <typename T>
int launch_lik_kd(polee_handle *h, const EcArgs &A, int K) {
    if (K > 8) return launch_lik<T, 8>(h, A);   // KP = 16: batches of 8
    switch (K) {
        case 1: return launch_lik<T, 1>(h, A);
        case 2: return launch_lik<T, 2>(h, A);
        case 3: case 4: return launch_lik<T, 4>(h, A);
        case 5: case 6: return launch_lik<T, 6>(h, A);
        default: return launch_lik<T, 8>(h, A);
    }
}

template <typename P, int KP>
void launch_combine(polee_handle *h, double *g, bool add_to_g) {
    if (h->ec_nunits > 0) {
        const int units_per_block = 8 * (32 / KP);
        const int blocks = (h->ec_nunits + units_per_block - 1) / units_per_block;
        launch_pdl(h, k_ec_combine1<P, KP>, blocks, 256, 0, h->stream, h->ec_units, h->ec_nunits,
                   reinterpret_cast<const P *>(h->ec_partial), g, h->ec_lvl2, add_to_g ? 1 : 0);
    }
    if (h->ec_nmulti > 0) {
        const int blocks = (h->ec_nmulti + 7) / 8;
        launch_pdl(h, k_ec_combine2<KP>, blocks, 256, 0, h->stream, h->ec_multi, h->ec_nmulti, h->ec_lvl2, g, add_to_g ? 1 : 0);
    }
}

template <typename P>
int launch_combine_kp(polee_handle *h, double *g, bool add_to_g, int KP) {
    switch (KP) {
        case 1: launch_combine<P, 1>(h, g, add_to_g); break;
        case 2: launch_combine<P, 2>(h, g, add_to_g); break;
        case 4: launch_combine<P, 4>(h, g, add_to_g); break;
        case 8: launch_combine<P, 8>(h, g, add_to_g); break;
        case 16: launch_combine<P, 16>(h, g, add_to_g); break;
        default: return h->fail(POLEE_EINVAL, "unsupported number of MC draws (1..16)");
    }
    return POLEE_OK;
}

template <typename T, int KD>
void preload_lik_kd() {
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, k_ec_lik<T, KD, false>);
}
template <typename P>
void preload_combine(int KP) {
    cudaFuncAttributes a;
    switch (KP) {
        case 1: cudaFuncGetAttributes(&a, k_ec_combine1<P, 1>); cudaFuncGetAttributes(&a, k_ec_combine2<1>); break;
        case 2: cudaFuncGetAttributes(&a, k_ec_combine1<P, 2>); cudaFuncGetAttributes(&a, k_ec_combine2<2>); break;
        case 4: cudaFuncGetAttributes(&a, k_ec_combine1<P, 4>); cudaFuncGetAttributes(&a, k_ec_combine2<4>); break;
        case 8: cudaFuncGetAttributes(&a, k_ec_combine1<P, 8>); cudaFuncGetAttributes(&a, k_ec_combine2<8>); break;
        case 16: cudaFuncGetAttributes(&a, k_ec_combine1<P, 16>); cudaFuncGetAttributes(&a, k_ec_combine2<16>); break;
        default: break;
    }
}
template <typename T>
void preload_ec(int KP, int K) {
    if (K > 8) preload_lik_kd<T, 8>();
    else if (K == 1) preload_lik_kd<T, 1>();
    else if (K == 2) preload_lik_kd<T, 2>();
    else if (K <= 4) preload_lik_kd<T, 4>();
    else if (K <= 6) preload_lik_kd<T, 6>();
    else preload_lik_kd<T, 8>();
    preload_combine<T>(KP);
}

}  // namespace

// see preload_tree_kernels (tree_kernels.cu): the class kernel and its second stage, gradient-only variant
void preload_ec_kernels(const polee_handle *h, int KP, int K) {
    if (ec_math_f32(h)) preload_ec<float>(KP, K);
    else preload_ec<double>(KP, K);
    cudaGetLastError();
}

// The arithmetic of the class kernel (see the header of this file): Float32 runs by default, Float64 with
// opts.exact_accumulation == 2.
bool ec_math_f32(const polee_handle *h) { return h->o.exact_accumulation != 2; }

int ec_grid(polee_handle *h, int KP) {
    (void)KP;
    int ctas = h->num_sms;  // one CTA of independent warp pipelines per SM (shared memory bound)
    if (const char *e = getenv("POLEE_EC_CTAS")) ctas = std::max(1, atoi(e));
    return std::max(1, ctas);
}

// K = the draws asked for (<= KP, the draws the [item][KP] buffers carry)
int launch_ec(polee_handle *h, const float *x, double *g, bool add_to_g, bool want_lp, double *lp_out, float *w_out, int KP, int K,
              bool lik_only) {
    EcArgs A;
    A.xf = x; A.partial = h->ec_partial; A.slot_weight = h->ec_slot_weight; A.row_of_slot = h->ec_row_of_slot;
    A.lp_partial = h->ec_lp_partial; A.w_out = w_out; A.KP = KP;
    A.flags = (want_lp ? EC_FLAG_LP : 0u) | (w_out ? EC_FLAG_WRITE_W : 0u);
    if (K < 1 || K > KP) K = KP;
    const bool f32 = ec_math_f32(h);
    int rc = f32 ? launch_lik_kd<float>(h, A, K) : launch_lik_kd<double>(h, A, K);
    if (rc || lik_only) return rc;
    rc = f32 ? launch_combine_kp<float>(h, g, add_to_g, KP) : launch_combine_kp<double>(h, g, add_to_g, KP);
    if (rc) return rc;
    if (want_lp && lp_out) k_ec_reduce_lp<<<1, 1024, 0, h->stream>>>(h->ec_lp_partial, h->ec_tasks, KP, lp_out, add_to_g ? 1 : 0);
    return POLEE_OK;
}

}  // namespace polee
