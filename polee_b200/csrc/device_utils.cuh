// device_utils.cuh -- small device helpers shared by the sparse kernels: vector loads/stores of the [item][KP]
// layouts, mbarrier + 1-D bulk-copy (TMA) wrappers, approximate reciprocal.
#pragma once
#include "common.cuh"

namespace polee {
namespace {

// ---------------------------------------------------------------- load / store helpers
__device__ __forceinline__ uint32_t ld_stream_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float ld_stream_f32(const float *p) {
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}

template <int KP>
struct Vec;
template <>
struct Vec<1> {
    static __device__ __forceinline__ void ld(const float *p, float *v) { v[0] = __ldg(p); }
    static __device__ __forceinline__ void st(float *p, const float *v) { p[0] = v[0]; }
};
template <>
struct Vec<2> {
    static __device__ __forceinline__ void ld(const float *p, float *v) {
        float2 t = __ldg(reinterpret_cast<const float2 *>(p));
        v[0] = t.x; v[1] = t.y;
    }
    static __device__ __forceinline__ void st(float *p, const float *v) {
        *reinterpret_cast<float2 *>(p) = make_float2(v[0], v[1]);
    }
};
template <>
struct Vec<4> {
    static __device__ __forceinline__ void ld(const float *p, float *v) {
        float4 t = __ldg(reinterpret_cast<const float4 *>(p));
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    }
    static __device__ __forceinline__ void st(float *p, const float *v) {
        *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
    }
};
template <>
struct Vec<8> {
    // one 256-bit request per lane (sm_100: LDG.E.ENL2.256): a whole 32-byte sector per entry
    static __device__ __forceinline__ void ld(const float *p, float *v) {
        asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
                     : "l"(p));
    }
    static __device__ __forceinline__ void st(float *p, const float *v) {
        asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]),
                     "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
                     : "memory");
    }
};
template <>
struct Vec<16> {
    static __device__ __forceinline__ void ld(const float *p, float *v) {
        Vec<8>::ld(p, v);
        Vec<8>::ld(p + 8, v + 8);
    }
    static __device__ __forceinline__ void st(float *p, const float *v) {
        Vec<8>::st(p, v);
        Vec<8>::st(p + 8, v + 8);
    }
};

// ---------------------------------------------------------------- mbarrier / bulk copy
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void consumer_bar_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// ---------------------------------------------------------------- programmatic dependent launch
// A kernel launched through launch_pdl (common.cuh) may start while the kernel before it on the stream is still running;
// pdl_wait() returns once that kernel has completed and its writes are visible.  The rule every such kernel follows:
//   - before pdl_wait() it reads only data that no kernel of the step loop writes: layouts, node records, schedules,
//     unit / task descriptors, the class blob, the seed and its arguments;
//   - x, ys, us, g, the partial sums, S, the StepCtl counters, the parameters and the ADAM state are read only after it,
//     and every write to global memory comes after it;
//   - every CTA executes pdl_wait(), on paths that exit early and write nothing too: a kernel's completion must still
//     imply the completion of every kernel before it, or a chain of early launches could run ahead of a kernel two
//     launches back.
// pdl_trigger() lets the next kernel's CTAs be scheduled once every CTA of this one has triggered or exited; it orders
// nothing, so where it stands is a matter of speed only.  Both are no-ops in a kernel launched without the attribute.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

__device__ __forceinline__ float rcp_approx(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

}  // namespace
}  // namespace polee
