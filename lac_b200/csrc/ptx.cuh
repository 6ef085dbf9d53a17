// ptx.cuh -- PTX helpers shared by the kernels: mbarrier / TMA bulk copies (SASS: UBLKCP, SYNCS), packed fp32x2
// math (FFMA2 / FADD2), warp collectives (REDUX where possible).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "lq32.cuh"

namespace lac {

// ------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ uint64_t evict_first_policy() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
// 1-D bulk copy global -> shared, completion counted in bytes on `bar` (SASS: UBLKCP)
__device__ __forceinline__ void tma_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t pol) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
        : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_acq_rel_cta() { asm volatile("fence.acq_rel.cta;" ::: "memory"); }

__device__ __forceinline__ float ldg_stream1(const float* p) {
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}

// ------------------------------------------------------------------ packed fp32x2 (FADD2 / FFMA2)
__device__ __forceinline__ uint64_t pk2(float a, float b) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ void upk2(uint64_t v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ uint64_t sub2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}

// Two elements per instruction (FFMA2 / FADD2), exactly lq::q_of's operations (explicit FMAs: ptxas
// contracts packed mul+add pairs on its own, so the spec fuses them by definition):
// FFMA2, FADD2, FFMA2, 3 x FFMA2 per pair, then sub / shl / funnel-shift per element.  No F2I.
__device__ __forceinline__ void q_of2(float xa, float xb, uint32_t nref, uint32_t& qa, uint32_t& qb) {
    const uint64_t L2 = pk2(lq::log2e(), lq::log2e());
    const uint64_t MG = pk2(lq::magic(), lq::magic());
    const uint64_t MZ = pk2(lq::magicz(), lq::magicz());
    const uint64_t x2 = pk2(xa, xb);
    uint64_t t = fma2(x2, L2, MG);
    uint64_t rn = sub2(MG, t);
    uint64_t f = fma2(x2, L2, rn);
    uint64_t p = pk2(__uint_as_float(lq::kC3), __uint_as_float(lq::kC3));
    p = fma2(p, f, pk2(__uint_as_float(lq::kC2), __uint_as_float(lq::kC2)));
    p = fma2(p, f, pk2(__uint_as_float(lq::kC1), __uint_as_float(lq::kC1)));
    uint64_t z = fma2(p, f, MZ);
    float za, zb, ta, tb;
    upk2(z, za, zb);
    upk2(t, ta, tb);
    qa = __funnelshift_rc(__float_as_uint(za) << 7, 0u, nref - __float_as_uint(ta));
    qb = __funnelshift_rc(__float_as_uint(zb) << 7, 0u, nref - __float_as_uint(tb));
}

// ------------------------------------------------------------------ warp collectives (REDUX where possible)
__device__ __forceinline__ int f2ord(float f) {  // order-preserving float -> int (no NaNs reach here)
    int b = __float_as_int(f);
    return b ^ ((b >> 31) & 0x7fffffff);
}
__device__ __forceinline__ float ord2f(int o) { return __int_as_float(o ^ ((o >> 31) & 0x7fffffff)); }
// sum over the warp of values < 2^48: three 16-bit limbs through REDUX.SUM
__device__ __forceinline__ uint64_t warp_sum48(uint64_t v) {
    uint32_t a = __reduce_add_sync(0xffffffffu, (uint32_t)v & 0xffffu);
    uint32_t b = __reduce_add_sync(0xffffffffu, (uint32_t)(v >> 16) & 0xffffu);
    uint32_t c = __reduce_add_sync(0xffffffffu, (uint32_t)(v >> 32));
    return (uint64_t)a + ((uint64_t)b << 16) + ((uint64_t)c << 32);
}
__device__ __forceinline__ uint64_t warp_incl_scan(uint64_t v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint64_t t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
    }
    return v;
}


}  // namespace lac
