// model_kernels.cu -- batch-invariant Llama kernels (include/lac_b200.h section (e)): GEMM on tcgen05 with the
// accumulator in tensor memory, RMSNorm, RoPE + KV-cache write, SwiGLU and GQA attention over the KV cache.
//
// The bits of output row r depend only on row r's inputs, the weights and (attention) the KV cache up to the row's
// position -- never on M, on how many query positions a launch covers, or on which CTA or tile row computes it:
//   * GEMM: tile 128 x 128 x 64 with a 3-stage ring; launches of M <= 128 whose 64-wide N tiles fit one wave use
//     128 x 64 x 64 tiles with an 8-stage ring (twice the CTAs, more weight bytes in flight).  K walked from 0
//     upwards in one accumulator, no split-K, no atomics.  A row's MMAs read its own A row and the same B columns in
//     the same K order whatever M is; that a 128 x 64 MMA gives an element the bits of the 128 x 128 one is checked
//     on the B200 (tests/test_gpu_any_batch.py).
//   * RMSNorm: one warp per row, a fixed per-lane order over the row, then a fixed xor butterfly.
//   * RoPE / SwiGLU: elementwise.
//   * attention: every query visits 64-key blocks from slot 0 upwards with an fp32 online softmax (exp2); a block
//     that lies wholly past a query's position is SKIPPED PER ROW (its (m, l, acc) are kept by a select), so a
//     query's result is the same whether its tile reaches further or not.
#include <cstdint>
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "launch.h"
#include "ptx.cuh"

namespace lac {
namespace {

constexpr int kBM = 128, kBN = 128, kBK = 64, kStages = 3;
constexpr int kSmallBN = 64, kSmallStages = 8;   // launches of M <= kBM: one tile row, so more and deeper N tiles
constexpr int kTileA = kBM * kBK * 2;            // bytes
constexpr int kAtomB = kBK * 64 * 2;             // one 64 x 64 B atom (64 columns of the 128-byte swizzle), bytes
template <int BN> __host__ __device__ constexpr int tile_b() { return kBK * BN * 2; }
template <int BN, int STAGES>  // + 1024-byte alignment slack
__host__ __device__ constexpr int gemm_smem() { return STAGES * (kTileA + tile_b<BN>()) + 1024; }
static_assert(gemm_smem<kSmallBN, kSmallStages>() <= 227 * 1024, "small-M ring exceeds the shared-memory limit");

// ------------------------------------------------------------------ tcgen05 / TMA helpers
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
// shared-memory matrix descriptor, 128-byte swizzle (start, leading and stride byte offsets >> 4)
__device__ __forceinline__ uint64_t sdesc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) |
           ((uint64_t)((sbo >> 4) & 0x3FFF) << 32) | (1ull << 46) | (2ull << 61);
}
// kind::f16 instruction descriptor: D fp32, A and B bf16, A K-major, B MN-major (W is [K, N] row-major), M x BN
template <int BN>
__host__ __device__ constexpr uint32_t idesc() {
    return (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(kBM >> 4) << 24);
}

template <int BN>
__device__ __forceinline__ void umma(uint32_t tmem, uint64_t a, uint64_t b, uint32_t accum) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem),
        "l"(a), "l"(b), "r"(idesc<BN>()), "r"(accum));
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float2 unpack_bf16(uint32_t v) {
    __nv_bfloat162 h = *reinterpret_cast<__nv_bfloat162*>(&v);
    return __bfloat1622float2(h);
}

// ------------------------------------------------------------------ GEMM  Y[M, N] = X[M, K] @ W[K, N]
// 128 threads: thread 0 feeds the smem ring by TMA, thread 32 issues the MMAs, warp 2 owns the tensor memory; then
// the four warps drain the 128 x BN fp32 accumulator (warp w: TMEM lanes = tile rows 32w .. 32w + 31).
template <int EPI, int BN, int STAGES>
__global__ void __launch_bounds__(128) gemm_kernel(const __grid_constant__ CUtensorMap ma,
                                                   const __grid_constant__ CUtensorMap mb, int64_t M, int N, int K,
                                                   const __nv_bfloat16* __restrict__ res, void* __restrict__ y) {
    constexpr int kTileB = tile_b<BN>(), kStage = kTileA + kTileB;
    extern __shared__ uint8_t dsm[];
    __shared__ uint64_t full[STAGES], empty[STAGES], done;
    __shared__ uint32_t tmem_slot;
    uint8_t* ring = (uint8_t*)(((uintptr_t)dsm + 1023) & ~(uintptr_t)1023);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * BN;
    const int m0 = blockIdx.y * kBM;
    const int nk = K / kBK;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        mbar_init(&done, 1);
        fence_mbar_init();
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)),
                     "r"(BN)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;

    if (threadIdx.x == 0) {  // producer
        for (int kb = 0; kb < nk; ++kb) {
            const int s = kb % STAGES;
            if (kb >= STAGES) mbar_wait(&empty[s], ((kb / STAGES) - 1) & 1);
            uint8_t* a = ring + s * kStage;
            uint8_t* b = a + kTileA;
            mbar_expect_tx(&full[s], kStage);
            tma_load_2d(a, &ma, kb * kBK, m0, &full[s]);
#pragma unroll
            for (int j = 0; j < BN / 64; ++j) tma_load_2d(b + j * kAtomB, &mb, n0 + 64 * j, kb * kBK, &full[s]);
        }
    } else if (threadIdx.x == 32) {  // MMA issuer
        for (int kb = 0; kb < nk; ++kb) {
            const int s = kb % STAGES;
            mbar_wait(&full[s], (kb / STAGES) & 1);
            tc_fence_after();
            const uint32_t a = smem_u32(ring + s * kStage), b = a + kTileA;
#pragma unroll
            for (int k = 0; k < kBK / 16; ++k) {
                // A: K-major, 8-row groups 1024 B apart, +32 B per 16 K.  B: MN-major, 64-column atoms 8 KB apart,
                // 8-K-row groups 1024 B apart, +2048 B per 16 K.
                umma<BN>(tmem, sdesc(a + k * 32, 16, 1024), sdesc(b + k * 2048, kAtomB, 1024), (kb | k) != 0);
            }
            umma_commit(&empty[s]);
        }
        umma_commit(&done);
    }
    __syncwarp();

    mbar_wait(&done, 0);
    tc_fence_after();
    const int64_t row = (int64_t)m0 + warp * 32 + lane;
    const bool live = row < M;
#pragma unroll 1
    for (int c = 0; c < BN; c += 16) {
        uint32_t r[16];
        tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + c, r);
        if (!live) continue;
        const int64_t off = row * N + n0 + c;
        if (EPI == LAC_MODEL_OUT_F32) {
            float4* dst = reinterpret_cast<float4*>((float*)y + off);
#pragma unroll
            for (int i = 0; i < 4; ++i)
                dst[i] = make_float4(__uint_as_float(r[4 * i]), __uint_as_float(r[4 * i + 1]),
                                     __uint_as_float(r[4 * i + 2]), __uint_as_float(r[4 * i + 3]));
        } else {
            uint32_t o[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) o[i] = pack_bf16(__uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1]));
            if (EPI == LAC_MODEL_OUT_BF16_ADD) {  // x + bf16(o @ w), rounded once more: what the bf16 torch op does
                const uint4* rp = reinterpret_cast<const uint4*>(res + off);
                uint4 q0 = rp[0], q1 = rp[1];
                const uint32_t rv[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    float2 a = unpack_bf16(o[i]), b = unpack_bf16(rv[i]);
                    o[i] = pack_bf16(b.x + a.x, b.y + a.y);
                }
            }
            uint4* dst = reinterpret_cast<uint4*>((__nv_bfloat16*)y + off);
            dst[0] = make_uint4(o[0], o[1], o[2], o[3]);
            dst[1] = make_uint4(o[4], o[5], o[6], o[7]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(BN) : "memory");
}

typedef CUresult (*EncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiled encode_tiled() {
    static EncodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &p, 12000, cudaEnableDefault, &q) ==
                cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiled)p;
    }
    return fn;
}

// 2-D bf16 row-major tensor [outer, inner], box [box_outer, 64] with the 128-byte swizzle; rows past `outer` read 0
bool make_map(CUtensorMap* m, const void* p, int64_t inner, int64_t outer, uint32_t box_outer) {
    EncodeTiled fn = encode_tiled();
    if (!fn) return false;
    cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
    cuuint64_t strides[1] = {(cuuint64_t)inner * 2};
    cuuint32_t box[2] = {64, box_outer};
    cuuint32_t es[2] = {1, 1};
    return fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(p), dims, strides, box, es,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int EPI, int BN, int STAGES>
cudaError_t gemm_launch(const CUtensorMap& ma, const CUtensorMap& mb, int64_t M, int N, int K, const void* res,
                        void* y, cudaStream_t st) {
    constexpr int smem = gemm_smem<BN, STAGES>();
    static bool attr = false;
    if (!attr) {
        cudaError_t e =
            cudaFuncSetAttribute(gemm_kernel<EPI, BN, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        attr = true;
    }
    dim3 grid(N / BN, (unsigned)((M + kBM - 1) / kBM));
    gemm_kernel<EPI, BN, STAGES><<<grid, 128, smem, st>>>(ma, mb, M, N, K, (const __nv_bfloat16*)res, y);
    return cudaGetLastError();
}

int sm_count() {
    static int n = 0;
    if (!n) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) !=
                                                      cudaSuccess)
            n = 1;
    }
    return n;
}

// M <= 128 is one tile row, so a 128-wide N tile leaves N / 128 CTAs (16 for a 2048-wide weight) each walking all of
// K: the step is bound by the weight loads those few SMs keep in flight.  64-wide tiles double the CTAs and the
// 8-stage ring keeps 8 K-steps of each in flight -- as long as they fit one wave: past the SM count (w13 and the
// head of `1b`) the 197 KB ring allows one CTA per SM against two of the 3-stage one, and the wide tile is faster.
// A row gets the same bits from either tile.
template <int EPI>
cudaError_t gemm_dispatch(const CUtensorMap& ma, const CUtensorMap& mb, int64_t M, int N, int K, const void* res,
                          void* y, cudaStream_t st) {
    if (M <= kBM && N / kSmallBN <= sm_count())
        return gemm_launch<EPI, kSmallBN, kSmallStages>(ma, mb, M, N, K, res, y, st);
    return gemm_launch<EPI, kBN, kStages>(ma, mb, M, N, K, res, y, st);
}

// ------------------------------------------------------------------ RMSNorm: one warp per row
__global__ void __launch_bounds__(256) rmsnorm_kernel(const __nv_bfloat16* __restrict__ x, int64_t rows, int dim,
                                                      float eps, __nv_bfloat16* __restrict__ y) {
    const int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= rows) return;
    const uint4* xr = reinterpret_cast<const uint4*>(x + r * dim);
    float ss = 0.f;
    for (int i = lane; i < dim / 8; i += 32) {
        uint4 v = xr[i];
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float2 f = unpack_bf16(w[j]);
            ss = fmaf(f.x, f.x, ss);
            ss = fmaf(f.y, f.y, ss);
        }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    const float rs = rsqrtf(ss / (float)dim + eps);
    uint4* yr = reinterpret_cast<uint4*>(y + r * dim);
    for (int i = lane; i < dim / 8; i += 32) {
        uint4 v = xr[i];
        uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float2 f = unpack_bf16(w[j]);
            w[j] = pack_bf16(f.x * rs, f.y * rs);
        }
        yr[i] = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

// ------------------------------------------------------------------ RoPE (rotate-half) + KV-cache write
// Row r = t * S + s is stream s at position base + t (base = *d_pos when d_pos is given, else p0).  q and k are
// rotated in place in the qkv row; k and v are written to cache[s, kv_head, pos, :].
__global__ void rope_kv_kernel(__nv_bfloat16* __restrict__ qkv, int S, int H, int KV, int hd,
                               const __nv_bfloat16* __restrict__ cosb, const __nv_bfloat16* __restrict__ sinb,
                               const int64_t* __restrict__ d_pos, int64_t p0, __nv_bfloat16* __restrict__ kc,
                               __nv_bfloat16* __restrict__ vc, int max_len) {
    const int64_t r = blockIdx.x;
    const int s = (int)(r % S);
    const int64_t pos = (d_pos ? *d_pos : p0) + r / S;
    if (pos < 0 || pos >= max_len) return;
    __nv_bfloat16* row = qkv + r * (int64_t)(H + 2 * KV) * hd;
    const int half = hd / 2;
    const __nv_bfloat16* c = cosb + pos * hd;
    const __nv_bfloat16* sn = sinb + pos * hd;
    for (int i = threadIdx.x; i < (H + KV) * half; i += blockDim.x) {
        const int h = i / half, j = i % half;
        __nv_bfloat16* v = row + h * hd;
        const float x1 = __bfloat162float(v[j]), x2 = __bfloat162float(v[j + half]);
        const __nv_bfloat16 o1 = __float2bfloat16_rn(x1 * __bfloat162float(c[j]) - x2 * __bfloat162float(sn[j]));
        const __nv_bfloat16 o2 =
            __float2bfloat16_rn(x2 * __bfloat162float(c[j + half]) + x1 * __bfloat162float(sn[j + half]));
        v[j] = o1;
        v[j + half] = o2;
        if (h >= H) {
            const int64_t at = (((int64_t)s * KV + (h - H)) * max_len + pos) * hd;
            kc[at + j] = o1;
            kc[at + j + half] = o2;
        }
    }
    for (int i = threadIdx.x; i < KV * hd; i += blockDim.x) {
        const int h = i / hd, j = i % hd;
        vc[(((int64_t)s * KV + h) * max_len + pos) * hd + j] = row[(H + KV) * hd + i];
    }
}

// ------------------------------------------------------------------ SwiGLU: y = bf16(silu(a)) * b, a | b = h[:, :F] | h[:, F:]
__global__ void swiglu_kernel(const __nv_bfloat16* __restrict__ h, int64_t rows, int F, __nv_bfloat16* __restrict__ y) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * F) return;
    const int64_t r = i / F, j = i % F;
    const float a = __bfloat162float(h[r * 2 * F + j]), b = __bfloat162float(h[r * 2 * F + F + j]);
    const float sa = __bfloat162float(__float2bfloat16_rn(a / (1.f + expf(-a))));
    y[i] = __float2bfloat16_rn(sa * b);
}

// ------------------------------------------------------------------ attention
// Grid (ceil(n_q * G / 64), kv_heads, S), G = heads / kv_heads.  A CTA's 64 rows are (query t, group head g),
// j = t * G + g, 16 per warp (mma.sync m16n8k16).  Every 64-key block from slot 0 up to the CTA's furthest position
// is staged in shared memory; each row folds in the blocks that start at or before its own position, and keeps its
// (m, l, acc) unchanged (a select, not arithmetic) for the others.
constexpr int kKB = 64;

__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
        "{%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

template <int HD>
__global__ void __launch_bounds__(128) attn_kernel(const __nv_bfloat16* __restrict__ qkv, int S, int n_q, int H,
                                                   int KV, const int64_t* __restrict__ d_pos, int64_t p0,
                                                   const __nv_bfloat16* __restrict__ kc,
                                                   const __nv_bfloat16* __restrict__ vc, int max_len,
                                                   __nv_bfloat16* __restrict__ out) {
    constexpr int KS = HD + 8, VS = kKB + 8;  // padded smem rows: conflict-free 32-bit fragment loads
    __shared__ __align__(16) __nv_bfloat16 Ks[kKB * KS];
    __shared__ __align__(16) __nv_bfloat16 Vt[HD * VS];
    const int G = H / KV;
    const int kvh = blockIdx.y, s = blockIdx.z;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, qd = lane & 3, gr = lane >> 2;
    const int64_t base = d_pos ? *d_pos : p0;
    const int rows = n_q * G;
    const int j0 = blockIdx.x * 64 + warp * 16 + gr;
    const int jr[2] = {j0, j0 + 8};
    int64_t pos[2];
    const __nv_bfloat16* qrow[2];
    const int64_t qkv_w = (int64_t)(H + 2 * KV) * HD;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const bool ok = jr[h] < rows;
        const int t = ok ? jr[h] / G : 0, g = ok ? jr[h] % G : 0;
        pos[h] = ok ? base + t : -1;
        qrow[h] = qkv + ((int64_t)t * S + s) * qkv_w + (int64_t)(kvh * G + g) * HD;
    }
    uint32_t qf[HD / 16][4];
#pragma unroll
    for (int ks = 0; ks < HD / 16; ++ks) {
        const int c = ks * 16 + 2 * qd;
        qf[ks][0] = pos[0] >= 0 ? *reinterpret_cast<const uint32_t*>(qrow[0] + c) : 0u;
        qf[ks][1] = pos[1] >= 0 ? *reinterpret_cast<const uint32_t*>(qrow[1] + c) : 0u;
        qf[ks][2] = pos[0] >= 0 ? *reinterpret_cast<const uint32_t*>(qrow[0] + c + 8) : 0u;
        qf[ks][3] = pos[1] >= 0 ? *reinterpret_cast<const uint32_t*>(qrow[1] + c + 8) : 0u;
    }
    const int last_j = min(rows - 1, (int)blockIdx.x * 64 + 63);
    const int64_t cta_max = base + last_j / G;
    const int warp_last = min(rows - 1, (int)blockIdx.x * 64 + warp * 16 + 15);
    const int64_t warp_max = blockIdx.x * 64 + warp * 16 < rows ? base + warp_last / G : -1;
    const float sl2 = 1.4426950408889634f * rsqrtf((float)HD);

    float m[2] = {-INFINITY, -INFINITY}, l[2] = {0.f, 0.f};
    float acc[HD / 8][4];
#pragma unroll
    for (int i = 0; i < HD / 8; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;

    const __nv_bfloat16* kbase = kc + ((int64_t)s * KV + kvh) * max_len * HD;
    const __nv_bfloat16* vbase = vc + ((int64_t)s * KV + kvh) * max_len * HD;
    const int nblk = (int)(min(cta_max, (int64_t)max_len - 1) / kKB) + 1;
    for (int b = 0; b < nblk; ++b) {
        __syncthreads();
        for (int i = threadIdx.x; i < kKB * HD / 8; i += 128) {
            const int key = i / (HD / 8), d8 = (i % (HD / 8)) * 8;
            const int64_t kk = (int64_t)b * kKB + key;
            uint4 kv = make_uint4(0, 0, 0, 0), vv = make_uint4(0, 0, 0, 0);
            if (kk < max_len) {
                kv = *reinterpret_cast<const uint4*>(kbase + kk * HD + d8);
                vv = *reinterpret_cast<const uint4*>(vbase + kk * HD + d8);
            }
            *reinterpret_cast<uint4*>(&Ks[key * KS + d8]) = kv;
            const __nv_bfloat16* ve = reinterpret_cast<const __nv_bfloat16*>(&vv);
#pragma unroll
            for (int e = 0; e < 8; ++e) Vt[(d8 + e) * VS + key] = ve[e];
        }
        __syncthreads();
        if (warp_max < (int64_t)b * kKB) continue;  // every row of this warp skips the block: nothing changes

        float sc[kKB / 8][4];
#pragma unroll
        for (int nt = 0; nt < kKB / 8; ++nt) {
            sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
#pragma unroll
            for (int ks = 0; ks < HD / 16; ++ks) {
                const __nv_bfloat16* kr = &Ks[(nt * 8 + gr) * KS + ks * 16 + 2 * qd];
                mma16816(sc[nt], qf[ks], *reinterpret_cast<const uint32_t*>(kr),
                         *reinterpret_cast<const uint32_t*>(kr + 8));
            }
        }
        float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
        for (int nt = 0; nt < kKB / 8; ++nt)
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int h = e >> 1;
                const int64_t key = (int64_t)b * kKB + nt * 8 + 2 * qd + (e & 1);
                const float v = key <= pos[h] ? sc[nt][e] * sl2 : -INFINITY;
                sc[nt][e] = v;
                mx[h] = fmaxf(mx[h], v);
            }
        float mn[2], alpha[2], ls[2] = {0.f, 0.f};
        bool take[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            mx[h] = fmaxf(mx[h], __shfl_xor_sync(0xffffffffu, mx[h], 1));
            mx[h] = fmaxf(mx[h], __shfl_xor_sync(0xffffffffu, mx[h], 2));
            take[h] = pos[h] >= (int64_t)b * kKB;
            mn[h] = fmaxf(m[h], mx[h]);
            alpha[h] = exp2f(m[h] - mn[h]);
        }
        uint32_t pf[kKB / 16][4];
#pragma unroll
        for (int nt = 0; nt < kKB / 8; ++nt) {
            const float p0_ = exp2f(sc[nt][0] - mn[0]), p1_ = exp2f(sc[nt][1] - mn[0]);
            const float p2_ = exp2f(sc[nt][2] - mn[1]), p3_ = exp2f(sc[nt][3] - mn[1]);
            ls[0] += p0_ + p1_;
            ls[1] += p2_ + p3_;
            pf[nt >> 1][(nt & 1) * 2 + 0] = pack_bf16(p0_, p1_);
            pf[nt >> 1][(nt & 1) * 2 + 1] = pack_bf16(p2_, p3_);
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            ls[h] += __shfl_xor_sync(0xffffffffu, ls[h], 1);
            ls[h] += __shfl_xor_sync(0xffffffffu, ls[h], 2);
            if (take[h]) {
                m[h] = mn[h];
                l[h] = fmaf(l[h], alpha[h], ls[h]);
            }
        }
#pragma unroll
        for (int half = 0; half < HD / 64; ++half) {
            float ob[8][4];
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                ob[nt][0] = ob[nt][1] = ob[nt][2] = ob[nt][3] = 0.f;
#pragma unroll
                for (int ks = 0; ks < kKB / 16; ++ks) {
                    const __nv_bfloat16* vr = &Vt[(half * 64 + nt * 8 + gr) * VS + ks * 16 + 2 * qd];
                    mma16816(ob[nt], pf[ks], *reinterpret_cast<const uint32_t*>(vr),
                             *reinterpret_cast<const uint32_t*>(vr + 8));
                }
            }
#pragma unroll
            for (int nt = 0; nt < 8; ++nt)
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int h = e >> 1;
                    float& a = acc[half * 8 + nt][e];
                    a = take[h] ? fmaf(a, alpha[h], ob[nt][e]) : a;
                }
        }
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        if (pos[h] < 0) continue;
        const int t = jr[h] / G, g = jr[h] % G;
        __nv_bfloat16* orow = out + ((int64_t)t * S + s) * H * HD + (int64_t)(kvh * G + g) * HD;
        const float inv = 1.f / l[h];
#pragma unroll
        for (int nt = 0; nt < HD / 8; ++nt)
            *reinterpret_cast<uint32_t*>(orow + nt * 8 + 2 * qd) =
                pack_bf16(acc[nt][2 * h] * inv, acc[nt][2 * h + 1] * inv);
    }
}

}  // namespace

bool model_gemm_shape_ok(int64_t M, int N, int K) { return M >= 1 && N >= kBN && N % kBN == 0 && K >= kBK && K % kBK == 0; }

cudaError_t launch_model_gemm(const void* x, const void* w, int64_t M, int N, int K, int epi, const void* res, void* y,
                              cudaStream_t st) {
    CUtensorMap ma, mb;
    if (!make_map(&ma, x, K, M, kBM) || !make_map(&mb, w, N, K, kBK)) return cudaErrorInvalidValue;
    switch (epi) {
        case LAC_MODEL_OUT_BF16: return gemm_dispatch<LAC_MODEL_OUT_BF16>(ma, mb, M, N, K, res, y, st);
        case LAC_MODEL_OUT_BF16_ADD: return gemm_dispatch<LAC_MODEL_OUT_BF16_ADD>(ma, mb, M, N, K, res, y, st);
        default: return gemm_dispatch<LAC_MODEL_OUT_F32>(ma, mb, M, N, K, res, y, st);
    }
}

cudaError_t launch_model_rmsnorm(const void* x, int64_t rows, int dim, float eps, void* y, cudaStream_t st) {
    rmsnorm_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>((const __nv_bfloat16*)x, rows, dim, eps,
                                                               (__nv_bfloat16*)y);
    return cudaGetLastError();
}

cudaError_t launch_model_rope_kv(void* qkv, int64_t rows, int S, int H, int KV, int hd, const void* cosb,
                                 const void* sinb, const int64_t* d_pos, int64_t p0, void* kc, void* vc, int max_len,
                                 cudaStream_t st) {
    rope_kv_kernel<<<(unsigned)rows, 128, 0, st>>>((__nv_bfloat16*)qkv, S, H, KV, hd, (const __nv_bfloat16*)cosb,
                                                   (const __nv_bfloat16*)sinb, d_pos, p0, (__nv_bfloat16*)kc,
                                                   (__nv_bfloat16*)vc, max_len);
    return cudaGetLastError();
}

cudaError_t launch_model_swiglu(const void* h, int64_t rows, int F, void* y, cudaStream_t st) {
    const int64_t n = rows * F;
    swiglu_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const __nv_bfloat16*)h, rows, F, (__nv_bfloat16*)y);
    return cudaGetLastError();
}

cudaError_t launch_model_attention(const void* qkv, int S, int n_q, int H, int KV, int hd, const int64_t* d_pos,
                                   int64_t p0, const void* kc, const void* vc, int max_len, void* out,
                                   cudaStream_t st) {
    dim3 grid((unsigned)(((int64_t)n_q * (H / KV) + 63) / 64), KV, S);
    const __nv_bfloat16 *q = (const __nv_bfloat16*)qkv, *k = (const __nv_bfloat16*)kc, *v = (const __nv_bfloat16*)vc;
    if (hd == 64)
        attn_kernel<64><<<grid, 128, 0, st>>>(q, S, n_q, H, KV, d_pos, p0, k, v, max_len, (__nv_bfloat16*)out);
    else
        attn_kernel<128><<<grid, 128, 0, st>>>(q, S, n_q, H, KV, d_pos, p0, k, v, max_len, (__nv_bfloat16*)out);
    return cudaGetLastError();
}

}  // namespace lac
