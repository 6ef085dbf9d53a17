// cdf_kernels.cu -- logits -> LQ32 CDF kernels (north-star part (a)).
//
// Both directions of the coder are ONE bandwidth-bound pass over the logits plus small dependent passes:
//
//   encode:  summary_kernel -> encode_fused_kernel (coder_kernels.cu: (lo, hi) of the coded symbols + range coder)
//   decode:  summary_kernel -> decode_serial_kernel (decode_kernels.cu: 1 warp / stream, walks its tokens)
//   tables:  summary_kernel -> table_kernel          (lac_cdf_build_f32, the calc_dist drop-in)
//
// summary_kernel: one persistent CTA of 1024 threads per SM walks TILES: a tile is one part of one row (at most
// 32768 elements = 32 warp segments); rows wider than that are simply several tiles, dealt round-robin to all SMs
// like everything else (LQ32's block form, lq32.cuh, has no row-wide dependency in this pass: no cluster, no DSMEM).
// Warp w owns segment w of the tile; the tile is read from HBM exactly once and then lives in registers:
//
//   staging  the tile arrives as 4 TMA bulk copies of 32 KB (cp.async.bulk) into a shared-memory ring, each
//            chunk with its own mbarrier; the warps of a chunk move it to registers.  Rows that are not 16-byte
//            aligned or have V % 4 != 0 take scalar loads instead (summary_kernel<1>: no ring, no barrier).
//   phase A  segment maximum (REDUX) and the ONE barrier of the tile, whose only purpose is the ring: right after
//            it the chunk leaders re-arm their mbarriers and issue the bulk copies of the CTA's NEXT tile, so
//            128 KB per SM are in flight during the compute phase.
//   phase B  q_i against the segment's own reference with packed fp32x2 math (FADD2 / FFMA2), exact integer sums
//   finish   lane 0 of every warp stores ONE word {segment sum, reference code}: 256 bytes per 128 KB tile.
//            No counter, no finishing warp, no scan, no division, no table.
//
// The second passes work from the summary words and re-read only the one segment (<= 4 KB) they need (rowsum.cuh).
#include <climits>
#include <cstdint>
#include <cstdlib>
#include <cuda_runtime.h>

#include "launch.h"
#include "lq32.cuh"
#include "ptx.cuh"
#include "rowsum.cuh"

namespace lac {

// A tile is one part of a row: 32 consecutive segments, one per warp of a CTA of 1024 threads, one CTA per SM.
// It arrives as 4 TMA chunks of 8 warps (32 KB).  Measured on B200 (profiles/microbench/tma_stream.cu): every
// cp.async.bulk costs ~0.2 us of per-SM TMA time regardless of size, so 16 KB chunks cap at 4.7 TB/s while 32 and
// 64 KB chunks reach 7.1 - 7.2 TB/s with the same 128 KB in flight per SM; 4 x 32 KB is 0.7 % faster than 2 x 64 KB.
constexpr int kTileWarps = 32;
constexpr int kChunks = 4;
constexpr int kWarpsPerChunk = kTileWarps / kChunks;
constexpr int kSlotGroups = kPerThread / 4 * 32 * kWarpsPerChunk + 1;  // float4 groups per slot
constexpr int kSlotBytes = kSlotGroups * 16;
constexpr int kRingBytes = kChunks * kSlotBytes;

// Everything the pass needs to find tile `tau`: row rho = tau / parts (row (s, t) = (rho / T, rho % T) at
// base + s * so + t * st), first segment (tau % parts) * 32.  Lives in the kernel-parameter constant bank.
struct SumParams {
    const float* base;
    int64_t so, st;
    uint32_t T, n_tiles;
    int V, G, parts;
    uint32_t inv_parts;  // ceil(2^31 / parts): floor(m / parts) = (m * inv_parts) >> 31 for m * parts < 2^31
    int keep_l2;         // 0: stream with evict-first (the logits are read once); 1: leave them in L2 for a second pass
};

__shared__ uint64_t g_full[kChunks];  // TMA chunk landed
__shared__ int g_red[2][kTileWarps];  // per-warp maxima, written before the tile's barrier (see tile())
extern __shared__ __align__(128) unsigned char g_ring[];

// VEC = 4: the TMA ring (rows 16-byte aligned, V % 4 == 0); VEC = 1: scalar loads straight to registers.
template <int VEC>
struct TileEngine {
    static constexpr bool kTma = VEC == 4;
    static constexpr int IT = kPerThread / VEC;

    static __device__ __forceinline__ int warp() { return threadIdx.x >> 5; }
    static __device__ __forceinline__ int lane() { return threadIdx.x & 31; }
    static __device__ __forceinline__ int chunk() { return warp() / kWarpsPerChunk; }
    static __device__ __forceinline__ bool leader() { return (threadIdx.x & (32 * kWarpsPerChunk - 1)) == 0; }
    static __device__ __forceinline__ unsigned char* slot() { return g_ring + chunk() * kSlotBytes; }
    // first 4-element group of row-wide segment gw (lq::seg_group with a run-time number of parts)
    static __device__ __forceinline__ int seg(const SumParams& sp, int gw) {
        const uint32_t m = ((uint32_t)gw * (uint32_t)sp.G) >> 5;
        return (int)(((uint64_t)m * sp.inv_parts) >> 31);
    }
    static __device__ __forceinline__ uint32_t row_index(const SumParams& sp, uint32_t tau) {
        return (uint32_t)(((uint64_t)tau * sp.inv_parts) >> 31);
    }
    // first row-wide segment of tile tau
    static __device__ __forceinline__ int seg0_of(const SumParams& sp, uint32_t tau) {
        return (int)(tau - row_index(sp, tau) * (uint32_t)sp.parts) * kTileWarps;
    }
    static __device__ __forceinline__ const float* row_of(const SumParams& sp, uint32_t tau) {
        const uint32_t rho = row_index(sp, tau);
        const uint32_t s = rho / sp.T, t = rho - s * sp.T;
        return sp.base + (int64_t)s * sp.so + (int64_t)t * sp.st;
    }

    static __device__ void setup() {
        if (threadIdx.x == 0) {
            for (int i = 0; i < kChunks; i++) mbar_init(&g_full[i], 1);
            fence_mbar_init();
        }
        __syncthreads();
    }
    // chunk leader: arm the chunk's mbarrier and issue its bulk copy for tile tau
    static __device__ __forceinline__ void issue(const SumParams& sp, uint32_t tau) {
        if (kTma && leader()) {
            const int gw0 = seg0_of(sp, tau) + chunk() * kWarpsPerChunk;
            const int g0 = seg(sp, gw0);
            const uint32_t nb = (uint32_t)(seg(sp, gw0 + kWarpsPerChunk) - g0) * 16u;
            if (nb) {
                mbar_expect_tx(&g_full[chunk()], nb);
                uint64_t pol;
                if (!sp.keep_l2) pol = evict_first_policy();
                else asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol));
                tma_load_1d(slot(), row_of(sp, tau) + 4 * (int64_t)g0, nb, &g_full[chunk()], pol);
            }
        }
    }

    // One tile: stage it into registers, segment maximum, the tile's single block barrier (after which the ring is
    // re-armed with the CTA's next tile), q against the segment's reference, segment sum -> one summary word.
    static __device__ __forceinline__ void tile(const SumParams& sp, uint32_t tau, uint32_t it,
                                                uint64_t* __restrict__ summ) {
        float x[kPerThread];
        {
            const int s0 = seg0_of(sp, tau);
            const int gw = s0 + warp();
            const int gb = seg(sp, gw), ge = seg(sp, gw + 1), ln = lane();
            if (kTma) {
                const int gw0 = s0 + chunk() * kWarpsPerChunk;
                const int c0 = seg(sp, gw0);
                if (seg(sp, gw0 + kWarpsPerChunk) > c0) mbar_wait(&g_full[chunk()], it & 1);
                const unsigned char* sl = slot() + (size_t)(gb + ln - c0) * 16;
                if (ge - gb > (IT - 1) * 32) {
                    // the usual shape (a segment longer than 7 slabs): slabs 0..6 are complete for every lane,
                    // no -inf initialisation and no predicates there (32 instructions per thread and tile less)
#pragma unroll
                    for (int k = 0; k < IT - 1; k++) {
                        const float4 v = *reinterpret_cast<const float4*>(sl + k * 512);
                        x[4 * k + 0] = v.x;
                        x[4 * k + 1] = v.y;
                        x[4 * k + 2] = v.z;
                        x[4 * k + 3] = v.w;
                    }
                    float4 v = make_float4(lq::neg_inf(), lq::neg_inf(), lq::neg_inf(), lq::neg_inf());
                    if (gb + (IT - 1) * 32 + ln < ge) v = *reinterpret_cast<const float4*>(sl + (IT - 1) * 512);
                    x[4 * (IT - 1) + 0] = v.x;
                    x[4 * (IT - 1) + 1] = v.y;
                    x[4 * (IT - 1) + 2] = v.z;
                    x[4 * (IT - 1) + 3] = v.w;
                } else {
#pragma unroll
                    for (int k = 0; k < IT; k++) {
                        float4 v = make_float4(lq::neg_inf(), lq::neg_inf(), lq::neg_inf(), lq::neg_inf());
                        if (gb + k * 32 + ln < ge) v = *reinterpret_cast<const float4*>(sl + k * 512);
                        x[4 * k + 0] = v.x;
                        x[4 * k + 1] = v.y;
                        x[4 * k + 2] = v.z;
                        x[4 * k + 3] = v.w;
                    }
                }
            } else {
                const float* row = row_of(sp, tau);
                const int e0 = 4 * gb, e1 = min(sp.V, 4 * ge);
#pragma unroll
                for (int k = 0; k < IT; k++) {
                    const int e = e0 + k * 32 + ln;
                    x[k] = e < e1 ? ldg_stream1(row + e) : lq::neg_inf();
                }
            }
        }
        // phase A: segment maximum (fmaxf drops NaNs; the running value starts at -inf, so it is never NaN)
        float m = lq::neg_inf();
#pragma unroll
        for (int i = 0; i < kPerThread; i++) m = fmaxf(m, x[i]);
        const int mw = __reduce_max_sync(0xffffffffu, f2ord(m));
        if (kTma) {
            // mw depends on every shared-memory load of the warp: storing it before the barrier means that after
            // the barrier the whole tile is in registers and the ring can be overwritten
            if (lane() == 0) *reinterpret_cast<volatile int*>(&g_red[it & 1][warp()]) = mw;
            __syncthreads();  // the only barrier of the tile
            if (leader()) {
                const uint32_t nt = tau + gridDim.x;
                if (nt < sp.n_tiles) {
                    fence_proxy_async();
                    issue(sp, nt);
                }
            }
        }
        // phase B against the segment's own reference
        const uint32_t code = lq::code_of_max(ord2f(mw));
        const uint32_t nref = lq::nref_of_code(code);
        uint64_t lane_sum = 0;
#pragma unroll
        for (int i = 0; i < kPerThread; i += 4) {
            uint32_t q0, q1, q2, q3;
            q_of2(x[i], x[i + 1], nref, q0, q1);
            q_of2(x[i + 2], x[i + 3], nref, q2, q3);
            lane_sum += (q0 + q1) + (q2 + q3);
        }
        const uint64_t ws = warp_sum48(lane_sum);
        if (lane() == 0) summ[(uint64_t)tau * kTileWarps + warp()] = lq::pack_word(ws, code);
    }
};

template <int VEC>
__global__ void __launch_bounds__(32 * kTileWarps, 1)
summary_kernel(const __grid_constant__ SumParams sp, uint64_t* __restrict__ summ) {
    using Eng = TileEngine<VEC>;
    if (Eng::kTma) Eng::setup();
    uint32_t tau = blockIdx.x;
    if (tau < sp.n_tiles) Eng::issue(sp, tau);
    for (uint32_t it = 0; tau < sp.n_tiles; tau += gridDim.x, it++) Eng::tile(sp, tau, it, summ);
}

// ------------------------------------------------------------------ LOOKUP (second pass of lac_cdf_lookup_f32)
// One warp per row, all rows independent (rowsum.cuh).  ~2 % extra HBM traffic.
// Row r = (s, t) = (r / T, r % T): logits at base + s * so + t * st, symbol at syms[s * sym_stride + t].
template <int VEC, int CL>
__global__ void __launch_bounds__(256)
pair_kernel(const float* __restrict__ logits, int64_t rows, int64_t T, int64_t so, int64_t st, int V,
            const uint64_t* __restrict__ summ, const int32_t* __restrict__ syms, int64_t sym_stride,
            uint32_t* __restrict__ pairs, uint32_t* __restrict__ status) {
    const int lane = threadIdx.x & 31;
    const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= rows) return;
    const int64_t s = r / T, t = r - s * T;
    const int sym = __ldg(syms + s * sym_stride + t);
    if (sym < 0 || sym >= V) {
        if (lane == 0) {
            // sentinel the coder turns into LAC_ST_SYMBOL on the stream (the reference raises "unknown symbol",
            // arith_code.py:100-101); never a silent no-op
            *reinterpret_cast<uint2*>(pairs + 2 * r) = make_uint2(0xFFFFFFFFu, 0xFFFFFFFFu);
            if (status) atomicOr(status + r, LAC_ST_SYMBOL);
        }
        return;
    }
    const uint2 o = warp_symbol_range<VEC, CL>(logits + s * so + t * st, V, summ + r * (32 * CL), sym, lane);
    if (lane == 0) *reinterpret_cast<uint2*>(pairs + 2 * r) = o;
}

// ------------------------------------------------------------------ TABLE (second pass of lac_cdf_build_f32)
// Full exclusive cumulative table: one warp per segment.  The logits are read a second time (from L2: the
// launcher keeps the row chunk small enough), the table is written once.  VEC = 4: slab k of the segment is the 32
// consecutive float4 groups g0 + 32 k + lane -- 512-byte coalesced loads and stores, one warp scan of the group sums
// per slab.  VEC = 1 (unaligned rows / V % 4 != 0): lane l walks 32 consecutive elements after one scan.
template <int VEC, int CL>
__global__ void __launch_bounds__(256)
table_kernel(const float* __restrict__ logits, int64_t rows, int64_t row_stride, int V,
             const uint64_t* __restrict__ summ, uint32_t* __restrict__ cum) {
    constexpr int NW = 32 * CL;
    const int lane = threadIdx.x & 31;
    const int64_t unit = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (unit >= rows * NW) return;
    const int64_t r = unit / NW;
    const int gw = (int)(unit - r * NW);
    const int G = lq::groups_of(V);
    const int gb = lq::seg_group<CL>(gw, G), ge = lq::seg_group<CL>(gw + 1, G);
    const int e0 = 4 * gb, e1 = min(V, 4 * ge);
    if (e0 >= e1) return;
    RowSum<CL> rs;
    rs.load(summ + r * NW, lane);
    rs.align();
    uint64_t front;
    const uint64_t Q = rs.total_and_front(gw, lane, front);
    const lq::Scale sc = lq::make_scale(Q, V);
    const uint32_t code = rs.code_of(gw);
    const int d = lq::shift_of(rs.r, code);
    const uint32_t nref = lq::nref_of_code(code);
    const float* row = logits + r * row_stride;
    uint32_t* out = cum + r * (int64_t)V;
    if (VEC == 4) {
        const bool out16 = (((uintptr_t)out) & 15) == 0;
        uint64_t c0 = 0;  // in-segment prefix at the start of the slab
#pragma unroll 1
        for (int k = 0; k < kPerThread / 4; k++) {
            if (gb + 32 * k >= ge) break;  // warp-uniform
            const int g = gb + 32 * k + lane;
            const bool in = g < ge;
            const float4 x = __ldg(reinterpret_cast<const float4*>(row) + (in ? g : ge - 1));
            uint32_t q[4];
            q_of2(x.x, x.y, nref, q[0], q[1]);
            q_of2(x.z, x.w, nref, q[2], q[3]);
            const uint64_t gs = in ? (uint64_t)q[0] + q[1] + (uint64_t)q[2] + q[3] : 0ull;
            const uint64_t inc = warp_incl_scan(gs, lane);
            uint64_t c = c0 + inc - gs;
            c0 += __shfl_sync(0xffffffffu, inc, 31);
            if (in) {
                uint32_t o[4];
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    o[e] = lq::cum_of(front + lq::shr64(c, d), (uint32_t)(4 * g + e), sc);
                    c += q[e];
                }
                if (out16) {
                    *reinterpret_cast<uint4*>(out + 4 * (int64_t)g) = make_uint4(o[0], o[1], o[2], o[3]);
                } else {
#pragma unroll
                    for (int e = 0; e < 4; e++) out[4 * (int64_t)g + e] = o[e];
                }
            }
        }
        return;
    }
    // lane l takes the 32 consecutive elements e0 + 32 l ...: one scan of the lane totals, then a serial walk
    const int b = e0 + 32 * lane;
    uint32_t q[kPerThread];
    uint64_t L = 0;
#pragma unroll
    for (int j = 0; j < kPerThread; j++) {
        const int e = b + j;
        q[j] = e < e1 ? lq::q_of(__ldg(row + min(e, e1 - 1)), nref) : 0u;
        L += q[j];
    }
    const uint64_t inc = warp_incl_scan(L, lane);
    uint64_t c = inc - L;
#pragma unroll
    for (int j = 0; j < kPerThread; j++) {
        const int e = b + j;
        if (e < e1) out[e] = lq::cum_of(front + lq::shr64(c, d), (uint32_t)e, sc);
        c += q[j];
    }
}

// ------------------------------------------------------------------ launchers
int sm_count() {
    static int cached[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
    if (!cached[dev]) {
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        cached[dev] = sms;
    }
    return cached[dev];
}

// Number of parts (1 .. 8) and the load width of pass 1 and the second passes: 4 for 16-byte aligned rows with
// V % 4 == 0 (the TMA ring, float4 loads), 1 for anything else (scalar loads), -1 if V is unsupported.
int path_for(const float* p, int V, int64_t s0, int64_t s1, int* parts) {
    *parts = lq::parts_of(V);
    if (V < 1 || *parts > lq::kMaxParts) return -1;
    const bool v4 = (V % 4 == 0) && ((((uintptr_t)p) & 15) == 0) && (s0 % 4 == 0) && (s1 % 4 == 0);
    return v4 ? 4 : 1;
}

// Row summaries of rows (s, t), s < n_outer, t < T, at base + s * so + t * st; summary of row (s, t) at
// summ + (s * T + t) * 32 * parts.  n_outer * T * parts must stay below 2^26 (summ_rows_for sees to it).
cudaError_t launch_summary(const float* base, int64_t n_outer, int64_t T, int64_t so, int64_t st_, int V, int parts,
                           int vec, int keep_l2, uint64_t* summ, cudaStream_t st) {
    SumParams sp;
    sp.base = base;
    sp.so = so;
    sp.st = st_;
    sp.T = (uint32_t)T;
    sp.n_tiles = (uint32_t)(n_outer * T * parts);
    sp.V = V;
    sp.G = lq::groups_of(V);
    sp.parts = parts;
    sp.inv_parts = (uint32_t)(((1ull << 31) + parts - 1) / parts);
    sp.keep_l2 = keep_l2;
    if (sp.n_tiles == 0) return cudaSuccess;
    const int ring_bytes = vec == 4 ? kRingBytes : 0;
    void (*kernel)(SumParams, uint64_t*) = vec == 4 ? summary_kernel<4> : summary_kernel<1>;
    if (ring_bytes > 0) {
        const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ring_bytes);
        if (e != cudaSuccess) return e;
    }
    const uint32_t sms = (uint32_t)sm_count();
    const unsigned grid = sp.n_tiles < sms ? sp.n_tiles : sms;
    kernel<<<grid, 32 * kTileWarps, ring_bytes, st>>>(sp, summ);
    return cudaGetLastError();
}

// Rows of summary a launch may cover: the scratch budget (LAC_SUMMARY_BYTES: test switch, forces many small
// chunks) and the tile index (the mul-shift division by parts is exact below 2^28 tiles).
int64_t summ_chunk_rows(int parts) {
    static const int64_t budget = getenv("LAC_SUMMARY_BYTES") ? atoll(getenv("LAC_SUMMARY_BYTES")) : (64ll << 20);
    int64_t rows = budget / (32 * parts * 8 + 8);
    const int64_t lim = ((1ll << 26) - 1) / (parts * 4);  // room for 4 tiles per part; changing it moves chunk bounds
    if (rows > lim) rows = lim;
    return rows < 1 ? 1 : rows;
}
size_t summ_only_bytes(int64_t rows, int parts) { return (size_t)rows * 32 * (size_t)parts * 8; }
size_t summ_bytes(int64_t rows, int parts) { return summ_only_bytes(rows, parts) + (size_t)rows * 8; }
// rows of summary that fit the scratch the call will use: the caller's workspace if it holds at least one row
int64_t summ_rows_for(int64_t want, int parts, const void* ws, size_t ws_bytes) {
    int64_t chunk = summ_chunk_rows(parts);
    if (ws && ws_bytes >= summ_bytes(1, parts)) {
        const int64_t fit = (int64_t)(ws_bytes / summ_bytes(1, parts));
        if (fit < chunk) chunk = fit;
    }
    return chunk > want ? want : chunk;
}

// Scratch: the caller's workspace when it is large enough, else a stream-ordered allocation (cudaMallocAsync; the
// default pool's release threshold is raised once so repeated calls do not go back to the OS).
cudaError_t scratch_get(Scratch* sc, size_t bytes, void* ws, size_t ws_bytes, cudaStream_t st) {
    sc->p = nullptr;
    sc->owned = false;
    if (ws && ws_bytes >= bytes && (((uintptr_t)ws) & 15) == 0) {
        sc->p = ws;
        return cudaSuccess;
    }
    int dev = 0;
    cudaGetDevice(&dev);
    static bool pool_ready[64] = {};
    if (dev >= 0 && dev < 64 && !pool_ready[dev]) {
        cudaMemPool_t mp;
        uint64_t keep = 1ull << 30;
        if (cudaDeviceGetDefaultMemPool(&mp, dev) == cudaSuccess)
            cudaMemPoolSetAttribute(mp, cudaMemPoolAttrReleaseThreshold, &keep);
        pool_ready[dev] = true;
    }
    sc->owned = true;
    return cudaMallocAsync(&sc->p, bytes ? bytes : 16, st);
}
cudaError_t scratch_put(Scratch* sc, cudaStream_t st) {
    if (sc->owned && sc->p) return cudaFreeAsync(sc->p, st);
    return cudaSuccess;
}

cudaError_t launch_pairs(const float* logits, int64_t n, int64_t T, int64_t so, int64_t st_, int V, int parts, int vec,
                         const uint64_t* summ, const int32_t* syms, int64_t sym_stride, uint32_t* pairs,
                         uint32_t* status, cudaStream_t st) {
    const int64_t rows = n * T;
    if (rows == 0) return cudaSuccess;
    const unsigned blocks = (unsigned)((rows + 7) / 8);
#define LAC_PAIR(CL_)                                                                                                 \
    if (vec == 1)                                                                                                     \
        pair_kernel<1, CL_><<<blocks, 256, 0, st>>>(logits, rows, T, so, st_, V, summ, syms, sym_stride, pairs, status); \
    else                                                                                                              \
        pair_kernel<4, CL_><<<blocks, 256, 0, st>>>(logits, rows, T, so, st_, V, summ, syms, sym_stride, pairs, status)
    LAC_BY_PARTS(parts, LAC_PAIR)
#undef LAC_PAIR
    return cudaGetLastError();
}

// lac_cdf_lookup_f32: summary pass + one warp per row for the pair.
cudaError_t launch_lookup(const float* logits, int64_t rows, int V, int64_t row_stride, const int32_t* syms,
                          uint32_t* pairs, uint32_t* status, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (rows == 0) return cudaSuccess;
    int parts = 1;
    const int vec = path_for(logits, V, row_stride, 0, &parts);
    if (vec < 0) return cudaErrorInvalidValue;
    const int64_t chunk = summ_rows_for(rows, parts, ws, ws_bytes);
    Scratch sc;
    cudaError_t e = scratch_get(&sc, summ_bytes(chunk, parts), ws, ws_bytes, st);
    if (e != cudaSuccess) return e;
    uint64_t* summ = (uint64_t*)sc.p;
    for (int64_t r0 = 0; r0 < rows && e == cudaSuccess; r0 += chunk) {
        const int64_t rn = rows - r0 < chunk ? rows - r0 : chunk;
        const float* base = logits + r0 * row_stride;
        e = launch_summary(base, rn, 1, row_stride, 0, V, parts, vec, 0, summ, st);
        if (e != cudaSuccess) break;
        e = launch_pairs(base, rn, 1, row_stride, 0, V, parts, vec, summ, syms + r0, 1, pairs + 2 * r0,
                         status ? status + r0 : nullptr, st);
        if (e != cudaSuccess) break;
        e = cudaGetLastError();
    }
    const cudaError_t ef = scratch_put(&sc, st);
    return e != cudaSuccess ? e : ef;
}

// lac_cdf_build_f32: per chunk of rows small enough to stay in L2 (~32 MB of logits), summary pass (L2-keeping
// policy) + table pass.
cudaError_t launch_build(const float* logits, int64_t rows, int V, int64_t row_stride, uint32_t* cum, void* ws,
                         size_t ws_bytes, cudaStream_t st) {
    if (rows == 0) return cudaSuccess;
    int parts = 1;
    const int vec = path_for(logits, V, row_stride, 0, &parts);
    if (vec < 0) return cudaErrorInvalidValue;
    int64_t l2rows = (32ll << 20) / ((int64_t)V * 4);
    l2rows = l2rows < 1 ? 1 : (l2rows > rows ? rows : l2rows);
    const int64_t chunk = summ_rows_for(l2rows, parts, ws, ws_bytes);
    Scratch sc;
    cudaError_t e = scratch_get(&sc, summ_bytes(chunk, parts), ws, ws_bytes, st);
    if (e != cudaSuccess) return e;
    uint64_t* summ = (uint64_t*)sc.p;
    for (int64_t r0 = 0; r0 < rows && e == cudaSuccess; r0 += chunk) {
        const int64_t rn = rows - r0 < chunk ? rows - r0 : chunk;
        const float* base = logits + r0 * row_stride;
        e = launch_summary(base, rn, 1, row_stride, 0, V, parts, vec, 1, summ, st);
        if (e != cudaSuccess) break;
        const unsigned blocks = (unsigned)((rn * 32 * parts + 7) / 8);
#define LAC_TABLE(CL_)                                                                                          \
    if (vec == 1) table_kernel<1, CL_><<<blocks, 256, 0, st>>>(base, rn, row_stride, V, summ, cum + r0 * (int64_t)V); \
    else table_kernel<4, CL_><<<blocks, 256, 0, st>>>(base, rn, row_stride, V, summ, cum + r0 * (int64_t)V)
        LAC_BY_PARTS(parts, LAC_TABLE)
#undef LAC_TABLE
        e = cudaGetLastError();
    }
    const cudaError_t ef = scratch_put(&sc, st);
    return e != cudaSuccess ? e : ef;
}

// Largest vocabulary the CDF kernels take.
int max_vocab() { return lq::kMaxParts * lq::kPartElems; }

}  // namespace lac
