// coder_kernels.cu -- batched multi-stream range coder kernels (north-star part (b)).
//
//   encode_pairs_staged_kernel   one lane per stream, 4 streams per warp; (lo, hi) pairs on the fixed total
//                         2^32 (output of the lookup) -> MSB-first bytes.  low / high live in registers, the k
//                         renormalisation bits of a token are appended in one step with carry resolution
//                         (coder.cuh) into a shared-memory stage that the whole warp flushes.
//   encode_fused_kernel   symbol ranges + coder in one launch for the model-in-the-loop step (T <= 4)
//   ac_tables_*           one warp per stream; int64 inclusive cumulative tables exactly as
//                         CDFPredictor.dist holds them, including fudged_dist
//                         (arith_code.py:83-93) evaluated as a parallel prefix-max:
//                           p_i = p_{i-1} + max(1, min(w - p_{i-1} - V + i + 1, f_i - p_{i-1}))
//                               = max(p_{i-1} + 1, g_i),   g_i = min(w - V + i + 1, f_i)
//                           =>  p_i - i = max(1, max_{j<=i} (g_j - j))
//                         which holds for arbitrary f_i (also the wrapped int64 products of
//                         Llama_AC, flag LAC_F_WRAP64).
//   acs_tables_*          ACSampler / Region semantics (arithmetic_coding.py).
#include <cstdint>
#include <cuda_runtime.h>

#include "coder.cuh"
#include "launch.h"
#include "rowsum.cuh"

namespace lac {

using coder::i128;
using coder::u128;

__device__ __forceinline__ i128 fdiv(i128 a, i128 b) {  // Python floor division, b > 0
    i128 q = a / b;
    if ((a % b != 0) && (a < 0)) q -= 1;
    return q;
}
__device__ __forceinline__ i128 cdiv(i128 a, i128 b) { return -fdiv(-a, b); }

__device__ __forceinline__ int64_t warp_max_i64(int64_t v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        int64_t t = __shfl_xor_sync(0xffffffffu, v, o);
        v = t > v ? t : v;
    }
    return v;
}
__device__ __forceinline__ int64_t warp_sum_i64(int64_t v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ------------------------------------------------------------------ pairs encoder
// One warp per kPairsSpb streams (lanes 0 .. kPairsSpb-1 run A_to_bin, low / high in registers).  The bytes of a
// batch of 16 tokens go to a per-stream shared-memory stage (coder::StagedWriter: carries resolved there); after
// every batch the WHOLE warp copies the stages to the streams' global buffers -- 32 consecutive bytes of one stream
// per store instruction instead of one byte per store and lane.  Each coder lane is a long dependent chain with
// data-dependent inner loops (bits per token differ per stream), so few streams per warp (less divergence) on many
// SMs (more schedulers) beat dense blocks.  Measured per [1024 x 16] slice inside the encode call (B200): 2 / 4 / 8
// streams per warp 0.347 / 0.348 / 0.350 ms, the same as one thread per stream with byte stores: 0.348 ms.
constexpr int kPairsSpb = 4;
__global__ void __launch_bounds__(32)
encode_pairs_staged_kernel(const uint2* __restrict__ pairs, int64_t n_streams, int64_t T, int64_t stream_stride,
                           int64_t tok_stride, const int32_t* __restrict__ ntok, int64_t t0,
                           lac_enc_state* __restrict__ state, uint8_t* __restrict__ out, int64_t out_stride,
                           int finish, int P) {
    __shared__ uint8_t s_stage[kPairsSpb][coder::StagedWriter::kStage + 1];
    __shared__ unsigned long long s_base[kPairsSpb];
    __shared__ int s_fill[kPairsSpb];
    const int lane = threadIdx.x;
    const int64_t s0 = (int64_t)blockIdx.x * kPairsSpb;
    const int ns = (int)min((int64_t)kPairsSpb, n_streams - s0);
    const bool is_coder = lane < ns;
    const int64_t s = s0 + lane;
    int64_t l = 0, h = 0, Ts = 0;
    coder::StagedWriter bw;
    const uint2* p = pairs;
    if (is_coder) {
        l = state[s].low;
        h = state[s].high;
        bw.open(out + s * out_stride, s_stage[lane], (uint64_t)out_stride, state[s].nbits, state[s].status);
        Ts = T;
        if (ntok) {
            Ts = (int64_t)ntok[s] - t0;
            Ts = Ts < 0 ? 0 : (Ts > T ? T : Ts);
        }
        p = pairs + s * stream_stride;
    }
    constexpr int kBatch = 8;  // pairs fetched together (independent loads in flight), two fetches per flush
    bool bad = false;
    int64_t tb0 = 0;
    do {
        const bool last = tb0 + 2 * kBatch >= T;
        if (is_coder) {
            for (int64_t tq = tb0; tq < tb0 + 2 * kBatch && tq < Ts && !bad; tq += kBatch) {
                uint2 pr[kBatch];
#pragma unroll
                for (int j = 0; j < kBatch; j++) {
                    const int64_t t = tq + j < Ts ? tq + j : Ts - 1;
                    pr[j] = p[t * tok_stride];
                }
#pragma unroll
                for (int j = 0; j < kBatch; j++)
                    if (tq + j < Ts && !bad) bad = !coder::code_pair(l, h, pr[j], P, bw);
            }
            if (last) {
                if (finish && !(bw.status & (LAC_ST_TABLE | LAC_ST_SYMBOL | LAC_ST_CAP))) coder::ac_flush(l, h, P, bw);
                bw.close();
            }
            s_base[lane] = bw.base;
            s_fill[lane] = bw.fill + bw.tail;
        }
        __syncwarp();
        for (int si = 0; si < ns; si++) {  // the whole warp moves one stream's staged bytes at a time
            uint8_t* dst = out + (s0 + si) * out_stride + s_base[si];
            const int nb = s_fill[si];
            for (int i = lane; i < nb; i += 32) dst[i] = s_stage[si][i];
        }
        __syncwarp();
        if (is_coder) bw.flushed();
        tb0 += 2 * kBatch;
    } while (tb0 < T);
    if (is_coder) {
        state[s].low = l;
        state[s].high = h;
        state[s].nbits = bw.nbits;
        state[s].status = bw.status;
    }
}

// ------------------------------------------------------------------ fused encoder (second pass of the encode side)
// One block per group of `spb` streams, 8 warps.  Per batch of `tb` tokens:
//   lookup  the warps share the batch's spb * tb rows: symbol_to_range from the row summary + the symbol's segment
//           (rowsum.cuh: 32 lanes per row, loads of a row issued together) -> (lo, hi) pairs in shared memory
//   code    thread i < spb runs A_to_bin (arith_code.py:169-202) over its stream's pairs, low / high in registers,
//           the k renormalisation bits of a token appended at once into the stream's shared-memory stage
//           (carries resolved there, coder.cuh:StagedWriter)
//   flush   every warp copies a stream's staged bytes to its global buffer (warp-wide coalesced stores)
// The pairs never go to global memory and there is one launch per call: the model-in-the-loop step (T = 1) is
// summary_kernel + this kernel.
struct EncParams {
    const float* base;
    int64_t n_streams, T, so, st;
    const int32_t* syms;
    int64_t sym_stride;
    const int32_t* ntok;  // per stream: tokens present counted from t0 tokens before `base` (nullptr: T everywhere)
    int64_t t0;
    const uint64_t* summ;
    lac_enc_state* state;
    uint8_t* out;
    int64_t out_stride;
    int V, P, finish, spb, tb;
};
constexpr int kEncWarps = 8;
constexpr int kEncRows = 32;  // rows (pairs) per batch and block: spb * tb <= kEncRows
constexpr int kEncMaxSpb = 16;

template <int VEC, int CL>
__global__ void __launch_bounds__(kEncWarps * 32)
encode_fused_kernel(const __grid_constant__ EncParams ep) {
    __shared__ uint2 s_pairs[kEncRows];
    __shared__ uint8_t s_stage[kEncMaxSpb][coder::StagedWriter::kStage + 1];
    __shared__ unsigned long long s_base[kEncMaxSpb];
    __shared__ int s_fill[kEncMaxSpb];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t s0 = (int64_t)blockIdx.x * ep.spb;
    const int ns = (int)min((int64_t)ep.spb, ep.n_streams - s0);  // streams of this block
    // coder threads: state in registers for the whole call
    const bool is_coder = threadIdx.x < ns;
    const int64_t sc = s0 + threadIdx.x;
    int64_t l = 0, h = 0;
    int my_tokens = 0;
    coder::StagedWriter bw;
    if (is_coder) {
        l = ep.state[sc].low;
        h = ep.state[sc].high;
        bw.open(ep.out + sc * ep.out_stride, s_stage[threadIdx.x], (uint64_t)ep.out_stride, ep.state[sc].nbits,
                ep.state[sc].status);
        int64_t n = ep.ntok ? (int64_t)ep.ntok[sc] - ep.t0 : ep.T;
        my_tokens = (int)(n < 0 ? 0 : (n > ep.T ? ep.T : n));
    }
    bool dead = false;  // coder thread: stream stopped (bad symbol / table, capacity)
    int64_t tb0 = 0;
    do {  // (a call with T = 0 still runs the flush / close of the last batch)
        const int nt = (int)min((int64_t)ep.tb, ep.T - tb0);
        // ---- lookup: row j of the batch = (stream j / nt, token tb0 + j % nt)
        for (int j = warp; j < ns * nt; j += kEncWarps) {
            const int si = j / nt, ti = j - si * nt;
            const int64_t s = s0 + si, t = tb0 + ti;
            const int64_t n = ep.ntok ? (int64_t)ep.ntok[s] - ep.t0 : ep.T;
            if (t >= n) continue;  // past the end of a ragged stream (warp-uniform)
            const int sym = __ldg(ep.syms + s * ep.sym_stride + t);
            uint2 pr = make_uint2(0xFFFFFFFFu, 0xFFFFFFFFu);  // symbol outside [0, V)
            if (sym >= 0 && sym < ep.V)
                pr = warp_symbol_range<VEC, CL>(ep.base + s * ep.so + t * ep.st, ep.V,
                                                ep.summ + (s * ep.T + t) * (32 * CL), sym, lane);
            if (lane == 0) s_pairs[j] = pr;
        }
        __syncthreads();
        // ---- code
        if (is_coder && !dead) {
            const int n_here = min(nt, my_tokens - (int)tb0);
            for (int ti = 0; ti < n_here; ti++) {
                // a stream stops at the token that truncates it
                if (!coder::code_pair(l, h, s_pairs[threadIdx.x * nt + ti], ep.P, bw) || (bw.status & LAC_ST_CAP)) {
                    dead = true;
                    break;
                }
            }
            if (tb0 + nt >= ep.T) {  // last batch of the call
                if (ep.finish && !(bw.status & (LAC_ST_TABLE | LAC_ST_SYMBOL | LAC_ST_CAP))) coder::ac_flush(l, h, ep.P, bw);
                bw.close();
            }
        }
        if (is_coder) {
            s_base[threadIdx.x] = bw.base;
            s_fill[threadIdx.x] = bw.fill + bw.tail;
        }
        __syncthreads();
        // ---- flush: warp w copies the staged bytes of streams w, w + 8, ...
        for (int si = warp; si < ns; si += kEncWarps) {
            uint8_t* dst = ep.out + (s0 + si) * ep.out_stride + s_base[si];
            const int nb = s_fill[si];
            for (int i = lane; i < nb; i += 32) dst[i] = s_stage[si][i];
        }
        if (is_coder) bw.flushed();
        __syncthreads();  // the stage and the pairs are reused by the next batch
        tb0 += ep.tb;
    } while (tb0 < ep.T);
    if (is_coder) {
        ep.state[sc].low = l;
        ep.state[sc].high = h;
        ep.state[sc].nbits = bw.nbits;
        ep.state[sc].status = bw.status;
    }
}

// ------------------------------------------------------------------ uniform Predictor(n) (arith_code.py:64-74)
// The reference's base class maps symbol s of n to [floor(s w / n), floor((s + 1) w / n)) -- floor, not the ceil of
// CDFPredictor.  AC() without arguments is AC(Predictor(3), 16).  One thread per stream.
__global__ void uniform_encode_kernel(const int32_t* __restrict__ syms, int64_t n_streams, int64_t T, int64_t sym_stride,
                                      const int32_t* __restrict__ ntok, int nsym, lac_enc_state* __restrict__ state,
                                      uint8_t* __restrict__ out, int64_t out_stride, int finish, int P) {
    int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= n_streams) return;
    int64_t l = state[s].low, h = state[s].high;
    coder::BitWriter bw;
    bw.open(out + s * out_stride, (uint64_t)out_stride, state[s].nbits);
    bw.status = state[s].status;
    const int64_t Ts = ntok ? (int64_t)ntok[s] : T;
    for (int64_t t = 0; t < Ts; t++) {
        const int sym = syms[s * sym_stride + t];
        if (sym < 0 || sym >= nsym) {
            bw.status |= LAC_ST_SYMBOL;
            break;
        }
        const u128 w = (u128)(uint64_t)(h - l + 1);
        const int64_t r0 = (int64_t)(((u128)(uint32_t)sym * w) / (uint32_t)nsym);          // symbol_to_range :69-70
        const int64_t r1 = (int64_t)((((u128)(uint32_t)sym + 1) * w) / (uint32_t)nsym);
        if (r1 <= r0) {  // zero-width symbol (w < n): the reference would never terminate
            bw.status |= LAC_ST_TABLE;
            break;
        }
        h = l + r1 - 1;  // receive_symbol :169-175
        l += r0;
        int k = coder::renorm_count((uint64_t)(h - l + 1), P);
        int64_t E = coder::renorm_apply(l, h, P, k);
        bw.append(E, k);
        if (bw.status & LAC_ST_CAP) break;
    }
    if (finish && !(bw.status & (LAC_ST_TABLE | LAC_ST_SYMBOL | LAC_ST_CAP))) coder::ac_flush(l, h, P, bw);
    bw.close();
    state[s].low = l;
    state[s].high = h;
    state[s].nbits = bw.nbits;
    state[s].status = bw.status;
}

// Decoder: the symbol whose floor-mapped range holds the code value, i.e. the largest s with
// floor(s w / n) <= v - l, s = floor(((v - l + 1) n - 1) / w).  (The reference's val_to_symbol, (v n) // w, is not
// that symbol at range boundaries; its decoder asserts there.  See tests/golden/ac_uniform.npz.)
__global__ void uniform_decode_kernel(int64_t n_streams, int64_t T, const int32_t* __restrict__ ntok, int nsym,
                                      lac_dec_state* __restrict__ state, const uint8_t* __restrict__ bytes,
                                      const int64_t* __restrict__ offsets, int32_t* __restrict__ syms,
                                      int64_t sym_stride, int P) {
    int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= n_streams) return;
    int64_t l = state[s].low, h = state[s].high, v = state[s].value;
    uint64_t pos = state[s].pos;
    uint32_t status = state[s].status;
    const uint8_t* data = bytes + offsets[s];
    const uint64_t nbytes = (uint64_t)(offsets[s + 1] - offsets[s]);
    const int64_t Ts = ntok ? (int64_t)ntok[s] : T;
    for (int64_t t = 0; t < Ts; t++) {
        const u128 w = (u128)(uint64_t)(h - l + 1);
        const u128 x = (u128)(uint64_t)(v - l);
        const int64_t sym = (int64_t)(((x + 1) * (uint32_t)nsym - 1) / w);
        const int64_t r0 = (int64_t)(((u128)(uint64_t)sym * w) / (uint32_t)nsym);
        const int64_t r1 = (int64_t)((((u128)(uint64_t)sym + 1) * w) / (uint32_t)nsym);
        if (sym >= nsym || r1 <= r0) {
            status |= LAC_ST_TABLE;
            break;
        }
        h = l + r1 - 1;
        l += r0;
        const int64_t off = v - l;
        int k = coder::renorm_count((uint64_t)(h - l + 1), P);
        coder::renorm_apply(l, h, P, k);
        v = l + (off << k) + (int64_t)coder::read_bits(data, nbytes, pos, k);
        pos += (uint64_t)k;
        syms[s * sym_stride + t] = (int32_t)sym;
    }
    state[s].low = l;
    state[s].high = h;
    state[s].value = v;
    state[s].pos = pos;
    state[s].status = status;
}

__global__ void enc_init_kernel(lac_enc_state* state, int64_t n, int P) {
    int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= n) return;
    state[s].low = 0;
    state[s].high = (1ll << P) - 1;
    state[s].nbits = 0;
    state[s].status = 0;
    state[s]._pad = 0;
}

// ------------------------------------------------------------------ CDFPredictor on a warp
struct TableCtx {
    const int64_t* tbl;
    int V;
    int64_t minp;
    int wrap;
};

// f_i of fudged_dist: (dist[i] * denom) // dist[-1]   (np.int64-wrapped under LAC_F_WRAP64)
__device__ __forceinline__ i128 fudge_f(const TableCtx& c, int i, int64_t w, int64_t last) {
    i128 prod = c.wrap ? (i128)(int64_t)((uint64_t)c.tbl[i] * (uint64_t)w) : (i128)c.tbl[i] * (i128)w;
    return fdiv(prod, (i128)last);
}
__device__ __forceinline__ bool is_fudged(const TableCtx& c, int64_t w, int64_t last) {
    i128 thr = c.wrap ? (i128)(int64_t)((uint64_t)w * (uint64_t)c.minp) : (i128)w * (i128)c.minp;
    return !((i128)last <= thr);
}
// g_i - i, clamped into int64 (|f| can reach 2^63 / 1 only for degenerate tables)
__device__ __forceinline__ int64_t fudge_key(const TableCtx& c, int i, int64_t w, int64_t last) {
    i128 f = fudge_f(c, i, w, last);
    i128 cap = (i128)w - c.V + i + 1;
    i128 g = f < cap ? f : cap;
    g -= i;
    const i128 lim = ((i128)1) << 62;
    if (g > lim) g = lim;
    if (g < -lim) g = -lim;
    return (int64_t)g;
}

// Warp-cooperative: the three fudged cumulative values p[a-1] (0 if a == 0), p[a], p[V-1].
__device__ inline void fudged_three(const TableCtx& c, int a, int64_t w, int64_t last, int lane,
                                    int64_t& p_lo, int64_t& p_hi, int64_t& p_last) {
    const int64_t NEG = -(1ll << 62);
    int64_t m_lo = NEG, m_hi = NEG, m_all = NEG;
    for (int i = lane; i < c.V; i += 32) {
        int64_t k = fudge_key(c, i, w, last);
        if (i < a) m_lo = k > m_lo ? k : m_lo;
        if (i <= a) m_hi = k > m_hi ? k : m_hi;
        m_all = k > m_all ? k : m_all;
    }
    m_lo = warp_max_i64(m_lo);
    m_hi = warp_max_i64(m_hi);
    m_all = warp_max_i64(m_all);
    p_lo = a > 0 ? (a - 1) + (m_lo > 1 ? m_lo : 1) : 0;
    p_hi = a + (m_hi > 1 ? m_hi : 1);
    p_last = (c.V - 1) + (m_all > 1 ? m_all : 1);
}

// symbol_to_range (arith_code.py:98-110): offsets r0, r1 inside a width-w interval.
__device__ inline bool table_range(const TableCtx& c, int sym, int64_t w, int lane, int64_t& r0, int64_t& r1) {
    const int64_t last = c.tbl[c.V - 1];
    int64_t ld, hd, d;
    if (is_fudged(c, w, last)) {
        fudged_three(c, sym, w, last, lane, ld, hd, d);
    } else {
        ld = sym > 0 ? c.tbl[sym - 1] : 0;
        hd = c.tbl[sym];
        d = last;
    }
    if (d <= 0) return false;
    r0 = (int64_t)cdiv((i128)ld * w, (i128)d);
    r1 = (int64_t)cdiv((i128)hd * w, (i128)d);
    return r1 > r0;
}

// val_to_symbol (arith_code.py:94-97): bisect_right(fudged_dist(w), (x * dist[-1]) // w).
__device__ inline int table_symbol(const TableCtx& c, int64_t x, int64_t w, int lane) {
    const int64_t last = c.tbl[c.V - 1];
    int64_t cnt = 0;
    if (!is_fudged(c, w, last)) {
        i128 target = fdiv((i128)x * last, (i128)w);
        for (int i = lane; i < c.V; i += 32) cnt += ((i128)c.tbl[i] <= target);
        return (int)warp_sum_i64(cnt);
    }
    // fudged: lane owns the contiguous block [b, e); running max of (g_j - j) carried across lanes
    const int64_t NEG = -(1ll << 62);
    const int per = (c.V + 31) / 32;
    const int b = lane * per < c.V ? lane * per : c.V, e = b + per < c.V ? b + per : c.V;
    int64_t m = NEG;
    for (int i = b; i < e; i++) {
        int64_t k = fudge_key(c, i, w, last);
        m = k > m ? k : m;
    }
    int64_t inc = m;  // inclusive max-scan over lanes
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int64_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc = t > inc ? t : inc;
    }
    int64_t m_all = __shfl_sync(0xffffffffu, inc, 31);
    int64_t run = __shfl_up_sync(0xffffffffu, inc, 1);
    if (lane == 0) run = NEG;
    const int64_t d = (c.V - 1) + (m_all > 1 ? m_all : 1);
    const i128 target = fdiv((i128)x * d, (i128)w);
    for (int i = b; i < e; i++) {
        int64_t k = fudge_key(c, i, w, last);
        run = k > run ? k : run;
        int64_t p = i + (run > 1 ? run : 1);
        cnt += ((i128)p <= target);
    }
    return (int)warp_sum_i64(cnt);
}

__device__ __forceinline__ TableCtx table_ctx(const int64_t* dist, int V, int64_t ss, int64_t ts,
                                              const int64_t* minp, int64_t mss, int64_t mts, int64_t s,
                                              int64_t t, int flags) {
    TableCtx c;
    c.tbl = dist + s * ss + t * ts;
    c.V = V;
    c.minp = minp[s * mss + t * mts];
    c.wrap = (flags & LAC_F_WRAP64) != 0;
    return c;
}

// ------------------------------------------------------------------ A_to_bin on tables
__global__ void ac_tables_encode_kernel(const int64_t* __restrict__ dist, int V, int64_t ss, int64_t ts,
                                        const int64_t* __restrict__ minp, int64_t mss, int64_t mts,
                                        const int32_t* __restrict__ syms, int64_t sym_stride, int64_t n_streams,
                                        int64_t T, const int32_t* __restrict__ ntok,
                                        lac_enc_state* __restrict__ state, uint8_t* __restrict__ out,
                                        int64_t out_stride, int finish, int P, int flags) {
    const int lane = threadIdx.x & 31;
    int64_t s = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (s >= n_streams) return;
    int64_t l = state[s].low, h = state[s].high;
    coder::BitWriter bw;
    bw.open(out + s * out_stride, (uint64_t)out_stride, state[s].nbits);
    bw.status = state[s].status;
    const int64_t Ts = ntok ? (int64_t)ntok[s] : T;
    for (int64_t t = 0; t < Ts; t++) {
        const int sym = syms[s * sym_stride + t];
        if (sym < 0 || sym >= V) {
            bw.status |= LAC_ST_SYMBOL;
            break;
        }
        TableCtx c = table_ctx(dist, V, ss, ts, minp, mss, mts, s, t, flags);
        int64_t r0, r1;
        if (!table_range(c, sym, h - l + 1, lane, r0, r1)) {
            bw.status |= LAC_ST_TABLE;
            break;
        }
        h = l + r1 - 1;
        l += r0;
        int k = coder::renorm_count((uint64_t)(h - l + 1), P);
        int64_t E = coder::renorm_apply(l, h, P, k);
        if (lane == 0) bw.append(E, k);
        if (__shfl_sync(0xffffffffu, bw.status, 0) & LAC_ST_CAP) break;
    }
    if (lane == 0) {
        if (finish && !(bw.status & (LAC_ST_TABLE | LAC_ST_SYMBOL | LAC_ST_CAP))) coder::ac_flush(l, h, P, bw);
        bw.close();
        state[s].low = l;
        state[s].high = h;
        state[s].nbits = bw.nbits;
        state[s].status = bw.status;
    }
}

__global__ void ac_tables_decode_kernel(const int64_t* __restrict__ dist, int V, int64_t ss, int64_t ts,
                                        const int64_t* __restrict__ minp, int64_t mss, int64_t mts,
                                        int64_t n_streams, int64_t T, const int32_t* __restrict__ ntok,
                                        lac_dec_state* __restrict__ state, const uint8_t* __restrict__ bytes,
                                        const int64_t* __restrict__ offsets, int32_t* __restrict__ syms,
                                        int64_t sym_stride, int P, int flags) {
    const int lane = threadIdx.x & 31;
    int64_t s = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (s >= n_streams) return;
    int64_t l = state[s].low, h = state[s].high, v = state[s].value;
    uint64_t pos = state[s].pos;
    uint32_t status = state[s].status;
    const uint8_t* data = bytes + offsets[s];
    const uint64_t nbytes = (uint64_t)(offsets[s + 1] - offsets[s]);
    const int64_t Ts = ntok ? (int64_t)ntok[s] : T;
    for (int64_t t = 0; t < Ts; t++) {
        TableCtx c = table_ctx(dist, V, ss, ts, minp, mss, mts, s, t, flags);
        const int64_t w = h - l + 1;
        int sym = table_symbol(c, v - l, w, lane);
        int64_t r0, r1;
        if (sym >= V || !table_range(c, sym, w, lane, r0, r1)) {
            status |= LAC_ST_TABLE;
            break;
        }
        h = l + r1 - 1;
        l += r0;
        const int64_t off = v - l;
        int k = coder::renorm_count((uint64_t)(h - l + 1), P);
        coder::renorm_apply(l, h, P, k);
        v = l + (off << k) + (int64_t)coder::read_bits(data, nbytes, pos, k);
        pos += (uint64_t)k;
        if (lane == 0) syms[s * sym_stride + t] = sym;
    }
    if (lane == 0) {
        state[s].low = l;
        state[s].high = h;
        state[s].value = v;
        state[s].pos = pos;
        state[s].status = status;
    }
}

// ------------------------------------------------------------------ ACSampler on tables
__global__ void acs_tables_encode_kernel(const uint64_t* __restrict__ cdf, int V, int64_t ss, int64_t ts,
                                         const int32_t* __restrict__ syms, int64_t sym_stride, int64_t n_streams,
                                         int64_t T, const int32_t* __restrict__ ntok,
                                         lac_enc_state* __restrict__ state, uint8_t* __restrict__ out,
                                         int64_t out_stride, int finish, int P) {
    int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= n_streams) return;
    int64_t low = state[s].low, high = state[s].high;
    coder::BitWriter bw;
    bw.open(out + s * out_stride, (uint64_t)out_stride, state[s].nbits);
    bw.status = state[s].status;
    const int64_t Ts = ntok ? (int64_t)ntok[s] : T;
    for (int64_t t = 0; t < Ts; t++) {
        const int tok = syms[s * sym_stride + t];
        if (tok < 0 || tok >= V) {
            bw.status |= LAC_ST_SYMBOL;
            break;
        }
        const uint64_t* c = cdf + s * ss + t * ts;
        // sample_scaled_cdf compress path, arithmetic_coding.py:85-87
        uint64_t cl = tok ? c[tok - 1] : 0, ch = c[tok], den = c[V - 1];
        if (den == 0 || ch <= cl) {
            bw.status |= LAC_ST_TABLE;
            break;
        }
        coder::acs_narrow(low, high, cl, ch, den);
        if (high < low) {
            bw.status |= LAC_ST_TABLE;
            break;
        }
        int k = coder::renorm_count((uint64_t)(high - low + 1), P);
        bw.append(coder::renorm_apply(low, high, P, k), k);
        if (bw.status & LAC_ST_CAP) break;
    }
    if (finish == 1 && !(bw.status & (LAC_ST_TABLE | LAC_ST_SYMBOL | LAC_ST_CAP))) {
        // flush_compress, arithmetic_coding.py:50-56: step(1, 2, 3), drain the carry buffer, reset.
        // Bit-exact with the reference, but the bits do not pin the final region (DESIGN.md
        // section 6): the last tokens may be undecodable by ANY decoder.
        coder::acs_narrow(low, high, 1, 2, 3);
        int k = coder::renorm_count((uint64_t)(high - low + 1), P);
        bw.append(coder::renorm_apply(low, high, P, k), k);
        low = 0;
        high = (1ll << P) - 1;
    } else if (finish == 2 && !(bw.status & (LAC_ST_TABLE | LAC_ST_SYMBOL | LAC_ST_CAP))) {
        // safe termination: shortest bit string whose every continuation stays inside [low, high]
        // (A_to_bin.flush, arith_code.py:193-202) -- always decodable
        coder::ac_flush(low, high, P, bw);
    }
    bw.close();
    state[s].low = low;
    state[s].high = high;
    state[s].nbits = bw.nbits;
    state[s].status = bw.status;
}

// Decoder for ACSampler streams: symbol whose encoder interval [map(c[i-1]), map(c[i]) - 1]
// contains the value; map(c) <= v  <=>  c <= ceil((v - low + 1) * den / span) - 1.
__global__ void acs_tables_decode_kernel(const uint64_t* __restrict__ cdf, int V, int64_t ss, int64_t ts,
                                         int64_t n_streams, int64_t T, const int32_t* __restrict__ ntok,
                                         lac_dec_state* __restrict__ state, const uint8_t* __restrict__ bytes,
                                         const int64_t* __restrict__ offsets, int32_t* __restrict__ syms,
                                         int64_t sym_stride, int P) {
    const int lane = threadIdx.x & 31;
    int64_t s = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (s >= n_streams) return;
    int64_t low = state[s].low, high = state[s].high, v = state[s].value;
    uint64_t pos = state[s].pos;
    uint32_t status = state[s].status;
    const uint8_t* data = bytes + offsets[s];
    const uint64_t nbytes = (uint64_t)(offsets[s + 1] - offsets[s]);
    const int64_t Ts = ntok ? (int64_t)ntok[s] : T;
    for (int64_t t = 0; t < Ts; t++) {
        const uint64_t* c = cdf + s * ss + t * ts;
        const uint64_t den = c[V - 1];
        const u128 span = (u128)(uint64_t)(high - low + 1);
        if (den == 0) {
            status |= LAC_ST_TABLE;
            break;
        }
        const u128 num = (u128)(uint64_t)(v - low + 1) * den;
        const u128 tau = (num + span - 1) / span - 1;
        int64_t cnt = 0;
        for (int i = lane; i < V; i += 32) cnt += ((u128)c[i] <= tau);
        const int tok = (int)warp_sum_i64(cnt);
        if (tok >= V) {
            status |= LAC_ST_TABLE;
            break;
        }
        uint64_t cl = tok ? c[tok - 1] : 0, ch = c[tok];
        coder::acs_narrow(low, high, cl, ch, den);
        const int64_t off = v - low;
        int k = coder::renorm_count((uint64_t)(high - low + 1), P);
        coder::renorm_apply(low, high, P, k);
        v = low + (off << k) + (int64_t)coder::read_bits(data, nbytes, pos, k);
        pos += (uint64_t)k;
        if (lane == 0) syms[s * sym_stride + t] = tok;
    }
    if (lane == 0) {
        state[s].low = low;
        state[s].high = high;
        state[s].value = v;
        state[s].pos = pos;
        state[s].status = status;
    }
}

// ------------------------------------------------------------------ status collection
__global__ void status_or_kernel(const uint32_t* __restrict__ state, int64_t n, int stride_words, int status_word,
                                 uint32_t* __restrict__ d_or) {
    uint32_t v = 0;
    for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < n; s += (int64_t)gridDim.x * blockDim.x)
        v |= state[s * stride_words + status_word];
    v = __reduce_or_sync(0xffffffffu, v);
    if ((threadIdx.x & 31) == 0 && v) atomicOr(d_or, v);
}
cudaError_t launch_status_or(const void* state, int64_t n, int stride_words, int status_word, uint32_t* d_or,
                             cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(d_or, 0, 4, st);
    if (e != cudaSuccess || n == 0) return e;
    const unsigned blocks = (unsigned)((n + 255) / 256 > 1024 ? 1024 : (n + 255) / 256);
    status_or_kernel<<<blocks, 256, 0, st>>>((const uint32_t*)state, n, stride_words, status_word, d_or);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ launchers
cudaError_t launch_enc_init(lac_enc_state* state, int64_t n, int P, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    enc_init_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(state, n, P);
    return cudaGetLastError();
}

// ntok counts tokens from t0 tokens before the first pair of the call
cudaError_t launch_encode_pairs(const uint32_t* pairs, int64_t n, int64_t T, int64_t ss, int64_t ts,
                                const int32_t* ntok, int64_t t0, lac_enc_state* state, uint8_t* out,
                                int64_t out_stride, int finish, int P, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    encode_pairs_staged_kernel<<<(unsigned)((n + kPairsSpb - 1) / kPairsSpb), 32, 0, st>>>(
        reinterpret_cast<const uint2*>(pairs), n, T, ss, ts, ntok, t0, state, out, out_stride, finish, P);
    return cudaGetLastError();
}

// lac_ac_encode_logits_f32: per token chunk (the scratch bounds it) the summary pass, then
//   T <= 4 (the model-in-the-loop step): ONE fused kernel (symbol ranges + coder, pairs in shared memory);
//   longer slices: pair_kernel over all rows at once (thousands of independent warps, ~20 us per 16k rows) into
//   the scratch, then the pairs coder (encode_pairs_staged_kernel).  A fused kernel keeps 8 warps of registers
//   resident per stream for the whole serial coding chain -- measured 52 us per [1024 x 16] slice against 37 us for
//   the two kernels.
cudaError_t launch_encode_logits(const float* logits, int64_t n, int64_t T, int64_t ss, int64_t ts, int V,
                                 const int32_t* syms, int64_t sym_stride, const int32_t* ntok, lac_enc_state* state,
                                 uint8_t* out, int64_t out_stride, int finish, int P, void* ws, size_t ws_bytes,
                                 cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    int parts = 1;
    const int vec = path_for(logits, V, ss, ts, &parts);
    if (vec < 0) return cudaErrorInvalidValue;
    const int64_t Tn = T < 1 ? 1 : T;
    int64_t tc = summ_rows_for(n * Tn, parts, ws, ws_bytes) / n;
    tc = tc < 1 ? 1 : (tc > Tn ? Tn : tc);
    const bool fused = T <= 4;
    Scratch sc;
    cudaError_t e = scratch_get(&sc, summ_bytes(n * tc, parts), ws, ws_bytes, st);
    if (e != cudaSuccess) return e;
    uint32_t* pairs = fused ? nullptr : (uint32_t*)((char*)sc.p + summ_only_bytes(n * tc, parts));
    for (int64_t t0 = 0; (t0 < T || (T == 0 && t0 == 0)) && e == cudaSuccess; t0 += tc) {
        const int64_t tn = T - t0 < tc ? T - t0 : tc;
        const float* base = logits + t0 * ts;
        if (tn > 0) e = launch_summary(base, n, tn, ss, ts, V, parts, vec, 0, (uint64_t*)sc.p, st);
        if (e != cudaSuccess) break;
        const int fin = (finish && t0 + tn >= T) ? 1 : 0;
        if (!fused) {
            e = launch_pairs(base, n, tn, ss, ts, V, parts, vec, (const uint64_t*)sc.p, syms + t0, sym_stride, pairs,
                             nullptr, st);
            if (e != cudaSuccess) break;
            // ntok counts from the start of the call: shift it by t0 inside the kernel
            e = launch_encode_pairs(pairs, n, tn, tn, 1, ntok, t0, state, out, out_stride, fin, P, st);
            continue;
        }
        EncParams ep;
        ep.base = base;
        ep.n_streams = n;
        ep.T = tn;
        ep.so = ss;
        ep.st = ts;
        ep.syms = syms + t0;
        ep.sym_stride = sym_stride;
        ep.ntok = ntok;
        ep.t0 = t0;
        ep.summ = (const uint64_t*)sc.p;
        ep.state = state;
        ep.out = out;
        ep.out_stride = out_stride;
        ep.V = V;
        ep.P = P;
        ep.finish = fin;
        // streams per block and tokens per batch: every warp of a block should have a row (T = 1: 8 streams)
        ep.tb = (int)(tn < 1 ? 1 : tn);
        ep.spb = kEncWarps / ep.tb < 1 ? 1 : kEncWarps / ep.tb;
        if (tn == 0) ep.spb = kEncMaxSpb;  // flush-only call: as many streams per block as the stage allows
        const unsigned blocks = (unsigned)((n + ep.spb - 1) / ep.spb);
#define LAC_ENC(CL_)                                                             \
    if (vec == 1) encode_fused_kernel<1, CL_><<<blocks, kEncWarps * 32, 0, st>>>(ep);  \
    else encode_fused_kernel<4, CL_><<<blocks, kEncWarps * 32, 0, st>>>(ep)
        LAC_BY_PARTS(parts, LAC_ENC)
#undef LAC_ENC
        e = cudaGetLastError();
        if (T == 0) break;
    }
    const cudaError_t ef = scratch_put(&sc, st);
    return e != cudaSuccess ? e : ef;
}

cudaError_t launch_uniform_encode(const int32_t* syms, int64_t n, int64_t T, int64_t sym_stride, const int32_t* ntok,
                                  int nsym, lac_enc_state* state, uint8_t* out, int64_t out_stride, int finish, int P,
                                  cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    uniform_encode_kernel<<<(unsigned)((n + 31) / 32), 32, 0, st>>>(syms, n, T, sym_stride, ntok, nsym, state, out,
                                                                    out_stride, finish, P);
    return cudaGetLastError();
}

cudaError_t launch_uniform_decode(int64_t n, int64_t T, const int32_t* ntok, int nsym, lac_dec_state* state,
                                  const uint8_t* bytes, const int64_t* offsets, int32_t* syms, int64_t sym_stride,
                                  int P, cudaStream_t st) {
    if (n == 0 || T == 0) return cudaSuccess;
    uniform_decode_kernel<<<(unsigned)((n + 31) / 32), 32, 0, st>>>(n, T, ntok, nsym, state, bytes, offsets, syms,
                                                                    sym_stride, P);
    return cudaGetLastError();
}

cudaError_t launch_ac_tables_encode(const int64_t* dist, int V, int64_t ss, int64_t ts, const int64_t* minp,
                                    int64_t mss, int64_t mts, const int32_t* syms, int64_t sym_stride, int64_t n,
                                    int64_t T, const int32_t* ntok, lac_enc_state* state, uint8_t* out,
                                    int64_t out_stride, int finish, int P, int flags, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    ac_tables_encode_kernel<<<(unsigned)((n + 3) / 4), 128, 0, st>>>(dist, V, ss, ts, minp, mss, mts, syms, sym_stride, n,
                                                                    T, ntok, state, out, out_stride, finish, P, flags);
    return cudaGetLastError();
}

cudaError_t launch_ac_tables_decode(const int64_t* dist, int V, int64_t ss, int64_t ts, const int64_t* minp,
                                    int64_t mss, int64_t mts, int64_t n, int64_t T, const int32_t* ntok,
                                    lac_dec_state* state, const uint8_t* bytes, const int64_t* offsets,
                                    int32_t* syms, int64_t sym_stride, int P, int flags, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    ac_tables_decode_kernel<<<(unsigned)((n + 3) / 4), 128, 0, st>>>(dist, V, ss, ts, minp, mss, mts, n, T, ntok,
                                                                    state, bytes, offsets, syms, sym_stride, P,
                                                                    flags);
    return cudaGetLastError();
}

cudaError_t launch_acs_tables_encode(const uint64_t* cdf, int V, int64_t ss, int64_t ts, const int32_t* syms,
                                     int64_t sym_stride, int64_t n, int64_t T, const int32_t* ntok,
                                     lac_enc_state* state, uint8_t* out, int64_t out_stride, int finish, int P,
                                     cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    acs_tables_encode_kernel<<<(unsigned)((n + 31) / 32), 32, 0, st>>>(cdf, V, ss, ts, syms, sym_stride, n, T, ntok,
                                                                      state, out, out_stride, finish, P);
    return cudaGetLastError();
}

cudaError_t launch_acs_tables_decode(const uint64_t* cdf, int V, int64_t ss, int64_t ts, int64_t n, int64_t T,
                                     const int32_t* ntok, lac_dec_state* state, const uint8_t* bytes,
                                     const int64_t* offsets, int32_t* syms, int64_t sym_stride, int P,
                                     cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    acs_tables_decode_kernel<<<(unsigned)((n + 3) / 4), 128, 0, st>>>(cdf, V, ss, ts, n, T, ntok, state, bytes,
                                                                     offsets, syms, sym_stride, P);
    return cudaGetLastError();
}

}  // namespace lac
