// coder_kernels.cu -- batched multi-stream range coder kernels on the logits path (north-star part (b)).
//
//   encode_pairs_staged_kernel   one lane per stream, 4 streams per warp; (lo, hi) pairs on the fixed total
//                         2^32 (output of the lookup) -> MSB-first bytes.  low / high live in registers, the k
//                         renormalisation bits of a token are appended in one step with carry resolution
//                         (coder.cuh) into a shared-memory stage that the whole warp flushes.
//   encode_fused_kernel   symbol ranges + coder in one launch for the model-in-the-loop step (T <= 4)
// The coders on tables the caller supplies (CDFPredictor, ACSampler, Predictor(n)) are in table_coders.cu.
#include <cstdint>
#include <cuda_runtime.h>

#include "coder.cuh"
#include "launch.h"
#include "rowsum.cuh"

namespace lac {

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

__global__ void enc_init_kernel(lac_enc_state* state, int64_t n, int P) {
    int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= n) return;
    state[s].low = 0;
    state[s].high = (1ll << P) - 1;
    state[s].nbits = 0;
    state[s].status = 0;
    state[s]._pad = 0;
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

}  // namespace lac
