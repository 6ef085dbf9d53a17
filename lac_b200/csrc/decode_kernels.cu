// decode_kernels.cu -- the decoder side of north-star part (b): A_from_bin (arith_code.py:248-334) driven by
// logits.  Decode = summary_kernel (cdf_kernels.cu, the bandwidth-bound pass) + decode_serial_kernel.
//
// val_to_symbol (arith_code.py:94-97) on the total d = 2^32: bisect_right(dist, target) with
// target = ((value - l) * 2^32) // w, i.e. the last symbol whose exclusive cumulative is <= target.  Every boundary
// test is a 96-bit multiply-shift and a compare.
#include <cstdint>
#include <cuda_runtime.h>

#include "coder.cuh"
#include "launch.h"
#include "lq32.cuh"
#include "ptx.cuh"
#include "rowsum.cuh"

namespace lac {

// 8 stream bytes at byte offset b as a big-endian word, zeros past the end
// Assembled as two 32-bit halves from unconditional loads at clamped addresses plus a mask.  (The obvious
// form -- a 64-bit accumulator fed by predicated byte loads -- was observed to be miscompiled by ptxas 12.9 in
// one instantiation: a CS2R-zeroed register pair was read 5 cycles later still holding its previous content,
// which corrupted the window of streams shorter than 22 bytes.  tests/test_gpu_parity.py pins that case.)
__device__ __forceinline__ uint64_t load_be64(const uint8_t* data, uint64_t nbytes, uint64_t b) {
    if (b >= nbytes) return 0;
    uint32_t w[2] = {0u, 0u};
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const uint64_t idx = b + i;
        const bool in = idx < nbytes;
        const uint32_t byte = (uint32_t)data[in ? idx : b] & (in ? 0xFFu : 0u);
        w[i >> 2] = (w[i >> 2] << 8) | byte;
    }
    return ((uint64_t)w[0] << 32) | w[1];
}

// One warp per stream; every lane carries the same A_from_bin state in registers.  Per token:
//   probe    target = floor(((value - low) << 32) / w)
//   level 1  the last non-empty segment of the row whose first cumulative is <= target (prefixes of the aligned
//            segment weights, from the summary words)
//   level 2  that segment (<= 1024 elements, <= 4 KB) is read again, lane-major (lane l = 32 consecutive elements),
//            q recomputed against the segment's reference (bit-identical to pass 1 by construction of LQ32), one warp
//            scan + ballot picks the lane, the rest of the search is independent work inside each lane
//   update   narrow, renormalise by k bits at once, pull k bits from a 24-byte register window of the stream
// The logits segment comes from HBM (pass 1 streamed the rows with evict-first), ~3 % extra traffic.
// The summary of token t + 1 is loaded while token t is being searched and its scale (the one division that does
// not depend on the coder state) is computed while token t's segment is in flight.
// LAC_ST_TRUNC: the decoder consumed more bits than the stream holds (a truncated or foreign stream; the reference
// raises "predictor range does not correspond to val", arith_code.py:277-278, on such input).
struct SerialParams {
    const float* base;
    int64_t n_streams, T, so, st;
    const int32_t* ntok;  // per stream: tokens present counted from t0 tokens before `base` (nullptr: T everywhere)
    int64_t t0;
};
__device__ __forceinline__ int tokens_of(const SerialParams& p, int64_t s) {
    if (!p.ntok) return (int)p.T;
    const int64_t n = (int64_t)p.ntok[s] - p.t0;
    return (int)(n < 0 ? 0 : (n > p.T ? p.T : n));
}

template <int VEC, int CL>
__global__ void __launch_bounds__(128, 1)
decode_serial_kernel(const __grid_constant__ SerialParams rp, int V, const uint64_t* __restrict__ summ,
                     lac_dec_state* __restrict__ state, const uint8_t* __restrict__ bytes,
                     const int64_t* __restrict__ offsets, int32_t* __restrict__ syms, int64_t sym_stride, int P) {
    const int lane = threadIdx.x & 31;
    const int64_t s = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (s >= rp.n_streams) return;
    const int Ts = tokens_of(rp, s);
    if (Ts <= 0) return;
    constexpr int words = 32 * CL;
    const int G = lq::groups_of(V);
    auto seg = [&](int gw) { return 4 * lq::seg_group<CL>(gw, G); };  // first element of segment gw
    int64_t low = state[s].low, high = state[s].high, value = state[s].value;
    uint64_t pos = state[s].pos;
    const uint8_t* data = bytes + offsets[s];
    const uint64_t nbytes = (uint64_t)(offsets[s + 1] - offsets[s]);
    uint64_t wb = pos >> 3;  // the window: stream bytes [wb, wb + 24), big-endian words
    uint64_t hi64 = load_be64(data, nbytes, wb), lo64 = load_be64(data, nbytes, wb + 8);
    uint64_t nx64 = load_be64(data, nbytes, wb + 16);
    const float* row = rp.base + s * rp.so;
    const uint64_t* tab = summ + (s * rp.T) * words;
    RowSum<CL> cur, nxt;
    cur.load(tab, lane);
    cur.align();
    cur.scan(lane);
    lq::Scale sc = lq::make_scale(cur.Q, V);
    nxt = cur;
    if (Ts > 1) nxt.load(tab + words, lane);
    for (int t = 0; t < Ts; t++, tab += words, row += rp.st) {
        const uint64_t w = (uint64_t)(high - low + 1), xr = (uint64_t)(value - low);
        const uint32_t target = lq::div_q32(xr >> 32, xr << 32, w);
        // ---- level 1: lane l looks at the segments l * CL .. l * CL + CL - 1
        int best = -1;
        uint64_t Cb = 0;
        uint32_t cb = 0;
#pragma unroll
        for (int c = 0; c < CL; c++) {
            const int gw = lane * CL + c;
            const uint64_t C = cur.W[c];
            const int eb = seg(gw), ee = seg(gw + 1);
            const bool okw = (eb < min(ee, V)) & (lq::cum_of(C, (uint32_t)eb, sc) <= target);
            best = okw ? gw : best;
            Cb = okw ? C : Cb;
            cb = okw ? cur.code[c] : cb;
        }
        const int gsel = __reduce_max_sync(0xffffffffu, best);  // >= 0: the first non-empty segment starts at cum 0
        Cb = __shfl_sync(0xffffffffu, Cb, gsel / CL);
        cb = __shfl_sync(0xffffffffu, cb, gsel / CL);
        const int d = lq::shift_of(cur.r, cb);
        const uint32_t nref = lq::nref_of_code(cb);
        const int e0 = seg(gsel) + 32 * lane, eend = min(V, seg(gsel + 1));
        // ---- level 2: q of this lane's 32 consecutive elements.  All loads first (unconditional, from addresses
        // clamped into the segment), then branch-free arithmetic: the HBM latency is paid once per token.
        const lq::Scale sc_now = sc;
        auto advance = [&]() {  // while the segment is in flight: next token's scale, then the summary after that
            cur = nxt;
            cur.align();
            cur.scan(lane);  // (harmless on the last token: it rescans values nobody reads)
            sc = lq::make_scale(cur.Q, V);
            if (t + 2 < Ts) nxt.load(tab + 2 * words, lane);
        };
        uint32_t r[kPerThread];
        if (VEC == 4) {
            const int glast = eend - 4;  // the segment is not empty
            float4 x[kPerThread / 4];
#pragma unroll
            for (int p = 0; p < kPerThread / 4; p++)
                x[p] = __ldg(reinterpret_cast<const float4*>(row + min(e0 + 4 * p, glast)));
            advance();
#pragma unroll
            for (int p = 0; p < kPerThread / 4; p++) {
                const uint32_t m = (e0 + 4 * p < eend) ? 0xFFFFFFFFu : 0u;
                q_of2(x[p].x, x[p].y, nref, r[4 * p], r[4 * p + 1]);
                q_of2(x[p].z, x[p].w, nref, r[4 * p + 2], r[4 * p + 3]);
#pragma unroll
                for (int e = 0; e < 4; e++) r[4 * p + e] &= m;
            }
        } else {
            const int elast = eend - 1;
            float x[kPerThread];
#pragma unroll
            for (int j = 0; j < kPerThread; j++) x[j] = __ldg(row + min(e0 + j, elast));
            advance();
#pragma unroll
            for (int j = 0; j < kPerThread; j += 2) {
                q_of2(x[j], x[j + 1], nref, r[j], r[j + 1]);
                r[j] &= (e0 + j < eend) ? 0xFFFFFFFFu : 0u;
                r[j + 1] &= (e0 + j + 1 < eend) ? 0xFFFFFFFFu : 0u;
            }
        }
        uint32_t s4[kPerThread / 4];  // sums of 4 consecutive elements (< 2^31.5)
        uint64_t L = 0;
#pragma unroll
        for (int p = 0; p < kPerThread / 4; p++) {
            s4[p] = (r[4 * p] + r[4 * p + 1]) + (r[4 * p + 2] + r[4 * p + 3]);
            L += s4[p];
        }
        // in-segment prefixes stay unshifted (c); a boundary's row-wide cumulative is Cb + (c >> d)
        const uint64_t inc = warp_incl_scan(L, lane);
        const uint64_t cl = inc - L;
        auto cum_at = [&](uint64_t c, int e) { return lq::cum_of(Cb + lq::shr64(c, d), (uint32_t)e, sc_now); };
        const bool ok = (e0 < eend) & (cum_at(cl, e0) <= target);
        const unsigned ball = __ballot_sync(0xffffffffu, ok);  // lane 0 always qualifies (same test as level 1)
        const int src = 31 - __clz((int)ball);
        // ---- inside each lane (only lane `src` matters), branch-free: last group of 4 whose start qualifies,
        // then the last element of that group
        uint64_t cp = cl, cg = cl;
        int psel = 0;
#pragma unroll
        for (int p = 1; p < kPerThread / 4; p++) {
            cp += s4[p - 1];
            const bool okp = (e0 + 4 * p < eend) & (cum_at(cp, e0 + 4 * p) <= target);
            psel = okp ? p : psel;
            cg = okp ? cp : cg;
        }
        uint32_t qe[4] = {r[0], r[1], r[2], r[3]};
#pragma unroll
        for (int p = 1; p < kPerThread / 4; p++) {
#pragma unroll
            for (int e = 0; e < 4; e++) qe[e] = (p == psel) ? r[4 * p + e] : qe[e];
        }
        const int eg = e0 + 4 * psel;
        int sym = eg;
        uint64_t cs = cg, ce = cg;
        uint32_t qsym = qe[0];
#pragma unroll
        for (int e = 1; e < 4; e++) {
            ce += qe[e - 1];
            const bool oke = (eg + e < eend) & (cum_at(ce, eg + e) <= target);
            sym = oke ? eg + e : sym;
            cs = oke ? ce : cs;
            qsym = oke ? qe[e] : qsym;
        }
        uint32_t lo = cum_at(cs, sym);
        uint32_t hi = (sym == V - 1) ? 0u : cum_at(cs + qsym, sym + 1);
        sym = __shfl_sync(0xffffffffu, sym, src);
        lo = __shfl_sync(0xffffffffu, lo, src);
        hi = __shfl_sync(0xffffffffu, hi, src);
        // ---- A_from_bin.emit_symbol + emit_bit loop (arith_code.py:274-291), the same in every lane
        int64_t nl = low, nh = high;
        coder::ac_narrow32(nl, nh, lo, hi);
        const int64_t off = value - nl;  // the value stays inside [nl, nh]
        const int k = coder::renorm_count((uint64_t)(nh - nl + 1), P);
        coder::renorm_apply(nl, nh, P, k);
        const int o = (int)(pos - (wb << 3));  // next k bits from the window (k <= 60, o < 64)
        const uint64_t comb = o ? ((hi64 << o) | (lo64 >> (64 - o))) : hi64;
        const uint64_t nb = k ? (comb >> (64 - k)) : 0;
        low = nl;
        high = nh;
        value = nl + (off << k) + (int64_t)nb;
        pos += (uint64_t)k;
        if (o + k >= 64) {  // slide by 8 bytes; the word loaded now is not needed before the next slide
            hi64 = lo64;
            lo64 = nx64;
            wb += 8;
            nx64 = load_be64(data, nbytes, wb + 16);
        }
        if (lane == 0) syms[s * sym_stride + t] = sym;
    }
    if (lane == 0) {
        state[s].low = low;
        state[s].high = high;
        state[s].value = value;
        state[s].pos = pos;
        // bits consumed by renormalisation = pos - P; a valid stream holds at least that many
        if (pos - (uint64_t)P > (nbytes << 3)) state[s].status |= LAC_ST_TRUNC;
    }
}

__global__ void dec_init_kernel(lac_dec_state* state, int64_t n, int P, const uint8_t* bytes,
                                const int64_t* offsets) {
    int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= n) return;
    const uint8_t* data = bytes + offsets[s];
    uint64_t nbytes = (uint64_t)(offsets[s + 1] - offsets[s]);
    state[s].low = 0;
    state[s].high = (1ll << P) - 1;
    state[s].value = (int64_t)coder::read_bits(data, nbytes, 0, P);
    state[s].pos = (uint64_t)P;
    state[s].status = 0;
    state[s]._pad = 0;
}

// Decode = summary pass + serial pass per token chunk (~240k rows of a 32000-element vocabulary per chunk).
cudaError_t launch_decode(const float* logits, int64_t n_streams, int64_t T, int64_t stream_stride,
                          int64_t tok_stride, int V, const int32_t* ntok, lac_dec_state* state,
                          const uint8_t* bytes, const int64_t* offsets, int32_t* syms, int64_t sym_stride,
                          int P, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (n_streams == 0 || T == 0) return cudaSuccess;
    int parts = 1;
    const int vec = path_for(logits, V, stream_stride, tok_stride, &parts);
    if (vec < 0) return cudaErrorInvalidValue;
    int64_t tc = summ_rows_for(n_streams * T, parts, ws, ws_bytes) / n_streams;
    tc = tc < 1 ? 1 : (tc > T ? T : tc);
    Scratch sc;
    cudaError_t e = scratch_get(&sc, summ_bytes(n_streams * tc, parts), ws, ws_bytes, st);
    if (e != cudaSuccess) return e;
    uint64_t* summ = (uint64_t*)sc.p;
    const unsigned serial_blocks = (unsigned)((n_streams + 3) / 4);
    for (int64_t t0 = 0; t0 < T && e == cudaSuccess; t0 += tc) {
        const int64_t tn = T - t0 < tc ? T - t0 : tc;
        const float* base = logits + t0 * tok_stride;
        e = launch_summary(base, n_streams, tn, stream_stride, tok_stride, V, parts, vec, 0, summ, st);
        if (e != cudaSuccess) break;
        const SerialParams rp{base, n_streams, tn, stream_stride, tok_stride, ntok, t0};
#define LAC_SERIAL(CL_)                                                                                             \
    if (vec == 1)                                                                                                   \
        decode_serial_kernel<1, CL_><<<serial_blocks, 128, 0, st>>>(rp, V, summ, state, bytes, offsets, syms + t0,   \
                                                                    sym_stride, P);                                 \
    else                                                                                                            \
        decode_serial_kernel<4, CL_><<<serial_blocks, 128, 0, st>>>(rp, V, summ, state, bytes, offsets, syms + t0,   \
                                                                    sym_stride, P)
        LAC_BY_PARTS(parts, LAC_SERIAL)
#undef LAC_SERIAL
        e = cudaGetLastError();
    }
    const cudaError_t ef = scratch_put(&sc, st);
    return e != cudaSuccess ? e : ef;
}

cudaError_t launch_dec_init(lac_dec_state* state, int64_t n, int P, const uint8_t* bytes,
                            const int64_t* offsets, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    dec_init_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(state, n, P, bytes, offsets);
    return cudaGetLastError();
}

}  // namespace lac
