// table_coders.cu -- A_to_bin / A_from_bin on tables the caller supplies (the reference-parity coders).
//
// One encode kernel and one decode kernel drive every table model.  The driver does the per-token step once: load
// the state, clip to ntok, check the symbol, narrow (h = l + r1 - 1, l += r0), renormalise, append the bits (encode)
// or pull k bits of the code value (decode), stop on LAC_ST_CAP, flush, close and store.  A model only says how a
// token becomes the offsets (r0, r1) inside the width w, and how a code value becomes a symbol:
//   Uniform  Predictor(n) (arith_code.py:64-74), one thread per stream
//   Cdf      int64 inclusive cumulative tables exactly as CDFPredictor.dist holds them, one warp per stream, including
//            fudged_dist (arith_code.py:83-93) evaluated as a parallel prefix-max:
//              p_i = p_{i-1} + max(1, min(w - p_{i-1} - V + i + 1, f_i - p_{i-1}))
//                  = max(p_{i-1} + 1, g_i),   g_i = min(w - V + i + 1, f_i)
//              =>  p_i - i = max(1, max_{j<=i} (g_j - j))
//            which holds for arbitrary f_i (also the wrapped int64 products of Llama_AC, flag LAC_F_WRAP64).
//   Acs      ACSampler / Region semantics (arithmetic_coding.py) on uint64 tables: one thread per stream encodes,
//            one warp per stream decodes.
//   Adaptive, AcsAdaptive   adaptive count models, prob(s) = counts[s] with counts[sym] += inc after every token, on
//            the Cdf resp. Acs arithmetic; one warp per stream keeps the stream's table in shared memory (the
//            per-stream hooks stream_begin / stream_accept / stream_end, empty for the static models).
// The models' data are in launch.h; range(m, ...) and symbol(m, ...) below are their device side.  Both return false,
// coding nothing, for a token the model cannot code (LAC_ST_TABLE).
#include <cstdint>
#include <cuda_runtime.h>

#include "coder.cuh"
#include "launch.h"

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

// ------------------------------------------------------------------ uniform Predictor(n) (arith_code.py:64-74)
// The reference's base class maps symbol s of n to [floor(s w / n), floor((s + 1) w / n)) -- floor, not the ceil of
// CDFPredictor.  AC() without arguments is AC(Predictor(3), 16).
__device__ __forceinline__ bool range(const Uniform& m, int64_t, int64_t, int sym, int64_t w, int, int64_t& r0,
                                      int64_t& r1) {
    const u128 W = (u128)(uint64_t)w;
    r0 = (int64_t)(((u128)(uint32_t)sym * W) / (uint32_t)m.n_symbols);  // symbol_to_range :69-70
    r1 = (int64_t)((((u128)(uint32_t)sym + 1) * W) / (uint32_t)m.n_symbols);
    return r1 > r0;  // zero-width symbol (w < n): the reference would never terminate
}
// The symbol whose floor-mapped range holds the code value, i.e. the largest s with floor(s w / n) <= x,
// s = floor(((x + 1) n - 1) / w).  (The reference's val_to_symbol, (v n) // w, is not that symbol at range
// boundaries; its decoder asserts there.  See tests/golden/ac_uniform.npz.)
__device__ __forceinline__ bool symbol(const Uniform& m, int64_t, int64_t, int64_t x, int64_t w, int, int& sym,
                                       int64_t& r0, int64_t& r1) {
    const u128 W = (u128)(uint64_t)w;
    const int64_t s = (int64_t)((((u128)(uint64_t)x + 1) * (uint32_t)m.n_symbols - 1) / W);
    r0 = (int64_t)(((u128)(uint64_t)s * W) / (uint32_t)m.n_symbols);
    r1 = (int64_t)((((u128)(uint64_t)s + 1) * W) / (uint32_t)m.n_symbols);
    sym = (int)s;
    return s < m.n_symbols && r1 > r0;
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

__device__ __forceinline__ bool range(const Cdf& m, int64_t s, int64_t t, int sym, int64_t w, int lane, int64_t& r0,
                                      int64_t& r1) {
    const TableCtx c = table_ctx(m.dist, m.n_symbols, m.ss, m.ts, m.minp, m.mss, m.mts, s, t, m.flags);
    return table_range(c, sym, w, lane, r0, r1);
}
__device__ __forceinline__ bool symbol(const Cdf& m, int64_t s, int64_t t, int64_t x, int64_t w, int lane, int& sym,
                                       int64_t& r0, int64_t& r1) {
    const TableCtx c = table_ctx(m.dist, m.n_symbols, m.ss, m.ts, m.minp, m.mss, m.mts, s, t, m.flags);
    sym = table_symbol(c, x, w, lane);
    return sym < m.n_symbols && table_range(c, sym, w, lane, r0, r1);
}

// ------------------------------------------------------------------ ACSampler on tables
// The token of the sample_scaled_cdf compress path (arithmetic_coding.py:85-87) narrows the region as Region.step does
// (arithmetic_coding.py:160-168): map(v, d) = low + span * v // d, the new region [map(c[i-1]), map(c[i]) - 1].  An
// empty region is LAC_ST_TABLE: the reference would never terminate.  c is one inclusive table of V entries.
__device__ __forceinline__ bool acs_range(const uint64_t* c, int V, int tok, int64_t w, int64_t& r0, int64_t& r1) {
    const uint64_t cl = tok ? c[tok - 1] : 0, ch = c[tok], den = c[V - 1];
    if (den == 0 || ch <= cl) return false;
    const u128 span = (u128)(uint64_t)w;
    r0 = (int64_t)(uint64_t)((span * cl) / den);
    r1 = (int64_t)(uint64_t)((span * ch) / den);
    return r1 > r0;
}
// The symbol whose encoder interval [map(c[i-1]), map(c[i]) - 1] contains the value:
// map(c) <= v  <=>  c <= ceil((v - low + 1) * den / span) - 1.  No zero-width check: that symbol holds the value.
__device__ __forceinline__ bool acs_symbol(const uint64_t* c, int V, int64_t x, int64_t w, int lane, int& tok,
                                           int64_t& r0, int64_t& r1) {
    const uint64_t den = c[V - 1];
    if (den == 0) return false;
    const u128 span = (u128)(uint64_t)w;
    const u128 tau = ((u128)(uint64_t)(x + 1) * den + span - 1) / span - 1;
    int64_t cnt = 0;
    for (int i = lane; i < V; i += 32) cnt += ((u128)c[i] <= tau);
    tok = (int)warp_sum_i64(cnt);
    if (tok >= V) return false;
    const uint64_t cl = tok ? c[tok - 1] : 0, ch = c[tok];
    r0 = (int64_t)(uint64_t)((span * cl) / den);
    r1 = (int64_t)(uint64_t)((span * ch) / den);
    return true;
}

__device__ __forceinline__ bool range(const Acs& m, int64_t s, int64_t t, int tok, int64_t w, int, int64_t& r0,
                                      int64_t& r1) {
    return acs_range(m.cdf + s * m.ss + t * m.ts, m.n_symbols, tok, w, r0, r1);
}
__device__ __forceinline__ bool symbol(const Acs& m, int64_t s, int64_t t, int64_t x, int64_t w, int lane, int& tok,
                                       int64_t& r0, int64_t& r1) {
    return acs_symbol(m.cdf + s * m.ss + t * m.ts, m.n_symbols, x, w, lane, tok, r0, r1);
}

// ------------------------------------------------------------------ adaptive count models
// prob(s) = counts[s], and after every token counts[sym] += inc (a ProbPredictor whose accept() counts).  The warp of
// a stream keeps the stream's table in shared memory as int64 inclusive cumulative values -- exactly the table the
// reference predictor builds before each token -- so the range and symbol arithmetic is that of the static models on
// the shared table: Adaptive is CDFPredictor (fudged_dist included, minp = the smallest positive count), AcsAdaptive
// is ACSampler.  Totals stay below 2^62 (kAdaptiveTotal): a token whose accept() would reach it is LAC_ST_TABLE.
constexpr int64_t kAdaptiveTotal = 1ll << 62;

__device__ __forceinline__ int64_t warp_min_i64(int64_t v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        int64_t t = __shfl_xor_sync(0xffffffffu, v, o);
        v = t < v ? t : v;
    }
    return v;
}

// One stream of an adaptive model M, as the drivers see it between begin and end.
template <class M>
struct CountTable {
    int64_t* tbl;     // shared: the stream's inclusive cumulative counts
    int64_t* counts;  // global: the stream's counts, read at begin, written at end
    int V;
    int64_t inc;
    bool loaded;      // false: a count was negative or the total reached kAdaptiveTotal; nothing is coded or stored
};

// Load the stream's counts into its shared table, 32 at a time: a warp scan of each chunk plus the running total.
// Sums saturate at kAdaptiveTotal, so a table that reaches it (and is rejected) cannot overflow on the way.
template <class M>
__device__ inline CountTable<M> count_table(const M& m, int64_t s, int lane) {
    extern __shared__ int64_t count_tables[];  // one table of V entries per warp of the block (count_shape)
    CountTable<M> a;
    a.V = m.n_symbols;
    a.inc = m.inc;
    a.tbl = count_tables + (int64_t)(threadIdx.x / 32) * a.V;
    a.counts = m.counts + s * a.V;
    const uint64_t lim = (uint64_t)kAdaptiveTotal;
    uint64_t run = 0;
    bool bad = false;
    for (int b = 0; b < a.V; b += 32) {
        const int i = b + lane;
        const int64_t c = i < a.V ? a.counts[i] : 0;
        bad |= c < 0;
        uint64_t v = c < 0 ? 0 : ((uint64_t)c < lim ? (uint64_t)c : lim);
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint64_t u = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o) v = v + u < lim ? v + u : lim;
        }
        v = v + run < lim ? v + run : lim;
        if (i < a.V) a.tbl[i] = (int64_t)v;
        run = __shfl_sync(0xffffffffu, v, 31);
    }
    a.loaded = !__any_sync(0xffffffffu, bad) && run < lim;
    __syncwarp();
    return a;
}

// CDFPredictor on the shared table.  minp only matters once the total exceeds the width (fudged_dist needs
// total > w * minp, and minp >= 1), so the warp looks for the smallest positive count only then.
template <class M>
__device__ __forceinline__ TableCtx count_ctx(const CountTable<M>& a, int64_t w, int lane) {
    TableCtx c;
    c.tbl = a.tbl;
    c.V = a.V;
    c.minp = 1;
    c.wrap = 0;
    if (a.tbl[a.V - 1] > w) {
        int64_t mn = kAdaptiveTotal;
        for (int i = lane; i < a.V; i += 32) {
            const int64_t f = a.tbl[i] - (i ? a.tbl[i - 1] : 0);
            if (f > 0 && f < mn) mn = f;
        }
        c.minp = warp_min_i64(mn);
    }
    return c;
}
// room for this token's accept() below kAdaptiveTotal
template <class M>
__device__ __forceinline__ bool count_room(const CountTable<M>& a) {
    return a.tbl[a.V - 1] < kAdaptiveTotal - a.inc;
}

__device__ __forceinline__ bool range(const CountTable<Adaptive>& a, int64_t, int64_t, int sym, int64_t w, int lane,
                                      int64_t& r0, int64_t& r1) {
    return count_room(a) && table_range(count_ctx(a, w, lane), sym, w, lane, r0, r1);
}
__device__ __forceinline__ bool symbol(const CountTable<Adaptive>& a, int64_t, int64_t, int64_t x, int64_t w, int lane,
                                       int& sym, int64_t& r0, int64_t& r1) {
    if (!count_room(a)) return false;
    const TableCtx c = count_ctx(a, w, lane);
    sym = table_symbol(c, x, w, lane);
    return sym < a.V && table_range(c, sym, w, lane, r0, r1);
}
__device__ __forceinline__ bool range(const CountTable<AcsAdaptive>& a, int64_t, int64_t, int tok, int64_t w, int,
                                      int64_t& r0, int64_t& r1) {
    return count_room(a) && acs_range((const uint64_t*)a.tbl, a.V, tok, w, r0, r1);
}
__device__ __forceinline__ bool symbol(const CountTable<AcsAdaptive>& a, int64_t, int64_t, int64_t x, int64_t w,
                                       int lane, int& tok, int64_t& r0, int64_t& r1) {
    return count_room(a) && acs_symbol((const uint64_t*)a.tbl, a.V, x, w, lane, tok, r0, r1);
}

// ------------------------------------------------------------------ per-stream model hooks
// stream_begin(m, s, lane) gives what range / symbol work on for stream s: the model itself for the static models,
// whose other hooks are empty, and the stream's shared table for the adaptive ones.  stream_accept follows every token
// that narrowed the interval, stream_end the last one.  Every lane of a stream calls every hook.
template <class M>
__device__ __forceinline__ const M& stream_begin(const M& m, int64_t, int) { return m; }
template <class M>
__device__ __forceinline__ bool stream_loaded(const M&) { return true; }
template <class M>
__device__ __forceinline__ void stream_accept(const M&, int, int) {}
template <class M>
__device__ __forceinline__ void stream_end(const M&, int) {}

__device__ __forceinline__ CountTable<Adaptive> stream_begin(const Adaptive& m, int64_t s, int lane) {
    return count_table(m, s, lane);
}
__device__ __forceinline__ CountTable<AcsAdaptive> stream_begin(const AcsAdaptive& m, int64_t s, int lane) {
    return count_table(m, s, lane);
}
template <class M>
__device__ __forceinline__ bool stream_loaded(const CountTable<M>& a) { return a.loaded; }
// counts[sym] += inc: entries sym .. V-1 of the cumulative table
template <class M>
__device__ __forceinline__ void stream_accept(const CountTable<M>& a, int sym, int lane) {
    if (a.inc == 0) return;
    __syncwarp();  // every lane has read this token's table
    for (int i = sym + lane; i < a.V; i += 32) a.tbl[i] += a.inc;
    __syncwarp();
}
// the table goes back as counts
template <class M>
__device__ __forceinline__ void stream_end(const CountTable<M>& a, int lane) {
    if (!a.loaded) return;
    for (int i = lane; i < a.V; i += 32) a.counts[i] = a.tbl[i] - (i ? a.tbl[i - 1] : 0);
}

// ------------------------------------------------------------------ drivers
// LANES threads per stream (1 or 32).  With 32, the model's lanes cooperate on a token and only lane 0 appends,
// writes symbols and stores the state.  With 1, threads past n_streams return early: no warp collectives there.
template <class Model, int LANES>
__global__ void table_encode_kernel(const Model m, const int32_t* __restrict__ syms, int64_t sym_stride,
                                    int64_t n_streams, int64_t T, const int32_t* __restrict__ ntok,
                                    lac_enc_state* __restrict__ state, uint8_t* __restrict__ out, int64_t out_stride,
                                    int flush, int P) {
    const int lane = threadIdx.x % LANES;
    const int64_t s = (int64_t)(((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) / LANES);
    if (s >= n_streams) return;
    int64_t l = state[s].low, h = state[s].high;
    coder::BitWriter bw;
    bw.open(out + s * out_stride, (uint64_t)out_stride, state[s].nbits, state[s].status);
    const auto& ms = stream_begin(m, s, lane);  // a stream whose table does not load codes nothing: LAC_ST_TABLE
    const int64_t Ts = !stream_loaded(ms) ? 0 : ntok ? (int64_t)ntok[s] : T;
    for (int64_t t = 0; t < Ts; t++) {
        const int sym = syms[s * sym_stride + t];
        if (sym < 0 || sym >= m.n_symbols) {
            bw.status |= LAC_ST_SYMBOL;
            break;
        }
        int64_t r0, r1;
        if (!range(ms, s, t, sym, h - l + 1, lane, r0, r1)) {
            bw.status |= LAC_ST_TABLE;
            break;
        }
        h = l + r1 - 1;  // receive_symbol :169-175
        l += r0;
        stream_accept(ms, sym, lane);
        const int k = coder::renorm_count((uint64_t)(h - l + 1), P);
        const int64_t E = coder::renorm_apply(l, h, P, k);
        if (lane == 0) bw.append(E, k);
        uint32_t st = bw.status;
        if constexpr (LANES > 1) st = __shfl_sync(0xffffffffu, st, 0);
        if (st & LAC_ST_CAP) break;
    }
    if (!stream_loaded(ms)) bw.status |= LAC_ST_TABLE;
    stream_end(ms, lane);
    if (lane != 0) return;
    if (flush != kFlushNone && !(bw.status & (LAC_ST_TABLE | LAC_ST_SYMBOL | LAC_ST_CAP))) {
        if (flush == kFlushCompress) {
            // ACSampler's flush_compress, arithmetic_coding.py:50-56: step(1, 2, 3), drain the carry buffer, reset.
            // Bit-exact with the reference, but the bits do not pin the final region (DESIGN.md section 6): the last
            // tokens may be undecodable by ANY decoder.
            const u128 span = (u128)(uint64_t)(h - l + 1);
            h = l + (int64_t)(uint64_t)(span * 2 / 3) - 1;
            l += (int64_t)(uint64_t)(span / 3);
            const int k = coder::renorm_count((uint64_t)(h - l + 1), P);
            bw.append(coder::renorm_apply(l, h, P, k), k);
            l = 0;
            h = (1ll << P) - 1;
        } else {
            // A_to_bin.flush (arith_code.py:193-202): shortest bit string whose every continuation stays inside
            // [l, h] -- always decodable
            coder::ac_flush(l, h, P, bw);
        }
    }
    bw.close();
    state[s].low = l;
    state[s].high = h;
    state[s].nbits = bw.nbits;
    state[s].status = bw.status;
}

// A value-tracking A_from_bin: the symbol is the one whose range holds the code value v, zeros past the end of the
// bytes.  A table decoder never sets LAC_ST_TRUNC.
template <class Model, int LANES>
__global__ void table_decode_kernel(const Model m, int64_t n_streams, int64_t T, const int32_t* __restrict__ ntok,
                                    lac_dec_state* __restrict__ state, const uint8_t* __restrict__ bytes,
                                    const int64_t* __restrict__ offsets, int32_t* __restrict__ syms,
                                    int64_t sym_stride, int P) {
    const int lane = threadIdx.x % LANES;
    const int64_t s = (int64_t)(((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) / LANES);
    if (s >= n_streams) return;
    int64_t l = state[s].low, h = state[s].high, v = state[s].value;
    uint64_t pos = state[s].pos;
    uint32_t status = state[s].status;
    const uint8_t* data = bytes + offsets[s];
    const uint64_t nbytes = (uint64_t)(offsets[s + 1] - offsets[s]);
    const auto& ms = stream_begin(m, s, lane);  // a stream whose table does not load decodes nothing: LAC_ST_TABLE
    const int64_t Ts = !stream_loaded(ms) ? 0 : ntok ? (int64_t)ntok[s] : T;
    for (int64_t t = 0; t < Ts; t++) {
        int sym;
        int64_t r0, r1;
        if (!symbol(ms, s, t, v - l, h - l + 1, lane, sym, r0, r1)) {
            status |= LAC_ST_TABLE;
            break;
        }
        h = l + r1 - 1;
        l += r0;
        stream_accept(ms, sym, lane);
        const int64_t off = v - l;
        const int k = coder::renorm_count((uint64_t)(h - l + 1), P);
        coder::renorm_apply(l, h, P, k);
        v = l + (off << k) + (int64_t)coder::read_bits(data, nbytes, pos, k);
        pos += (uint64_t)k;
        if (lane == 0) syms[s * sym_stride + t] = sym;
    }
    if (!stream_loaded(ms)) status |= LAC_ST_TABLE;
    stream_end(ms, lane);
    if (lane == 0) {
        state[s].low = l;
        state[s].high = h;
        state[s].value = v;
        state[s].pos = pos;
        state[s].status = status;
    }
}

// ------------------------------------------------------------------ launchers
// One lane per stream: blocks of 32 threads.  32 lanes per stream: blocks of 128 threads, 4 streams per block.  The
// adaptive models keep a V-entry int64 table per stream in dynamic shared memory: up to 4 streams per block within
// 48 KB, so V = 4096 (32 KB) runs one stream per block and no block needs the opt-in above 48 KB.
struct Shape {
    unsigned threads;
    size_t smem;
};
template <int LANES, class M>
Shape launch_shape(const M&) {
    return {LANES == 1 ? 32u : 128u, 0};
}
inline Shape count_shape(int V) {
    const size_t per = (size_t)V * sizeof(int64_t);
    size_t spb = (size_t(48) << 10) / per;
    spb = spb < 1 ? 1 : (spb > 4 ? 4 : spb);
    return {(unsigned)(32 * spb), spb * per};
}
template <int LANES>
Shape launch_shape(const Adaptive& m) {
    return count_shape(m.n_symbols);
}
template <int LANES>
Shape launch_shape(const AcsAdaptive& m) {
    return count_shape(m.n_symbols);
}

template <class M>
cudaError_t launch_table_encode(const M& m, const int32_t* syms, int64_t sym_stride, int64_t n, int64_t T,
                                const int32_t* ntok, lac_enc_state* state, uint8_t* out, int64_t out_stride, int flush,
                                int P, cudaStream_t st) {
    if (n == 0) return cudaSuccess;  // T == 0 is the flush-only call
    constexpr int lanes = M::kEncLanes;
    const Shape sh = launch_shape<lanes>(m);
    const unsigned spb = sh.threads / lanes;
    table_encode_kernel<M, lanes><<<(unsigned)((n + spb - 1) / spb), sh.threads, sh.smem, st>>>(
        m, syms, sym_stride, n, T, ntok, state, out, out_stride, flush, P);
    return cudaGetLastError();
}

template <class M>
cudaError_t launch_table_decode(const M& m, int64_t n, int64_t T, const int32_t* ntok, lac_dec_state* state,
                                const uint8_t* bytes, const int64_t* offsets, int32_t* syms, int64_t sym_stride, int P,
                                cudaStream_t st) {
    if (n == 0 || T == 0) return cudaSuccess;
    constexpr int lanes = M::kDecLanes;
    const Shape sh = launch_shape<lanes>(m);
    const unsigned spb = sh.threads / lanes;
    table_decode_kernel<M, lanes><<<(unsigned)((n + spb - 1) / spb), sh.threads, sh.smem, st>>>(
        m, n, T, ntok, state, bytes, offsets, syms, sym_stride, P);
    return cudaGetLastError();
}

#define LAC_TABLE_CODER(M)                                                                                          \
    template cudaError_t launch_table_encode(const M&, const int32_t*, int64_t, int64_t, int64_t, const int32_t*,    \
                                             lac_enc_state*, uint8_t*, int64_t, int, int, cudaStream_t);            \
    template cudaError_t launch_table_decode(const M&, int64_t, int64_t, const int32_t*, lac_dec_state*,            \
                                             const uint8_t*, const int64_t*, int32_t*, int64_t, int, cudaStream_t);
LAC_TABLE_CODER(Uniform)
LAC_TABLE_CODER(Cdf)
LAC_TABLE_CODER(Acs)
LAC_TABLE_CODER(Adaptive)
LAC_TABLE_CODER(AcsAdaptive)
#undef LAC_TABLE_CODER

}  // namespace lac
