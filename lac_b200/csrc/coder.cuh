// coder.cuh -- range-narrowing state machines of the reference, device side.
//
//   arith_code.py:156-246    A_to_bin   (receive_symbol, decide_bit/emit_bit, flush)
//   arith_code.py:248-334    A_from_bin (as a value-tracking decoder: the symbol emitted is
//                            always the one whose range contains the stream's value)
//   arithmetic_coding.py:129-208  Region.step/emit + CarryBuffer (same renormalisation,
//                            floor-mapped sub-intervals, middle-third flush)
//
// The reference emits one bit per loop iteration; here the k renormalisation bits of a
// token are produced at once: after k doublings l_k = (l_0 mod 2^(P-k)) * 2^k and the bits
// are E = floor(l_0 / 2^(P-k)), which may carry (E >= 2^k) into bits already written, or
// borrow (E < 0, flush only).  BitWriter resolves that exactly like A_to_bin.encode's
// r = (r << 1) + v (arith_code.py:212-219) / CarryBuffer.add (arithmetic_coding.py:198-202).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/lac_b200.h"

namespace coder {

typedef unsigned __int128 u128;
typedef __int128 i128;

// ---------------------------------------------------------------- bit output
struct BitWriter {
    uint8_t* out;
    uint64_t cap;    // bytes
    uint64_t nbits;  // bits emitted so far, including the `nacc` bits still in `acc`
    int64_t acc;     // value of the last nacc bits
    int nacc;        // 0..7 between calls
    uint32_t status;

    __device__ void open(uint8_t* o, uint64_t c, uint64_t nb, uint32_t st) {
        out = o;
        cap = c;
        nbits = nb;
        nacc = (int)(nb & 7);
        acc = 0;
        status = st;
        if (nacc && (nb >> 3) < cap) acc = out[nb >> 3] >> (8 - nacc);
    }
    // add E (signed, |E| < 2^(k+3)) as the next k bits, k <= 40
    __device__ void append_small(int64_t E, int k) {
        if (status & LAC_ST_CAP) {  // a truncated stream is never touched again (no ripple into foreign bytes)
            nbits += (uint64_t)k;
            return;
        }
        int64_t a = (acc << k) + E;
        int n = nacc + k;
        int64_t c = a >> n;  // carry (>0) or borrow (<0) into bytes already stored
        a -= c << n;
        uint64_t stored = (nbits - (uint64_t)nacc) >> 3;
        while (c != 0 && stored > 0) {
            stored--;
            int64_t t = (int64_t)out[stored] + c;
            out[stored] = (uint8_t)(t & 255);
            c = t >> 8;
        }
        nbits += (uint64_t)k;
        while (n >= 8) {
            uint64_t pos = (nbits - (uint64_t)n) >> 3;
            n -= 8;
            if (pos < cap) out[pos] = (uint8_t)((a >> n) & 255);
            else status |= LAC_ST_CAP;
        }
        acc = a & ((1ll << n) - 1);
        nacc = n;
    }
    __device__ void append(int64_t E, int k) {
        if (k > 32) {
            int k2 = k - 32;
            append_small(E >> k2, 32);  // arithmetic shift keeps carries / borrows in the high part
            append_small(E & ((1ll << k2) - 1), k2);
        } else if (k > 0 || E != 0) {
            append_small(E, k);
        }
    }
    // store the partial byte zero-padded (group_bits' tail, arith_code.py:343-347); the bits
    // stay accounted in nbits so a later open() resumes mid-byte.
    __device__ void close() {
        if (nacc && !(status & LAC_ST_CAP)) {
            uint64_t pos = nbits >> 3;
            if (pos < cap) out[pos] = (uint8_t)(acc << (8 - nacc));
            else status |= LAC_ST_CAP;
        }
    }
};

// ---------------------------------------------------------------- staged bit output (fused encoder)
// Same arithmetic as BitWriter, but complete bytes go to a per-stream shared-memory stage that the whole block
// flushes to global memory in coalesced pieces after the coding phase; carries and borrows ripple through the
// stage first and only reach global memory (read-modify-write of bytes flushed by an earlier pass) in the rare case
// that they run past it.  The caller flushes stage[0 .. fill) to out[base .. base + fill) and calls flushed().
struct StagedWriter {
    uint8_t* out;    // the stream's region in global memory
    uint8_t* stage;  // shared memory, kStage bytes
    uint64_t cap;    // bytes of the stream's region
    uint64_t nbits;  // bits emitted so far, including the nacc bits still in acc
    uint64_t base;   // stream byte index of stage[0]
    int64_t acc;     // value of the last nacc bits
    int nacc;        // 0..7 between calls
    int fill;        // staged bytes
    int tail;        // 1: stage[fill] holds the zero-padded partial byte (flush fill + tail bytes)
    uint32_t status;
    static constexpr int kStage = 160;

    __device__ void open(uint8_t* o, uint8_t* stg, uint64_t c, uint64_t nb, uint32_t st) {
        out = o;
        stage = stg;
        cap = c;
        nbits = nb;
        nacc = (int)(nb & 7);
        base = nb >> 3;
        fill = 0;
        tail = 0;
        acc = 0;
        status = st;
        if (nacc && base < cap) acc = out[base] >> (8 - nacc);
    }
    __device__ void spill() {  // stage full inside a pass (k near 60 for many tokens in a row): the thread writes it out
        for (int i = 0; i < fill; i++) out[base + (uint64_t)i] = stage[i];
        base += (uint64_t)fill;
        fill = 0;
    }
    __device__ void flushed() {
        base += (uint64_t)fill;
        fill = 0;
    }
    __device__ void append_small(int64_t E, int k) {  // add E (signed, |E| < 2^(k+3)) as the next k bits, k <= 40
        if (status & LAC_ST_CAP) {  // a truncated stream is never touched again
            nbits += (uint64_t)k;
            return;
        }
        int64_t a = (acc << k) + E;
        int n = nacc + k;
        int64_t c = a >> n;  // carry (>0) or borrow (<0) into bytes already produced
        a -= c << n;
        if (c != 0) {
            int i = fill;
            while (c != 0 && i > 0) {
                i--;
                const int64_t t = (int64_t)stage[i] + c;
                stage[i] = (uint8_t)(t & 255);
                c = t >> 8;
            }
            uint64_t g = base;
            while (c != 0 && g > 0) {
                g--;
                const int64_t t = (int64_t)out[g] + c;
                out[g] = (uint8_t)(t & 255);
                c = t >> 8;
            }
        }
        nbits += (uint64_t)k;
        while (n >= 8) {
            n -= 8;
            if (base + (uint64_t)fill < cap) {
                if (fill == kStage) spill();
                stage[fill++] = (uint8_t)((a >> n) & 255);
            } else {
                status |= LAC_ST_CAP;
            }
        }
        acc = a & ((1ll << n) - 1);
        nacc = n;
    }
    __device__ void append(int64_t E, int k) {
        if (k > 32) {
            const int k2 = k - 32;
            append_small(E >> k2, 32);  // arithmetic shift keeps carries / borrows in the high part
            append_small(E & ((1ll << k2) - 1), k2);
        } else if (k > 0 || E != 0) {
            append_small(E, k);
        }
    }
    // the partial byte, zero-padded (group_bits' tail, arith_code.py:343-347), goes behind the staged bytes; it stays
    // accounted in nbits only, so a later open() resumes mid-byte
    __device__ void close() {
        if (nacc && !(status & LAC_ST_CAP)) {
            if (base + (uint64_t)fill < cap) {
                if (fill == kStage) spill();
                stage[fill] = (uint8_t)(acc << (8 - nacc));
                tail = 1;
            } else {
                status |= LAC_ST_CAP;
            }
        }
    }
};

// ---------------------------------------------------------------- bit input
// k bits starting at bit `pos` of data[0..nbytes), MSB first, zeros past the end
// (A_from_bin sees no more bits; ACSampler substitutes 0, arithmetic_coding.py:102-107).
__device__ __forceinline__ uint64_t read_bits(const uint8_t* data, uint64_t nbytes, uint64_t pos, int k) {
    if (k <= 0) return 0;
    uint64_t first = pos >> 3, last = (pos + (uint64_t)k - 1) >> 3;
    u128 acc = 0;
    for (uint64_t b = first; b <= last; b++) acc = (acc << 8) | (u128)(b < nbytes ? data[b] : 0);
    int drop = (int)(((last + 1) << 3) - (pos + (uint64_t)k));
    return (uint64_t)((acc >> drop) & ((((u128)1) << k) - 1));
}

// ---------------------------------------------------------------- renormalisation
// Number of doublings the reference loop performs for a width `span` (arith_code.py:176-180
// `(h-l) < decision`; arithmetic_coding.py:170 `span*2 <= one`).
__device__ __forceinline__ int renorm_count(uint64_t span, int P) {
    if (span > (1ull << (P - 1))) return 0;
    int e = 63 - __clzll((long long)span);
    return ((span & (span - 1)) == 0) ? (P - e) : (P - 1 - e);
}

// Apply k doublings to (l, h); returns the emitted bit value E (see file header).
__device__ __forceinline__ int64_t renorm_apply(int64_t& l, int64_t& h, int P, int k) {
    if (k == 0) return 0;
    uint64_t span = (uint64_t)(h - l + 1);
    int64_t E = l >> (P - k);
    l = (l & ((1ll << (P - k)) - 1)) << k;
    h = l + (int64_t)(span << k) - 1;
    return E;
}

// ---------------------------------------------------------------- A_to_bin pieces
// ceil(c * w / 2^32) for c <= 2^32, w <= 2^62: symbol_to_range (arith_code.py:105-109) on the
// fixed total d = 2^32.
__device__ __forceinline__ uint64_t scale32_ceil(uint64_t c, uint64_t w) {
    u128 p = (u128)c * w + 0xFFFFFFFFull;
    return (uint64_t)(p >> 32);
}

// receive_symbol (arith_code.py:169-175) with (lo, hi) on total 2^32; hi == 0 means 2^32.
__device__ __forceinline__ void ac_narrow32(int64_t& l, int64_t& h, uint32_t lo, uint32_t hi) {
    uint64_t w = (uint64_t)(h - l + 1);
    uint64_t r0 = scale32_ceil(lo, w);
    uint64_t r1 = hi ? scale32_ceil(hi, w) : w;
    h = l + (int64_t)r1 - 1;
    l += (int64_t)r0;
}

// One token of A_to_bin on a (lo, hi) pair of the lookup: narrow, renormalise, append the k bits.  Returns false,
// coding nothing, when the stream must stop.  A pair with hi != 0 && hi <= lo codes no interval:
// (0xFFFFFFFF, 0xFFFFFFFF) is the lookup's sentinel for a symbol outside [0, V) -> LAC_ST_SYMBOL (the reference
// raises "unknown symbol", arith_code.py:100-101), any other such pair is a zero-width symbol -> LAC_ST_TABLE (the
// reference would never terminate).  A stream that is already truncated (LAC_ST_CAP) codes nothing more.
template <class Writer>
__device__ __forceinline__ bool code_pair(int64_t& l, int64_t& h, uint2 pr, int P, Writer& bw) {
    if (pr.y != 0 && pr.y <= pr.x) {
        bw.status |= (pr.x == 0xFFFFFFFFu && pr.y == 0xFFFFFFFFu) ? LAC_ST_SYMBOL : LAC_ST_TABLE;
        return false;
    }
    if (bw.status & LAC_ST_CAP) return false;
    ac_narrow32(l, h, pr.x, pr.y);
    const int k = renorm_count((uint64_t)(h - l + 1), P);
    bw.append(renorm_apply(l, h, P, k), k);
    return true;
}

__device__ __forceinline__ int64_t region_overlap(int64_t a, int64_t b, int64_t c, int64_t d) {
    int64_t lo = a > c ? a : c, hi = b < d ? b : d;
    int64_t v = hi - lo + 1;
    return v > 0 ? v : 0;
}

// A_to_bin.flush (arith_code.py:193-202), literal: at most P + 2 iterations.
template <class Writer>
__device__ inline void ac_flush(int64_t& l, int64_t& h, int P, Writer& bw) {
    const int64_t denom = 1ll << P, decision = 1ll << (P - 1);
    while (l > 0 || h + 1 < denom) {
        int64_t b = l >> (P - 1);  // floor(l / decision), l may be negative
        if (region_overlap(l, h, b * decision, (b + 1) * decision) <
            region_overlap(l, h, (b + 1) * decision, (b + 2) * decision))
            b += 1;
        l = l * 2 - b * denom;
        h = h * 2 + 1 - b * denom;
        bw.append(b, 1);
    }
    l = 0;
    h = denom - 1;
}

}  // namespace coder
