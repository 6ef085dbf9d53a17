// lq32.cuh -- the LQ32 logits -> integer CDF quantisation (DESIGN.md section 3), device side.
//
// Everything here is defined in individually rounded IEEE fp32 operations plus exact integer arithmetic, so
// oracle/lac_oracle.c (orc_lq32_*) reproduces it bit for bit, and as a function of (x, V) only: the result does not
// depend on how the work is spread over threads, warps or CTAs.
//
// Block form: the row is cut into NW = 32 * parts(V) segments of <= 1024 elements (one warp's work), every segment
// is quantised against ITS OWN reference exponent and the segment totals are aligned to the row-wide reference
// afterwards -- nothing needs the row maximum before the element pass, so the bandwidth-bound pass has no row-wide
// dependency at all (no cluster, no DSMEM, no second look at the data).
//
//   parts = ceil(V / 32768),  NW = 32 * parts,  G = ceil(V / 4)
//   segment w = elements [4 floor(w G / NW), min(V, 4 floor((w + 1) G / NW)))
// per segment:
//   m_w  = max x_i (NaN dropped),  n_w = bits(fma(m_w, log2e, 1.5 * 2^23))     t = fma(x, log2e, 1.5*2^23) is monotone
//                                               in x; its low mantissa bits are rne(x * log2e).  No "x - m" is formed.
//   r_w  = 0 (EMPTY) if n_w < kRefLo,  0xFFFFFF (POISON) if n_w >= kRefHi,  else n_w - kRefLo + 1
//   t_i  = fma(x_i, log2e, 1.5 * 2^23),  sh_i = n_w - bits(t_i)      (unsigned; >= 32 for -inf and NaN)
//   f_i  = fma(x_i, log2e, 1.5 * 2^23 - t_i)       in [-0.5, 0.5], single rounding
//   z_i  = fma(fma(fma(c3, f, c2), f, c1), f, 1.5 * 2^25)     c_k = minimax 2^f coefficients * 2^24; z in [2^25, 2^26)
//   q_i  = sh_i >= 32 ? 0 : (bits(z_i) << 7) >> sh_i   mantissa(z) = rne(2^22 2^f) (max rel. error 1.02e-4); the
//                                               exponent field of that binade ends in 00, so bits(z) << 7 is the
//                                               clean integer mantissa << 7 < 2^29.5 and four q fit a uint32 sum.
//          No F2I anywhere: float->int conversion runs at 16 threads/clk/SM on B200 (measured limiter).
//   S_w  = sum q_i (< 2^39.5),  c_i = sum of q_j, j < i inside the segment;  summary word = (S_w << 24) | r_w
// per row:
//   r    = max r_w;  DEGENERATE when r is EMPTY or POISON: cum_i = i, so every symbol but the last gets 2^-32 and the
//                    last takes the rest (not a uniform table)
//   d_w  = r - r_w,  W_w = (r_w == 0 || d_w >= 40) ? 0 : S_w >> d_w,  Q = sum W_w
//   C_i  = sum_{w' < w} W_w' + (c_i >> d_w)
//   s    = bitlen(Q) - 1,  Qn = Q normalised to [2^31, 2^32),  R = floor(((2^32 - V) << 31) / (Qn + 1))
//   cum_i = ((C_i * R) >> s) + i,  cum_V = 2^32     => every frequency >= 1
//
// Replaces the reference's float table builders (llama_compress.py:24-30, arithmetic_coding.py:57-62); the
// quantisation differs from theirs by design.  Per element (DESIGN.md section 3, tests/test_lq32_accuracy.py):
// p_hat_i >= (1 - V/2^32)(1 - 2^-29)[(1 - d)/(1 + d) p_i - 2^-27.5 p_max], d = 1.025e-4, up to the fp32 rounding of
// log2e, for every element outside an EMPTY segment -- the polynomial's error is in the normaliser Q as well as in
// the element, so the relative deficit reaches 2d + V/2^32, not d.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace lq {

__device__ __forceinline__ float log2e() { return __uint_as_float(0x3FB8AA3Bu); }
__device__ __forceinline__ float magic() { return __uint_as_float(0x4B400000u); }   // 1.5 * 2^23
__device__ __forceinline__ float magicz() { return __uint_as_float(0x4C400000u); }  // 1.5 * 2^25
constexpr uint32_t kC1 = 0x4b317afdu, kC2 = 0x4a780626u, kC3 = 0x4961510cu;  // minimax 2^f, degree 3, * 2^24

__device__ __forceinline__ float neg_inf() { return __uint_as_float(0xFF800000u); }

constexpr int kRefLo = 0x4B000040, kRefHi = 0x4B800000;
constexpr uint32_t kPoison = 0xFFFFFFu;
constexpr int kPartElems = 32768;  // elements per part (one CTA tile of pass 1), 32 segments each
constexpr int kMaxParts = 8;

__host__ __device__ __forceinline__ int parts_of(int V) { return (V + kPartElems - 1) / kPartElems; }
__host__ __device__ __forceinline__ int groups_of(int V) { return (V + 3) >> 2; }
// first 4-element group of segment gw (gw = NW: one past the last group), NW = 32 * PARTS
template <int PARTS>
__device__ __forceinline__ int seg_group(int gw, int G) { return (int)(((uint32_t)gw * (uint32_t)G) / (uint32_t)(32 * PARTS)); }

// reference code of a segment from its float maximum
__device__ __forceinline__ uint32_t code_of_max(float m) {
    const int n = __float_as_int(__fmaf_rn(m, log2e(), magic()));
    return n < kRefLo ? 0u : (n >= kRefHi ? kPoison : (uint32_t)(n - kRefLo + 1));
}
// the exponent reference to quantise a segment against; dead codes give 0xFFFFFFFF, which makes every shift >= 32
__device__ __forceinline__ uint32_t nref_of_code(uint32_t code) {
    return (code == 0u || code == kPoison) ? 0xFFFFFFFFu : code - 1u + (uint32_t)kRefLo;
}
__device__ __forceinline__ uint64_t pack_word(uint64_t S, uint32_t code) { return (S << 24) | (uint64_t)code; }
__device__ __forceinline__ uint32_t word_code(uint64_t w) { return (uint32_t)w & 0xFFFFFFu; }
__device__ __forceinline__ uint64_t word_sum(uint64_t w) { return w >> 24; }
// right shift that aligns a segment (code) to the row reference r; 64 = the segment (or the whole row) counts as 0
__device__ __forceinline__ int shift_of(uint32_t r, uint32_t code) {
    const uint32_t d = r - code;
    return (r == 0u || r == kPoison || code == 0u || d >= 40u) ? 64 : (int)d;
}
__device__ __forceinline__ uint64_t shr64(uint64_t v, int d) { return d >= 64 ? 0ull : (v >> d); }

// scalar form of the per-element step (the kernels use the packed two-lane version)
__device__ __forceinline__ uint32_t q_of(float x, uint32_t nref) {
    float t = __fmaf_rn(x, log2e(), magic());
    uint32_t sh = nref - __float_as_uint(t);
    float f = __fmaf_rn(x, log2e(), __fsub_rn(magic(), t));
    float p = __uint_as_float(kC3);
    p = __fmaf_rn(p, f, __uint_as_float(kC2));
    p = __fmaf_rn(p, f, __uint_as_float(kC1));
    float z = __fmaf_rn(p, f, magicz());
    return __funnelshift_rc(__float_as_uint(z) << 7, 0u, sh);  // (mantissa << 7) >> min(sh, 32)
}

struct Scale {
    uint64_t Q;
    uint32_t R;
    int s;
};

// floor(((hi << 64) | lo) / den) for a quotient known to fit 32 bits (den < 2^62, den >= 1): fp64 estimate, then
// an exact fix-up.  The estimate is num * (1 / den) with the reciprocal from MUFU.RCP64H (rcp.approx.ftz.f64,
// ~20 bits) refined by two Newton steps (relative error ~2^-52), so the truncated product is within one of the
// true quotient; the remainder test below corrects up to two in either direction.  (A __ddiv_rz here costs a
// ~150-clock subroutine call on the serial decode path.)  Branch-free, so lanes can divide different operands.
__device__ __forceinline__ uint32_t div_q32(uint64_t hi, uint64_t lo, uint64_t den) {
    const double d = (double)den;
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
    r = __fma_rn(__fma_rn(-d, r, 1.0), r, r);
    r = __fma_rn(__fma_rn(-d, r, 1.0), r, r);
    const double num = __fma_rn((double)hi, 18446744073709551616.0, (double)lo);
    uint64_t q = (uint64_t)__dmul_rz(num, r);
#pragma unroll
    for (int pass = 0; pass < 2; pass++) {
        // remainder rem = num - q * den as a signed 128-bit value, via 64-bit halves
        const uint64_t plo = q * den, phi = __umul64hi(q, den);
        const uint64_t rlo = lo - plo;
        const int64_t rhi = (int64_t)(hi - phi - (lo < plo ? 1u : 0u));
        const bool neg = rhi < 0;
        const bool big = !neg && (rhi > 0 || rlo >= den);
        q = q - (neg ? 1u : 0u) + (big ? 1u : 0u);
    }
    return (uint32_t)q;
}

__device__ __forceinline__ Scale make_scale(uint64_t Q, int V) {
    Scale k;
    k.Q = Q;
    k.R = 0;
    k.s = 0;
    if (Q >= (1ull << 28)) {  // else: the degenerate Q == 0 row
        k.s = 63 - __clzll((long long)Q);  // >= 28: the row maximum contributes q >= 2^28.5
        const uint64_t N = ((1ull << 32) - (uint64_t)V) << 31;
        const uint64_t D = (k.s >= 31 ? (Q >> (k.s - 31)) : (Q << (31 - k.s))) + 1;  // (2^31, 2^32]
        k.R = div_q32(0, N, D);  // R = floor(N / D) <= M * 2^s / Q
    }
    return k;
}

// ((C * R) >> s) + i ; C < 2^49, R < 2^32, s <= 48.
__device__ __forceinline__ uint32_t cum_of(uint64_t C, uint32_t i, const Scale& k) {
    uint64_t lo = C * (uint64_t)k.R;
    uint64_t hi = __umul64hi(C, (uint64_t)k.R);
    uint64_t v = k.s == 0 ? lo : ((lo >> k.s) | (hi << (64 - k.s)));
    return (uint32_t)v + i;
}

}  // namespace lq
