/*
 * oracle/lac_oracle.c -- CPU restatement of pramasoul/lac's arithmetic-coding path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under lac_b200/ may import, link or call
 * this file; only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs use it, and only as the checker / reported CPU baseline.
 *
 * Parity status: PINNED.  Every orc_ac_* / orc_acs_* function below is checked
 * bit-for-bit against outputs of the real Python reference (imported from
 * /root/reference in the build container) by tests/golden/make_golden.py ->
 * tests/golden/*.npz -> tests/test_oracle_golden.py.
 *
 * Part 1 restates the reference (file:line cited per function).
 * Part 2 restates THIS repo's LQ32 logits->CDF quantisation spec (DESIGN.md
 * section 3) in exactly-rounded IEEE fp32 + integer ops so the CUDA kernels can be
 * compared bit-for-bit, plus the value-based N-token decoder the GPU uses.
 * Part 3 is the bulk CPU baseline (reference algorithm, C port, pthreads).
 *
 * All big-integer Python arithmetic is carried in __int128 (max magnitude on
 * this path: dist < 2^63 times width <= 2^62 -> < 2^125).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <pthread.h>
#include <unistd.h>

typedef __int128 i128;
typedef unsigned __int128 u128;

#define ORC_OK 0
#define ORC_E_ARG (-1)
#define ORC_E_CAP (-2)      /* output buffer too small */
#define ORC_E_SYMBOL (-3)   /* AssertionError("unknown symbol") arith_code.py:100-101 */
#define ORC_E_RANGE (-4)    /* AssertionError("predictor range does not correspond to val") arith_code.py:277-278 */
#define ORC_E_CARRY (-5)    /* carry out of the first bit / negative bit: cannot happen for valid input */
#define ORC_E_EMPTY (-6)    /* max() of empty range in A_from_bin.flush, arith_code.py:312 */
#define ORC_E_ZERODIV (-7)  /* ZeroDivisionError in A_from_bin.flush key, arith_code.py:305-307 */
#define ORC_E_INDEX (-8)    /* IndexError: ACSampler lookup ran off the cdf, arithmetic_coding.py:114-115 */

/* Python floor division for b > 0. */
static inline i128 fdiv(i128 a, i128 b) {
    i128 q = a / b;
    if ((a % b != 0) && ((a < 0) != (b < 0))) q -= 1;
    return q;
}
/* Python -(-(a)//b): ceil for b > 0.  arith_code.py:107,109 */
static inline i128 cdiv(i128 a, i128 b) { return -fdiv(-a, b); }
static inline i128 imin(i128 a, i128 b) { return a < b ? a : b; }
static inline i128 imax(i128 a, i128 b) { return a > b ? a : b; }

/* region_overlap, arith_code.py:59-61: inclusive [a,b] with inclusive [c,d]. */
static inline i128 region_overlap(i128 a, i128 b, i128 c, i128 d) {
    return imax(0, imin(d, b) - imax(a, c) + 1);
}

/* ------------------------------------------------------------------ */
/* Bit sink with carry resolution.  Restates what A_to_bin.encode       */
/* (arith_code.py:212-219: r = (r<<1) + v) and A_to_bin.bits            */
/* (arith_code.py:230-246) / CarryBuffer (arithmetic_coding.py:198-208) */
/* compute: the binary expansion of sum_i v_i 2^-i, v_i small signed ints. */
/* ------------------------------------------------------------------ */
typedef struct {
    uint8_t *bits;
    int64_t n, cap;
    int err;
} bitsink;

static void sink_push(bitsink *s, i128 v) {
    /* v may be negative: A_to_bin.flush (arith_code.py:193-202) emits floor(l/decision)
     * with l < 0, and encode()'s r = (r<<1) + v absorbs it as a borrow. */
    if (s->err) return;
    if (s->n >= s->cap) { s->err = ORC_E_CAP; return; }
    s->bits[s->n] = (uint8_t)(v & 1);
    i128 carry = v >> 1; /* arithmetic shift: floor */
    int64_t k = s->n - 1;
    while (carry) {
        if (k < 0) { s->err = ORC_E_CARRY; return; }
        i128 t = s->bits[k] + carry;
        s->bits[k] = (uint8_t)(t & 1);
        carry = t >> 1;
        k--;
    }
    s->n++;
}

/* group_bits (arith_code.py:336-347) == packbits + packbits.flush
 * (arithmetic_coding.py:212-225): MSB first, zero-pad the last byte. */
int64_t orc_pack_bits(const uint8_t *bits, int64_t nbits, uint8_t *out) {
    int64_t nb = (nbits + 7) / 8;
    memset(out, 0, (size_t)nb);
    for (int64_t i = 0; i < nbits; i++)
        if (bits[i]) out[i >> 3] |= (uint8_t)(0x80u >> (i & 7));
    return nb;
}
/* ungroup_bits (arith_code.py:348-351) == unpackbits (arithmetic_coding.py:227-230). */
void orc_unpack_bits(const uint8_t *bytes, int64_t nbytes, uint8_t *bits) {
    for (int64_t i = 0; i < nbytes; i++)
        for (int b = 0; b < 8; b++) bits[i * 8 + b] = (bytes[i] >> (7 - b)) & 1;
}

/* ------------------------------------------------------------------ */
/* CDFPredictor (arith_code.py:76-110)                                  */
/* ------------------------------------------------------------------ */
/* fudged_dist, arith_code.py:83-93.  Returns the table to use (dist or scratch). */
/* wrap64: Llama_AC keeps dist as a numpy int64 array (llama_compress.py:29), so the
 * inherited loop's `self.dist[i]*denom` is an np.int64 product that wraps mod 2^64
 * (numpy only warns).  wrap64=1 restates that literally; wrap64=0 is the exact-integer
 * behaviour CDFPredictor has with Python-int tables. */
static const int64_t *fudged_dist(const int64_t *dist, int V, i128 minp, i128 denom,
                                  int64_t *scratch, int wrap64) {
    /* arith_code.py:84; with Llama_AC, minp is np.int64 so denom*minp wraps as well */
    i128 thr = wrap64 ? (i128)(int64_t)((uint64_t)(int64_t)denom * (uint64_t)(int64_t)minp) : denom * minp;
    if ((i128)dist[V - 1] <= thr) return dist;
    i128 p = 0, last = dist[V - 1];
    for (int i = 0; i < V; i++) {
        i128 prod = wrap64 ? (i128)(int64_t)((uint64_t)dist[i] * (uint64_t)(int64_t)denom)
                           : (i128)dist[i] * denom;
        i128 d = fdiv(prod, last) - p;
        d = imax(1, imin(denom - p - V + i + 1, d));
        p += d;
        scratch[i] = (int64_t)p;
    }
    return scratch;
}
/* CDFPredictor.minp, arith_code.py:79: min positive pdf entry (0 if none: the
 * reference would raise ValueError; callers never pass such a table). */
int64_t orc_cdf_minp(const int64_t *dist, int V) {
    int64_t best = 0, prev = 0;
    for (int i = 0; i < V; i++) {
        int64_t p = dist[i] - prev;
        prev = dist[i];
        if (p > 0 && (best == 0 || p < best)) best = p;
    }
    return best;
}
/* Llama_AC.minp, llama_compress.py:43-45: min(dist[0], min(diff(dist))), zero allowed. */
int64_t orc_llama_minp(const int64_t *dist, int V) {
    int64_t best = dist[0];
    for (int i = 1; i < V; i++) {
        int64_t p = dist[i] - dist[i - 1];
        if (p < best) best = p;
    }
    return best;
}
/* symbol_to_range, arith_code.py:98-110 (same body as llama_compress.py:49-61). */
/* tbl == NULL: the uniform base class Predictor(V), arith_code.py:64-74 (floor-mapped). */
static int symbol_to_range(const int64_t *tbl, int V, int64_t s, i128 denom, i128 *r0, i128 *r1) {
    if (!tbl) {                                   /* Predictor.symbol_to_range :68-69: no bound on s (the */
        *r0 = fdiv((i128)s * denom, V);           /* decoder's flush() probes symbols past n - 1)          */
        *r1 = fdiv((i128)(s + 1) * denom, V);
        return ORC_OK;
    }
    if (s >= V || s < 0) return ORC_E_SYMBOL;
    i128 hd = tbl[s];
    i128 ld = s > 0 ? tbl[s - 1] : 0;
    i128 d = tbl[V - 1];
    *r0 = cdiv(ld * denom, d);
    *r1 = cdiv(hd * denom, d);
    return ORC_OK;
}
/* val_to_symbol, arith_code.py:94-97: bisect_right(dist, (v*dist[-1])//denom). */
static int64_t val_to_symbol(const int64_t *tbl, int V, i128 v, i128 denom) {
    if (!tbl) return (int64_t)fdiv(v * (i128)V, denom);   /* Predictor.val_to_symbol :66-67 */
    i128 target = fdiv(v * (i128)tbl[V - 1], denom);
    int64_t lo = 0, hi = V;
    while (lo < hi) {
        int64_t mid = (lo + hi) / 2;
        if (target < (i128)tbl[mid]) hi = mid; else lo = mid + 1;
    }
    return lo;
}

static inline const int64_t *table_at(const int64_t *dist, int64_t stride, int64_t ntab, int V,
                                      int64_t k, const int64_t *minp, i128 *mp) {
    if (stride == 0) { *mp = minp[0]; return dist; }
    if (k >= ntab) k = ntab - 1;   /* tests' TablePredictor repeats its last table */
    *mp = minp[k];
    return dist + k * stride;
}

/* ------------------------------------------------------------------ */
/* A_to_bin (arith_code.py:156-246)                                     */
/* ------------------------------------------------------------------ */
/*
 * dist     inclusive cumulative table(s) (CDFPredictor.dist), V entries each
 * stride   elements between consecutive positions' tables, 0 => one shared table
 * ntab     number of tables when stride != 0
 * minp     predictor.minp per table (1 entry when shared)
 * stop     run(..., stop): call flush() at the end (arith_code.py:207-211)
 * bits     carry-resolved bit string == list(A_to_bin.bits(symbols, stop))
 *          == binary digits of A_to_bin.encode(symbols, stop)
 * state_out (optional, 3 x int64): l, h, emitted_bits before flush.
 */
int orc_ac_encode(int prec, const int64_t *dist, int64_t stride, int64_t ntab, const int64_t *minp,
                  int V, const int32_t *syms, int64_t n, int stop, uint8_t *bits, int64_t cap,
                  int64_t *nbits, int64_t *state_out, int wrap64) {
    if (prec < 2 || prec > 62 || V < 1) return ORC_E_ARG;
    const i128 denom = (i128)1 << prec, decision = (i128)1 << (prec - 1);
    i128 l = 0, h = denom - 1;                                   /* :161-162 */
    int64_t *scratch = (int64_t *)malloc(sizeof(int64_t) * (size_t)V);
    bitsink sk = {bits, 0, cap, 0};
    int rc = ORC_OK;
    for (int64_t t = 0; t < n && !sk.err; t++) {
        /* receive_symbol :169-175 */
        i128 w = h - l + 1, mp, r0, r1;
        const int64_t *tbl = NULL;
        if (dist) {
            const int64_t *raw = table_at(dist, stride, ntab, V, t, minp, &mp);
            tbl = fudged_dist(raw, V, mp, w, scratch, wrap64);
        }
        if (syms[t] < 0 || syms[t] >= V) { rc = ORC_E_SYMBOL; break; }
        rc = symbol_to_range(tbl, V, syms[t], w, &r0, &r1);
        if (rc) break;
        if (r1 <= r0) { rc = ORC_E_ZERODIV; break; }   /* zero-width symbol: the reference loops forever */
        h = l + r1 - 1;
        l += r0;
        /* step :187-192 / decide_bit :176-180 / emit_bit :181-186 */
        while ((h - l) < decision) {
            i128 b = fdiv(l, decision);
            l = l * 2 - b * denom;
            h = h * 2 + 1 - b * denom;
            sink_push(&sk, b);
            if (sk.err) break;
        }
    }
    if (state_out) { state_out[0] = (int64_t)l; state_out[1] = (int64_t)h; state_out[2] = sk.n; }
    if (!rc && !sk.err && stop) {
        /* flush :193-202 */
        while (l > 0 || h + 1 < denom) {
            i128 b = fdiv(l, decision);
            if (region_overlap(l, h, b * decision, (b + 1) * decision) <
                region_overlap(l, h, (b + 1) * decision, (b + 2) * decision))
                b += 1;
            l = l * 2 - b * denom;
            h = h * 2 + 1 - b * denom;
            sink_push(&sk, b);
            if (sk.err) break;
        }
    }
    free(scratch);
    *nbits = sk.n;
    return rc ? rc : sk.err;
}

/* ------------------------------------------------------------------ */
/* A_from_bin (arith_code.py:248-334): literal bit-at-a-time decoder,   */
/* including its flush() heuristic (extra trailing symbols).            */
/* ------------------------------------------------------------------ */
typedef struct {
    int prec, V;
    i128 denom, decision, l, h, lb, hb;
    const int64_t *dist; int64_t stride, ntab; const int64_t *minp;
    int64_t *scratch; int wrap64;
    int32_t *out; int64_t nout, cap;
} afb;

static const int64_t *afb_table(afb *d, i128 w) {
    i128 mp;
    if (!d->dist) return NULL;   /* uniform Predictor(V) */
    const int64_t *raw = table_at(d->dist, d->stride, d->ntab, d->V, d->nout, d->minp, &mp);
    return fudged_dist(raw, d->V, mp, w, d->scratch, d->wrap64);
}
/* emit_symbol :278-289 */
static int afb_emit_symbol(afb *d, int64_t s) {
    i128 w = d->h - d->l + 1, r0, r1;
    const int64_t *tbl = afb_table(d, w);
    int rc = symbol_to_range(tbl, d->V, s, w, &r0, &r1);
    if (rc) return rc;
    if (region_overlap(d->l + r0, d->l + r1 - 1, d->lb, d->hb) == 0) return ORC_E_RANGE;
    d->h = d->l + r1 - 1;
    d->l += r0;
    if (d->nout >= d->cap) return ORC_E_CAP;
    d->out[d->nout++] = (int32_t)s;       /* predictor.accept(s) advances the table index */
    return ORC_OK;
}
/* decide_symbol :272-277; returns 1 if a symbol was emitted, 0 if undecided, <0 error */
static int afb_decide_symbol(afb *d) {
    i128 w = d->h - d->l + 1;
    const int64_t *tbl = afb_table(d, w);
    int64_t ls = val_to_symbol(tbl, d->V, d->lb - d->l, w);
    int64_t hs = val_to_symbol(tbl, d->V, d->hb - d->l, w);
    if (ls != hs) return 0;
    int rc = afb_emit_symbol(d, ls);
    return rc ? rc : 1;
}
/* emit_bit :290-298 */
static int afb_emit_bit(afb *d) {
    i128 b = fdiv(d->l, d->decision);
    if (d->h - d->l < d->decision) {
        d->l = d->l * 2 - b * d->denom;
        d->h = d->h * 2 + 1 - b * d->denom;
        d->lb = d->lb * 2 - b * d->denom;
        d->hb = d->hb * 2 + 1 - b * d->denom;
        return 1;
    }
    return 0;
}
/* flush :307-331 */
static int afb_flush(afb *d) {
    while (!(d->lb <= d->l && d->h <= d->hb)) {
        i128 w = d->h - d->l + 1;
        const int64_t *tbl = afb_table(d, w);
        int64_t ls = val_to_symbol(tbl, d->V, d->lb - d->l, w);
        int64_t hs = val_to_symbol(tbl, d->V, d->hb - d->l, w);
        if (ls > hs) return ORC_E_EMPTY;
        int64_t best = 0; double bestk = 0; int have = 0;   /* the uniform Predictor can probe negative symbols */
        for (int64_t s = ls; s <= hs; s++) {
            i128 r0, r1;
            int rc = symbol_to_range(tbl, d->V, s, w, &r0, &r1);
            if (rc) return rc;
            if (r1 == r0) return ORC_E_ZERODIV;
            double k = (double)region_overlap(d->lb - d->l, d->hb - d->l, r0, r1 - 1) /
                       (double)(r1 - r0);
            if (!have || k > bestk) { best = s; bestk = k; have = 1; }
        }
        int rc = afb_emit_symbol(d, best);
        if (rc) return rc;
    }
    d->l = 0; d->h = d->denom - 1; d->lb = 0; d->hb = d->denom - 1;
    return ORC_OK;
}

/*
 * == list(A_from_bin(...).run(bits, stop))  (arith_code.py:322-326).
 * max_syms > 0 stops (ORC_OK) once that many symbols are out: the reference has no
 * length framing, its decoder keeps emitting while the bit window allows.
 */
int orc_ac_decode(int prec, const int64_t *dist, int64_t stride, int64_t ntab, const int64_t *minp,
                  int V, const uint8_t *bits, int64_t nbits, int stop, int64_t max_syms,
                  int32_t *out, int64_t cap, int64_t *nout, int wrap64) {
    if (prec < 2 || prec > 62 || V < 1) return ORC_E_ARG;
    afb d;
    d.prec = prec; d.V = V;
    d.denom = (i128)1 << prec; d.decision = (i128)1 << (prec - 1);
    d.l = 0; d.h = d.denom - 1; d.lb = 0; d.hb = d.denom - 1;       /* :237-242 */
    d.dist = dist; d.stride = stride; d.ntab = ntab; d.minp = minp;
    d.scratch = (int64_t *)malloc(sizeof(int64_t) * (size_t)V);
    d.out = out; d.nout = 0; d.cap = cap; d.wrap64 = wrap64;
    int rc = ORC_OK;
    for (int64_t i = 0; i < nbits && rc == ORC_OK; i++) {
        /* receive_bit :268-271 */
        i128 w = fdiv(d.hb - d.lb + 1, 2);
        d.lb += w * bits[i];
        d.hb = d.lb + w - 1;
        /* step :299-306 */
        int r = afb_decide_symbol(&d);
        while (r == 1) {
            while (afb_emit_bit(&d)) {}
            if (max_syms > 0 && d.nout >= max_syms) { *nout = d.nout; free(d.scratch); return ORC_OK; }
            r = afb_decide_symbol(&d);
        }
        if (r < 0) rc = r;
    }
    if (rc == ORC_OK && stop) rc = afb_flush(&d);
    free(d.scratch);
    *nout = d.nout;
    return rc;
}

/* ------------------------------------------------------------------ */
/* ACSampler / Region / CarryBuffer (arithmetic_coding.py)              */
/* ------------------------------------------------------------------ */
typedef struct { int prec; i128 one, low, high; } region;
static inline i128 rg_span(const region *r) { return r->high - r->low + 1; }            /* :151-153 */
static inline i128 rg_map(const region *r, i128 v, i128 d) { return r->low + fdiv(rg_span(r) * v, d); } /* :160-162 */
/* Region.step + emit :166-174; every emitted bit goes through CarryBuffer.add :186-190 */
static void rg_step(region *r, i128 l, i128 h, i128 d, bitsink *sk) {
    i128 nl = rg_map(r, l, d), nh = rg_map(r, h, d) - 1;
    r->low = nl; r->high = nh;
    while (rg_span(r) * 2 <= r->one) {
        i128 bit = r->low >> (r->prec - 1);
        r->low = (r->low << 1) - (bit << r->prec);
        r->high = ((r->high << 1) + 1) - (bit << r->prec);
        sink_push(sk, bit);
        if (sk->err) return;
    }
}

/*
 * Compress path of ACSampler.sample_scaled_cdf (arithmetic_coding.py:73-95) driven
 * over n tokens, then flush_compress (:52-58).  cdf: inclusive cumulative tables
 * (uint64 in the reference: cumsum(...).astype(np.uint64)), denom = cdf[-1].
 * bits == everything the reference hands to compress_output.
 */
int orc_acs_encode(int prec, const uint64_t *cdf, int64_t stride, int64_t ntab, int V,
                   const int32_t *toks, int64_t n, int flush, uint8_t *bits, int64_t cap,
                   int64_t *nbits) {
    if (prec < 2 || prec > 62 || V < 1) return ORC_E_ARG;
    region rg = {prec, (i128)1 << prec, 0, ((i128)1 << prec) - 1};
    bitsink sk = {bits, 0, cap, 0};
    for (int64_t t = 0; t < n && !sk.err; t++) {
        const uint64_t *c = stride ? cdf + (t < ntab ? t : ntab - 1) * stride : cdf;
        int32_t tok = toks[t];
        if (tok < 0 || tok >= V) { *nbits = sk.n; return ORC_E_SYMBOL; }
        i128 low = tok ? (i128)c[tok - 1] : 0, high = (i128)c[tok], den = (i128)c[V - 1];
        rg_step(&rg, low, high, den, &sk);
    }
    if (flush && !sk.err) rg_step(&rg, 1, 2, 3, &sk);   /* :53 ; accumulator.flush adds nothing new */
    *nbits = sk.n;
    return sk.err;
}

/*
 * Expand path of ACSampler.sample_scaled_cdf (arithmetic_coding.py:96-124), LITERALLY,
 * with exact integers (the reference multiplies a Python int by np.uint64, which
 * overflows silently under numpy 2; goldens are made with object-dtype cdfs).  Includes
 * the reference's bisect_left / d=one quirks (:96), so it does NOT always round-trip.
 * Bits past the end read as 0 (:103-106).
 */
static int64_t acs_lookup(const region *r, const uint64_t *c, int V, i128 p) {
    int64_t lo = 0, hi = V;                 /* bisect_left(cdf, p, key=region.map) */
    while (lo < hi) {
        int64_t mid = (lo + hi) / 2;
        if (rg_map(r, (i128)c[mid], r->one) < p) lo = mid + 1; else hi = mid;
    }
    return lo;
}
int orc_acs_decode(int prec, const uint64_t *cdf, int64_t stride, int64_t ntab, int V,
                   const uint8_t *bits, int64_t nbits, int64_t n, int32_t *out) {
    if (prec < 2 || prec > 62 || V < 1) return ORC_E_ARG;
    region rg = {prec, (i128)1 << prec, 0, ((i128)1 << prec) - 1};
    i128 d_bits = 0, ulp = rg.one;
    int64_t pos = 0;
    bitsink nul = {NULL, 0, 0, 0};
    for (int64_t t = 0; t < n; t++) {
        const uint64_t *c = stride ? cdf + (t < ntab ? t : ntab - 1) * stride : cdf;
        while (acs_lookup(&rg, c, V, d_bits) != acs_lookup(&rg, c, V, d_bits + ulp - 1)) {
            int bit = pos < nbits ? bits[pos] : 0;
            pos++;
            ulp >>= 1;
            d_bits += bit * ulp;
        }
        int64_t tok = acs_lookup(&rg, c, V, d_bits);
        if (tok >= V) return ORC_E_INDEX;
        i128 low = tok ? (i128)c[tok - 1] : 0, high = (i128)c[tok], den = (i128)c[V - 1];
        /* region.step bits drive the d_bits window :118-122 */
        i128 nl = rg_map(&rg, low, den), nh = rg_map(&rg, high, den) - 1;
        rg.low = nl; rg.high = nh;
        while (rg_span(&rg) * 2 <= rg.one) {
            i128 bit = rg.low >> (rg.prec - 1);
            rg.low = (rg.low << 1) - (bit << rg.prec);
            rg.high = ((rg.high << 1) + 1) - (bit << rg.prec);
            ulp += ulp + (ulp == 0);
            d_bits = (d_bits << 1) - rg.one * bit;
        }
        out[t] = (int32_t)tok;
    }
    (void)nul;
    return ORC_OK;
}

/* ================================================================== */
/* Part 2: this repo's LQ32 quantisation + value-based decoder          */
/* ================================================================== */
#define LQ_LOG2E 0x3FB8AA3Bu
#define LQ_MAGIC 0x4B400000u /* 1.5 * 2^23 */
/* minimax 2^f on [-0.5, 0.5], degree 3, scaled by 2^24: c1..c3 (max rel. error 1.02e-4); the constant
 * term is folded into LQ_MAGICZ = 1.5 * 2^25, so z lands in [2^25, 2^26) where one ulp is 4 */
#define LQ_MAGICZ 0x4C400000u
static const uint32_t LQ_C[4] = {0x4b800000u, 0x4b317afdu, 0x4a780626u, 0x4961510cu};
static inline float u2f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
static inline uint32_t f2u(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }

/* LQ32 (DESIGN.md section 3), block form: the row is cut into NW = 32 * parts(V) segments of at most 1024
 * elements, every segment is quantised against ITS OWN reference exponent, and the segment totals are aligned to
 * the row-wide reference afterwards (block floating point).  Nothing needs the row maximum before the element
 * pass.  No subtraction of a maximum, no float->int conversion: integers are read out of float mantissas.
 *
 *   parts = ceil(V / 32768),  NW = 32 * parts,  G = ceil(V / 4)
 *   segment w = elements [4 * floor(w * G / NW), min(V, 4 * floor((w + 1) * G / NW)))       (a function of V only)
 * per segment w:
 *   m_w   = max x_i  (NaN dropped; -inf when nothing is left)
 *   n_w   = bits(fma(m_w, log2e, MAGIC))   MAGIC = 1.5 * 2^23; t = fma(x, log2e, MAGIC) is monotone in x, so this is
 *                                   max bits(t_i); for |x*log2e| < 2^22 the low mantissa bits of t hold rne(x*log2e).
 *   r_w   = 0 (EMPTY)            if n_w <  LQ_REF_LO    (nothing finite, or m_w * log2e <= -(2^22 - 64))
 *           0xFFFFFF (POISON)    if n_w >= LQ_REF_HI    (+inf, or m_w * log2e >= 2^22)
 *           n_w - LQ_REF_LO + 1  otherwise              (24-bit reference code)
 *   t_i   = fma(x_i, log2e, MAGIC),  sh_i = n_w - bits(t_i)   (unsigned; >= 32 for -inf; NaN -> q = 0)
 *   f_i   = fma(x_i, log2e, MAGIC - t_i)     residual in [-0.5, 0.5], single rounding
 *   z_i   = fma(fma(fma(c3, f, c2), f, c1), f, MAGICZ)   = 1.5*2^25 + 2^24 (2^f - 1); mantissa = rne(2^22 2^f)
 *   q_i   = sh_i >= 32 ? 0 : (bits(z_i) << 7) >> sh_i    (bits(z) << 7 = mantissa << 7 in [2^28.5, 2^29.5): the
 *                                   exponent field of [2^25, 2^26) ends in 00, so four q fit a uint32 sum)
 *   S_w   = sum q_i  (< 2^39.5; 0 for EMPTY / POISON segments),  c_i = sum of q_j over j < i inside the segment
 * per row:
 *   r     = max_w r_w ;  the row is DEGENERATE (every W_w = 0, cum_i = i: not uniform, the last symbol takes the rest) when r is 0 or POISON
 *   d_w   = r - r_w ,  W_w = (r_w == 0 || d_w >= 40) ? 0 : S_w >> d_w ,  Q = sum W_w
 *   C_i   = sum_{w' < w} W_w' + (c_i >> d_w)        (0 instead of the shifted term when W_w is forced to 0)
 *   cum_i = ((C_i * R) >> s) + i  with (R, s) from Q as below,  cum_V = 2^32
 */
#define LQ_REF_LO 0x4B000040
#define LQ_REF_HI 0x4B800000
#define LQ_POISON 0xFFFFFFu
static inline float lq_max(float a, float b) { /* PTX max.f32 / fmaxf: a NaN operand is dropped */
    if (a != a) return b;
    if (b != b) return a;
    return a > b ? a : b;
}
static inline int lq_parts(int V) { return (V + 32767) / 32768; }
static inline int lq_seg_begin(int w, int V) { /* first ELEMENT of segment w (w = NW: V rounded up to 4) */
    int64_t G = (V + 3) / 4;
    return (int)(4 * ((w * G) / (32 * lq_parts(V))));
}
static inline uint32_t lq_segcode(const float *x, int e0, int e1) {
    float m = u2f(0xFF800000u); /* -inf */
    for (int i = e0; i < e1; i++) m = lq_max(m, x[i]);
    int32_t n = (int32_t)f2u(fmaf(m, u2f(LQ_LOG2E), u2f(LQ_MAGIC)));
    if (n < LQ_REF_LO) return 0u;
    if (n >= LQ_REF_HI) return LQ_POISON;
    return (uint32_t)(n - LQ_REF_LO + 1);
}
static inline uint32_t lq_q(float x, uint32_t code) { /* q of one element against its segment's reference code */
    if (code == 0u || code == LQ_POISON || x != x) return 0u;
    uint32_t nref = code - 1u + (uint32_t)LQ_REF_LO;
    float t = fmaf(x, u2f(LQ_LOG2E), u2f(LQ_MAGIC));
    uint32_t sh = nref - f2u(t);
    if (sh >= 32) return 0u;
    float rn = u2f(LQ_MAGIC) - t;
    float f = fmaf(x, u2f(LQ_LOG2E), rn);
    float p = u2f(LQ_C[3]);
    p = fmaf(p, f, u2f(LQ_C[2]));
    p = fmaf(p, f, u2f(LQ_C[1]));
    float z = fmaf(p, f, u2f(LQ_MAGICZ));
    return (f2u(z) << 7) >> sh;
}
typedef struct { uint64_t Q; uint32_t R; int s; } lq_scale;
static inline lq_scale lq_make_scale(uint64_t Q, int V) {
    /* s = bitlen(Q) - 1 (>= 28 whenever Q != 0: the row maximum contributes q >= 2^28.5);
     * Qn = Q normalised to [2^31, 2^32);  D = Qn + 1;  R = floor((M << 31) / D) <= M * 2^s / Q,
     * so the scaled prefix sums never exceed M = 2^32 - V. */
    lq_scale k = {Q, 0, 0};
    if (Q < ((uint64_t)1 << 28)) return k; /* only the degenerate Q == 0 row */
    int b = 64 - __builtin_clzll(Q);
    k.s = b - 1;
    uint64_t M = ((uint64_t)1 << 32) - (uint64_t)V;
    uint64_t Qn = k.s >= 31 ? (Q >> (k.s - 31)) : (Q << (31 - k.s));
    k.R = (uint32_t)((M << 31) / (Qn + 1));
    return k;
}
static inline uint32_t lq_cum(uint64_t C, uint32_t i, lq_scale k) {
    return (uint32_t)(((u128)C * k.R) >> k.s) + i;
}
/* Row-level pieces: codes[w], weights W[w] (aligned to the row reference), shifts d[w] (64 = forced to zero). */
#define LQ_MAX_NW 1024
typedef struct { int nw; uint32_t code[LQ_MAX_NW]; uint64_t W[LQ_MAX_NW]; int d[LQ_MAX_NW]; uint64_t Q; } lq_row;
static void lq_row_summary(const float *x, int V, lq_row *r) {
    r->nw = 32 * lq_parts(V);
    uint32_t rmax = 0;
    for (int w = 0; w < r->nw; w++) {
        int e0 = lq_seg_begin(w, V), e1 = lq_seg_begin(w + 1, V);
        if (e1 > V) e1 = V;
        r->code[w] = e0 < e1 ? lq_segcode(x, e0, e1) : 0u;
        if (r->code[w] > rmax) rmax = r->code[w];
    }
    r->Q = 0;
    for (int w = 0; w < r->nw; w++) {
        int e0 = lq_seg_begin(w, V), e1 = lq_seg_begin(w + 1, V);
        if (e1 > V) e1 = V;
        uint64_t S = 0;
        for (int i = e0; i < e1; i++) S += lq_q(x[i], r->code[w]);
        uint32_t dw = rmax - r->code[w];
        int dead = (rmax == 0u || rmax == LQ_POISON || r->code[w] == 0u || dw >= 40u);
        r->d[w] = dead ? 64 : (int)dw;
        r->W[w] = dead ? 0 : (S >> dw);
        r->Q += r->W[w];
    }
}
/* Exclusive cumulative table, V entries (cum[0] = 0); the total 2^32 is implicit. */
int orc_lq32_cdf(const float *logits, int64_t rows, int V, int64_t row_stride, uint32_t *cum) {
    if (V < 1 || V > 32768 * (LQ_MAX_NW / 32)) return ORC_E_ARG;
    lq_row *R = (lq_row *)malloc(sizeof(lq_row));
    if (!R) return ORC_E_ARG;
    for (int64_t r = 0; r < rows; r++) {
        const float *x = logits + r * row_stride;
        lq_row_summary(x, V, R);
        lq_scale k = lq_make_scale(R->Q, V);
        uint64_t front = 0;
        for (int w = 0; w < R->nw; w++) {
            int e0 = lq_seg_begin(w, V), e1 = lq_seg_begin(w + 1, V);
            if (e1 > V) e1 = V;
            uint64_t c = 0;
            for (int i = e0; i < e1; i++) {
                uint64_t C = front + (R->d[w] >= 64 ? 0 : (c >> R->d[w]));
                cum[r * V + i] = lq_cum(C, (uint32_t)i, k);
                c += lq_q(x[i], R->code[w]);
            }
            front += R->W[w];
        }
    }
    free(R);
    return ORC_OK;
}
/* (cum[sym], cum[sym+1]) per row without materialising the table; hi of the last symbol is 2^32. */
int orc_lq32_lookup(const float *logits, int64_t rows, int V, int64_t row_stride,
                    const int32_t *syms, uint32_t *lo, uint64_t *hi) {
    if (V < 1 || V > 32768 * (LQ_MAX_NW / 32)) return ORC_E_ARG;
    lq_row *R = (lq_row *)malloc(sizeof(lq_row));
    if (!R) return ORC_E_ARG;
    int rc = ORC_OK;
    for (int64_t r = 0; r < rows; r++) {
        const float *x = logits + r * row_stride;
        int32_t s = syms[r];
        if (s < 0 || s >= V) { rc = ORC_E_SYMBOL; break; }
        lq_row_summary(x, V, R);
        lq_scale k = lq_make_scale(R->Q, V);
        uint64_t front = 0;
        int w = 0;
        while (lq_seg_begin(w + 1, V) <= s) front += R->W[w++];
        uint64_t c = 0;
        for (int i = lq_seg_begin(w, V); i < s; i++) c += lq_q(x[i], R->code[w]);
        uint64_t qs = lq_q(x[s], R->code[w]);
        int d = R->d[w];
        lo[r] = lq_cum(front + (d >= 64 ? 0 : (c >> d)), (uint32_t)s, k);
        hi[r] = (s == V - 1) ? ((uint64_t)1 << 32)
                             : (uint64_t)lq_cum(front + (d >= 64 ? 0 : ((c + qs) >> d)), (uint32_t)s + 1, k);
    }
    free(R);
    return rc;
}

/*
 * Value-based N-token decoder (the algorithm the GPU runs): keeps the code value v in
 * the encoder's own (l, h) coordinates, zero-padding past the end of the stream.  For
 * every stream produced by A_to_bin it returns the first n symbols A_from_bin returns
 * (tests/test_oracle_golden.py checks that against the reference itself).
 * Tables: int64 inclusive cumulative, fudged exactly like the encoder's.
 */
int orc_ac_decode_n(int prec, const int64_t *dist, int64_t stride, int64_t ntab, const int64_t *minp,
                    int V, const uint8_t *bits, int64_t nbits, int64_t n, int32_t *out, int wrap64) {
    if (prec < 2 || prec > 62 || V < 1) return ORC_E_ARG;
    const i128 denom = (i128)1 << prec, decision = (i128)1 << (prec - 1);
    i128 l = 0, h = denom - 1, v = 0;
    int64_t pos = 0;
    for (int i = 0; i < prec; i++) { v = (v << 1) | (pos < nbits ? bits[pos] : 0); pos++; }
    int64_t *scratch = (int64_t *)malloc(sizeof(int64_t) * (size_t)V);
    int rc = ORC_OK;
    for (int64_t t = 0; t < n; t++) {
        i128 w = h - l + 1, mp, r0, r1;
        const int64_t *tbl = NULL;
        int64_t s;
        if (dist) {
            const int64_t *raw = table_at(dist, stride, ntab, V, t, minp, &mp);
            tbl = fudged_dist(raw, V, mp, w, scratch, wrap64);
            s = val_to_symbol(tbl, V, v - l, w);
        } else {
            /* the symbol whose floor-mapped range holds v - l: largest s with floor(s w / V) <= v - l */
            s = (int64_t)fdiv((v - l + 1) * (i128)V - 1, w);
        }
        rc = symbol_to_range(tbl, V, s, w, &r0, &r1);
        if (rc) break;
        h = l + r1 - 1;
        l += r0;
        out[t] = (int32_t)s;
        while ((h - l) < decision) {
            i128 b = fdiv(l, decision);
            l = l * 2 - b * denom;
            h = h * 2 + 1 - b * denom;
            v = v * 2 - b * denom + (pos < nbits ? bits[pos] : 0);
            pos++;
        }
    }
    free(scratch);
    return rc;
}

/*
 * Range-pair coder on a fixed total 2^32 (what the GPU hot path feeds the coder): the
 * A_to_bin state machine with symbol_to_range(ld, hd, d = 2^32) and minp >= 1, i.e. the
 * unfudged branch of arith_code.py:84-85 (2^32 <= w * 1 always holds for prec >= 34).
 */
int orc_ac_encode_pairs(int prec, const uint32_t *lo, const uint64_t *hi, int64_t n, int stop,
                        uint8_t *bits, int64_t cap, int64_t *nbits) {
    if (prec < 34 || prec > 62) return ORC_E_ARG;
    const i128 denom = (i128)1 << prec, decision = (i128)1 << (prec - 1), d = (i128)1 << 32;
    i128 l = 0, h = denom - 1;
    bitsink sk = {bits, 0, cap, 0};
    for (int64_t t = 0; t < n && !sk.err; t++) {
        i128 w = h - l + 1;
        i128 r0 = cdiv((i128)lo[t] * w, d), r1 = cdiv((i128)hi[t] * w, d);
        h = l + r1 - 1;
        l += r0;
        while ((h - l) < decision) {
            i128 b = fdiv(l, decision);
            l = l * 2 - b * denom;
            h = h * 2 + 1 - b * denom;
            sink_push(&sk, b);
            if (sk.err) break;
        }
    }
    if (!sk.err && stop) {
        while (l > 0 || h + 1 < denom) {
            i128 b = fdiv(l, decision);
            if (region_overlap(l, h, b * decision, (b + 1) * decision) <
                region_overlap(l, h, (b + 1) * decision, (b + 2) * decision))
                b += 1;
            l = l * 2 - b * denom;
            h = h * 2 + 1 - b * denom;
            sink_push(&sk, b);
            if (sk.err) break;
        }
    }
    *nbits = sk.n;
    return sk.err;
}

/* ================================================================== */
/* Part 3: bulk CPU baseline -- the reference's own per-token work      */
/* (llama_compress.py:24-30 calc_dist + arith_code.py encode / decode), */
/* C port, pthreads over streams.                                       */
/* ================================================================== */
/* calc_dist, llama_compress.py:24-30 (float32 exp / normalise, float64 cumsum). */
void orc_ref_calc_dist(const float *logits, int V, int64_t *dist) {
    float sum = 0.f;
    float *pdf = (float *)malloc(sizeof(float) * (size_t)V);
    for (int i = 0; i < V; i++) { pdf[i] = expf(logits[i]); sum += pdf[i]; }
    double acc = 0.0;
    for (int i = 0; i < V; i++) {
        float p = pdf[i] / sum;
        double f = (double)(p * 1152921504606846976.0f); /* pdf*(1<<60) in float32, then .astype(float) */
        if (f < 2.0) f = 2.0;
        acc += f;
        dist[i] = (int64_t)acc;
    }
    free(pdf);
}

/*
 * Encode then decode `streams` independent streams of `T` tokens from precomputed logits
 * [streams, T, V] with the reference algorithm end to end, `threads` pthreads taking
 * streams from a shared counter.  Returns the number of round-trip mismatches (0
 * expected); total_bits gets the coded size.
 */
typedef struct {
    const float *logits; const int32_t *syms; int64_t streams, T; int V, prec;
    int64_t next, bad, tot; pthread_mutex_t mu;
} bulk_job;

static void *bulk_worker(void *arg) {
    bulk_job *j = (bulk_job *)arg;
    int64_t T = j->T; int V = j->V;
    int64_t *dist = (int64_t *)malloc(sizeof(int64_t) * (size_t)V * (size_t)T);
    int64_t *minp = (int64_t *)malloc(sizeof(int64_t) * (size_t)T);
    int64_t cap = T * 64 + 256;
    uint8_t *bits = (uint8_t *)malloc((size_t)cap);
    int32_t *out = (int32_t *)malloc(sizeof(int32_t) * (size_t)T);
    for (;;) {
        pthread_mutex_lock(&j->mu);
        int64_t s = j->next++;
        pthread_mutex_unlock(&j->mu);
        if (s >= j->streams) break;
        for (int64_t t = 0; t < T; t++) {
            orc_ref_calc_dist(j->logits + (s * T + t) * V, V, dist + t * V);
            minp[t] = orc_llama_minp(dist + t * V, V);
        }
        int64_t nb = 0, bad = 0;
        int rc = orc_ac_encode(j->prec, dist, V, T, minp, V, j->syms + s * T, T, 1, bits, cap, &nb, NULL, 1);
        if (rc == ORC_OK) rc = orc_ac_decode_n(j->prec, dist, V, T, minp, V, bits, nb, T, out, 1);
        if (rc != ORC_OK) bad = T;
        else for (int64_t t = 0; t < T; t++) bad += (out[t] != j->syms[s * T + t]);
        pthread_mutex_lock(&j->mu);
        j->bad += bad; j->tot += nb;
        pthread_mutex_unlock(&j->mu);
    }
    free(dist); free(minp); free(bits); free(out);
    return NULL;
}

int orc_num_threads(void) {
    long n = sysconf(_SC_NPROCESSORS_ONLN);
    return n < 1 ? 1 : (int)n;
}

int64_t orc_ref_roundtrip_bulk(const float *logits, const int32_t *syms, int64_t streams, int64_t T,
                               int V, int prec, int threads, int64_t *total_bits) {
    bulk_job j = {logits, syms, streams, T, V, prec, 0, 0, 0, PTHREAD_MUTEX_INITIALIZER};
    if (threads < 1) threads = orc_num_threads();
    if (threads > streams) threads = (int)streams;
    if (threads < 1) threads = 1;
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * (size_t)threads);
    for (int i = 0; i < threads; i++) pthread_create(&th[i], NULL, bulk_worker, &j);
    for (int i = 0; i < threads; i++) pthread_join(th[i], NULL);
    free(th);
    *total_bits = j.tot;
    return j.bad;
}
