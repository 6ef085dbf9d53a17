"""Exact restatement of the reference's integer coding path in plain Python ints.

TEST INFRASTRUCTURE ONLY, like lac_oracle.c: tests/ import it, nothing under lac_b200/ does.  It is written from
the reference lines that lac_oracle.c cites (arith_code.py, arithmetic_coding.py, llama_compress.py), not from the C,
so the two are independent restatements of one specification.  Every value is a Python int (arbitrary precision);
the only place that models fixed-width arithmetic is Llama_AC's wrap64 products, ((a * b + 2^63) mod 2^64) - 2^63,
because the reference computes those in numpy int64.  tests/test_exact_reference.py pins this module to every golden
file and then compares the oracle with it where the goldens do not reach (prec 49 .. 60, totals up to 2^62,
vocabularies above 256).
"""
from __future__ import annotations

from bisect import bisect_right


def wrap64(x: int) -> int:
    """numpy int64 product semantics: the value mod 2^64, read back as signed."""
    return ((x + (1 << 63)) % (1 << 64)) - (1 << 63)


def cdf_minp(dist) -> int:
    """CDFPredictor.minp (arith_code.py:79): the smallest positive pdf entry of an inclusive cumulative table."""
    prev, pos = 0, []
    for c in dist:
        if c - prev > 0:
            pos.append(c - prev)
        prev = c
    return min(pos)


def llama_minp(dist) -> int:
    """Llama_AC.minp (llama_compress.py:43-45): min(dist[0], min(diff(dist))), zero and negative allowed."""
    return min([dist[0]] + [dist[i] - dist[i - 1] for i in range(1, len(dist))])


class CDFPredictor:
    """CDFPredictor (arith_code.py:76-110) on an inclusive cumulative table `dist`.

    wrap=True restates Llama_AC (llama_compress.py:29), whose dist and minp are numpy int64: the products
    `denom * minp` and `dist[i] * denom` of the inherited fudged_dist wrap mod 2^64."""

    def __init__(self, dist, minp: int | None = None, wrap: bool = False):
        self.dist = [int(c) for c in dist]
        self.minp = cdf_minp(self.dist) if minp is None else int(minp)
        self.wrap = wrap
        self._memo = (None, None)  # (denom, table): a decoder step asks for the same width twice

    def fudged_dist(self, denom: int):
        """arith_code.py:83-93: the table rescaled to `denom` with every entry >= 1, if the total exceeds
        denom * minp; the table itself otherwise."""
        dist, V = self.dist, len(self.dist)
        thr = wrap64(denom * self.minp) if self.wrap else denom * self.minp
        if dist[-1] <= thr:
            return dist
        if self._memo[0] == denom:
            return self._memo[1]
        out, p = [], 0
        for i in range(V):
            prod = wrap64(dist[i] * denom) if self.wrap else dist[i] * denom
            d = prod // dist[-1] - p
            d = max(1, min(denom - p - V + i + 1, d))
            p += d
            out.append(p)
        self._memo = (denom, out)
        return out

    def symbol_to_range(self, s: int, denom: int):
        """arith_code.py:98-110: ceil-mapped [r0, r1) of symbol s inside a width-denom interval."""
        if not 0 <= s < len(self.dist):
            raise ValueError("unknown symbol")
        tbl = self.fudged_dist(denom)
        ld = tbl[s - 1] if s > 0 else 0
        return -(-ld * denom // tbl[-1]), -(-tbl[s] * denom // tbl[-1])

    def val_to_symbol(self, v: int, denom: int) -> int:
        """arith_code.py:94-97: bisect_right(dist, (v * dist[-1]) // denom) on the fudged table."""
        tbl = self.fudged_dist(denom)
        return bisect_right(tbl, v * tbl[-1] // denom)


class Predictor:
    """The uniform base class Predictor(n) (arith_code.py:64-74): floor-mapped ranges."""

    def __init__(self, n: int):
        self.n = int(n)

    def symbol_to_range(self, s: int, denom: int):
        return s * denom // self.n, (s + 1) * denom // self.n

    def val_to_symbol(self, v: int, denom: int) -> int:
        return v * self.n // denom


class BitSum:
    """The bit sink of A_to_bin.encode (arith_code.py:212-219): r = (r << 1) + v over the emitted digits v, which may
    be 2 (a carry) or negative (a borrow, flush only); the carry-resolved bits are the binary digits of r."""

    def __init__(self):
        self.r, self.n = 0, 0

    def push(self, v: int):
        self.r = (self.r << 1) + v
        self.n += 1

    def bits(self):
        assert 0 <= self.r < (1 << self.n) or self.n == 0, "carry out of the first bit"
        return [(self.r >> (self.n - 1 - i)) & 1 for i in range(self.n)]


class A_to_bin:
    """A_to_bin (arith_code.py:156-246): receive_symbol, step, flush."""

    def __init__(self, prec: int):
        self.prec = prec
        self.denom, self.decision = 1 << prec, 1 << (prec - 1)
        self.l, self.h = 0, self.denom - 1
        self.out = BitSum()

    def receive_symbol(self, pred, s: int):
        """arith_code.py:169-175, then step()."""
        r0, r1 = pred.symbol_to_range(s, self.h - self.l + 1)
        if r1 <= r0:
            raise ZeroDivisionError("zero-width symbol")  # the reference would loop forever in step()
        self.h = self.l + r1 - 1
        self.l += r0
        self.step()

    def _emit(self, b: int):
        self.l = self.l * 2 - b * self.denom
        self.h = self.h * 2 + 1 - b * self.denom
        self.out.push(b)

    def step(self):
        """decide_bit / emit_bit (arith_code.py:176-192)."""
        while self.h - self.l < self.decision:
            self._emit(self.l // self.decision)

    def flush(self):
        """arith_code.py:193-202: emit digits until [l, h] covers the whole range, each time towards the half-range
        that overlaps [l, h] more."""
        dec = self.decision
        while self.l > 0 or self.h + 1 < self.denom:
            b = self.l // dec
            if _overlap(self.l, self.h, b * dec, (b + 1) * dec) < _overlap(self.l, self.h, (b + 1) * dec, (b + 2) * dec):
                b += 1
            self._emit(b)

    def state(self):
        return self.l, self.h, self.out.n


def _overlap(a, b, c, d):
    """region_overlap (arith_code.py:59-61): size of inclusive [a, b] intersected with inclusive [c, d]."""
    return max(0, min(d, b) - max(a, c) + 1)


def _pred_at(preds, t):
    return preds[t] if isinstance(preds, (list, tuple)) else preds


def ac_encode(preds, syms, prec: int, stop: bool = True):
    """Carry-resolved bits of A_to_bin(prec) over syms; preds is one predictor or one per position."""
    enc = A_to_bin(prec)
    for t, s in enumerate(syms):
        enc.receive_symbol(_pred_at(preds, t), int(s))
    if stop:
        enc.flush()
    return enc.out.bits()


def ac_decode_n(preds, bits, n: int, prec: int):
    """The first n symbols of a stream, tracking the code value v in the encoder's own (l, h) coordinates (zeros past
    the end of the bits).  The symbol is the one whose range holds v - l: val_to_symbol for CDFPredictor; for the
    uniform Predictor the largest s with floor(s w / n) <= v - l, since its val_to_symbol is not that symbol at range
    boundaries."""
    denom, dec = 1 << prec, 1 << (prec - 1)
    l, h, pos = 0, denom - 1, 0

    def nxt():
        nonlocal pos
        b = bits[pos] if pos < len(bits) else 0
        pos += 1
        return int(b)

    v = 0
    for _ in range(prec):
        v = (v << 1) | nxt()
    out = []
    for t in range(n):
        p, w = _pred_at(preds, t), h - l + 1
        s = ((v - l + 1) * p.n - 1) // w if isinstance(p, Predictor) else p.val_to_symbol(v - l, w)
        r0, r1 = p.symbol_to_range(s, w)
        h, l = l + r1 - 1, l + r0
        out.append(s)
        while h - l < dec:
            b = l // dec
            l, h = l * 2 - b * denom, h * 2 + 1 - b * denom
            v = v * 2 - b * denom + nxt()
    return out


class Region:
    """ACSampler's Region (arithmetic_coding.py:129-174): floor-mapped sub-intervals, one bit per doubling."""

    def __init__(self, prec: int):
        self.prec, self.one = prec, 1 << prec
        self.low, self.high = 0, self.one - 1
        self.out = BitSum()

    def map(self, v: int, d: int) -> int:
        return self.low + (self.high - self.low + 1) * v // d

    def step(self, l: int, h: int, d: int):
        self.low, self.high = self.map(l, d), self.map(h, d) - 1
        if self.high < self.low:
            raise ZeroDivisionError("empty region")  # the reference would never terminate
        while (self.high - self.low + 1) * 2 <= self.one:
            bit = self.low >> (self.prec - 1)
            self.low = (self.low << 1) - (bit << self.prec)
            self.high = ((self.high << 1) + 1) - (bit << self.prec)
            self.out.push(bit)


def acs_encode(cdfs, toks, prec: int, finish: int = 1):
    """Bits of ACSampler(prec)'s compress path (sample_scaled_cdf, arithmetic_coding.py:73-95) over toks; cdfs is one
    inclusive uint64 cumulative table or one per position.
    finish 1: flush_compress (arithmetic_coding.py:50-56), step(1, 2, 3);
    finish 2: the safe termination, A_to_bin.flush (arith_code.py:193-202) applied to the region."""
    rg = Region(prec)
    for t, tok in enumerate(toks):
        c = [int(x) for x in _pred_at(cdfs, t)]
        tok = int(tok)
        if not 0 <= tok < len(c):
            raise ValueError("unknown symbol")
        rg.step(c[tok - 1] if tok else 0, c[tok], c[-1])
    if finish == 1:
        rg.step(1, 2, 3)
    elif finish == 2:
        enc = A_to_bin(prec)
        enc.l, enc.h, enc.out = rg.low, rg.high, rg.out
        enc.flush()
    return rg.out.bits()
