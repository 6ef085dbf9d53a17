"""Host-side mirror of the reference's arith_code.py interface (same class and method names, same argument
meaning), with the coding done by the CUDA library through the C ABI.

What maps to what (pramasoul/lac arith_code.py):
    Predictor / CDFPredictor / ProbPredictor   :64-135   table providers: .dist, .minp, .accept(), .copy()
    CountPredictor                             (new)     ProbPredictor with prob(s) = counts[s], coded adaptively on
                                                         the device
    AC(predictor, prec).to_bin / .from_bin     :144-155
    A_to_bin                                   :156-246  incremental (__call__, step, flush, info, certain, ...) and
                                                         whole-sequence (run, encode, bits, compress) coding
    A_from_bin                                 :248-334  incremental (__call__, step, receive_bit, ...) and counted
                                                         whole-stream decoding (decompress)
    group_bits / ungroup_bits                  :336-351  byte layout of every stream
    measure_compress                           :401-420

Where the work happens.  The coder state (l, h) lives in a lac_enc_state / lac_dec_state ON THE DEVICE; every
symbol is narrowed and renormalised by a kernel (lac_ac_encode_tables / _uniform / _logits_f32 and the decode
counterparts), also in the one-symbol-at-a-time API.  The host only reads the state back and formats what the
kernels produced into the reference's return values:

  * A_to_bin.step: the k renormalisation bits of a token come out of the kernel as one integer E appended to the
    stream (carries resolved in the stream bytes).  E is recovered from the tail of the stream bytes, and the
    reference's raw digits are E's first digit floor(E / 2^(k-1)) -- which is 2 or 3 exactly when the reference
    yields a 2 or 3 ("expecting to later maybe output a 2", arith_code.py:26-28) -- followed by the k - 1 low bits.
  * A_from_bin: (lb, hb), the window of code values the bits received so far allow (receive_bit, :264-267), is
    the state of the bit READER and is kept on the host; decide_symbol (:268-273) asks the device decoder for the
    symbol at both ends of the window -- two device states that share (l, h) and carry lb resp. hb as their code
    value -- and a symbol is emitted when both agree; the kernel then does emit_symbol + the emit_bit loop
    (:274-291) for (l, h, lb, hb) at once.

Differences that cannot be avoided, both documented in DESIGN.md:
  * A_from_bin.flush() (:300-317) guesses "the shortest A string fully within [lb, hb]" symbol by symbol; that
    heuristic is not reproduced.  Every symbol the encoder coded is already determined once all bits have been
    received (the final window lies inside every coded symbol's range), so run(bits) yields all coded symbols;
    the reference's flush() then appends guessed extra symbols (51 for 50 coded in the first golden case), the
    mirror's flush() appends nothing.  decompress(data, count) decodes a known number of symbols in one call.
  * A_to_bin.flush() is one kernel call; its digits are returned in the same first-digit + bits form as a
    step's, which is the reference's digit string after carry / borrow resolution within the flush (encode(),
    bits() and the packed bytes are identical; a consumer of the raw unresolved digits of flush() may see e.g.
    (1, 0) where the reference yields (0, 2)).
There is no CPU coding path in this module: without the CUDA library every coding call raises.
"""
from __future__ import annotations

import itertools
import math
from typing import Iterable, Iterator, List, Optional, Sequence

import numpy as np


# ------------------------------------------------------------------ predictors (table providers)
class Predictor:
    """Uniform predictor over n symbols (arith_code.py:64-74): symbol s maps to
    [floor(s w / n), floor((s + 1) w / n)).  Coded by the dedicated uniform kernels, bit-exact with the reference
    (tests/golden/ac_uniform.npz)."""

    def __init__(self, n: int):
        self.n = n

    def accept(self, symbol):
        pass

    def copy(self):
        return self


class CDFPredictor(Predictor):
    """Fixed inclusive cumulative table (arith_code.py:76-110)."""

    def __init__(self, dist):
        self._dist = dist
        self._minp = min(filter(lambda v: v > 0, self.pdf_iter))

    @property
    def dist(self):
        return self._dist

    @property
    def minp(self):
        return self._minp

    @property
    def pdf_iter(self):
        d = self.dist
        return itertools.chain([d[0]], (d[i + 1] - d[i] for i in range(len(d) - 1)))


class ProbPredictor(CDFPredictor):
    """Adaptive model defined by prob(symbol) (arith_code.py:111-135)."""

    def __init__(self, n: int):
        self.n = n
        self.dcache: Optional[list] = None

    def prob(self, symbol):
        return 1

    def calc_dist(self):
        p = 0
        self.dcache = []
        for s in range(self.n):
            p += self.prob(s)
            self.dcache.append(p)
        return self.dcache

    @property
    def dist(self):
        if self.dcache is None:
            return self.calc_dist()
        return self.dcache

    @property
    def minp(self):
        return min(filter(lambda v: v > 0, self.pdf_iter))

    def accept(self, symbol):
        self.dcache = None

    def copy(self):
        return self


class CountPredictor(ProbPredictor):
    """The adaptive frequency model: prob(s) = counts[s] (ones by default), and accept(s) adds `inc` to counts[s].
    CountPredictor(256) is the byte model of the goldens ac_adaptive.npz and acs_64k.npz.  A_to_bin.compress /
    encode / bits and A_from_bin.decompress code a whole sequence in one adaptive kernel call (lac_ac_encode_adaptive
    / lac_ac_decode_adaptive, counts on the device) when the counts fit the device bounds: n <= 4096, counts >= 0,
    inc >= 0 and a total that stays below 2^62; otherwise they take the table path.  Afterwards `counts` are those
    the predictor holds after accepting every coded symbol."""

    def __init__(self, n: int, counts=None, inc: int = 1):
        super().__init__(n)
        self.counts = [1] * n if counts is None else [int(c) for c in counts]
        if len(self.counts) != n:
            raise ValueError(f"{len(self.counts)} counts for {n} symbols")
        self.inc = int(inc)

    def prob(self, symbol):
        return self.counts[symbol]

    def accept(self, symbol):
        self.counts[symbol] += self.inc
        self.dcache = None


def _counts_fit(predictor, T: int, wrap64: bool) -> bool:
    """Whether T symbols of a CountPredictor stay inside the adaptive kernels' bounds (else: the table path)."""
    from ._ffi import LAC_ADAPTIVE_MAX_VOCAB
    c = predictor.counts
    return (not wrap64 and 1 <= predictor.n <= LAC_ADAPTIVE_MAX_VOCAB and predictor.inc >= 0 and min(c) >= 0
            and sum(c) + predictor.inc * T < 1 << 62)


def _device_counts(predictor):
    from . import coder
    return coder.Counts(1, predictor.n, init=np.asarray(predictor.counts, dtype=np.int64), inc=predictor.inc)


def _take_counts(predictor, counts):
    predictor.counts = [int(c) for c in counts.counts[0].cpu().tolist()]
    predictor.dcache = None


def materialise_tables(predictor, symbols: Sequence[int]):
    """Walk a predictor along `symbols` exactly as A_to_bin.receive_symbol does (table, then accept):
    returns (dist int64 [T, V], minp int64 [T])."""
    tabs, minps = [], []
    for s in symbols:
        tabs.append(np.asarray(predictor.dist, dtype=np.int64))
        minps.append(int(predictor.minp))
        predictor.accept(s)
    if not tabs:
        return np.zeros((0, len(predictor.dist)), dtype=np.int64), np.zeros(0, dtype=np.int64)
    return np.stack(tabs), np.asarray(minps, dtype=np.int64)


# ------------------------------------------------------------------ bit packing (arith_code.py:336-351)
def group_bits(bits: Iterable[int], b: int = 8) -> Iterator[int]:
    r = 1
    for v in bits:
        r = (r << 1) | v
        if r >> b:
            yield r ^ (1 << b)
            r >>= b
    if r > 1:
        while r >> b == 0:
            r <<= 1
        yield r ^ (1 << b)


def ungroup_bits(groups: Iterable[int], b: int = 8) -> Iterator[int]:
    for g in groups:
        for i in range(b):
            yield (g >> (b - i - 1)) & 1


def _bits_of(data: bytes, nbits: int) -> List[int]:
    a = np.unpackbits(np.frombuffer(data, dtype=np.uint8))[:nbits]
    return a.astype(int).tolist()


# ------------------------------------------------------------------ how a predictor reaches the kernels
def _kind(predictor) -> str:
    if type(predictor) is Predictor:
        return "uniform"
    if type(predictor) is CountPredictor:  # whole sequences: one adaptive call; one symbol at a time: its table
        return "counts"
    if hasattr(predictor, "logits_row"):     # llama_compress.Llama_AC: fp32 logits -> LQ32 on the device
        return "logits"
    return "tables"


class _Step:
    """One symbol through the device coder for any predictor kind (encode side: StreamEncoder of 1 stream; decode
    side: StreamDecoder of 2 streams, the two ends of the bit window)."""

    @staticmethod
    def encode(enc, predictor, symbol: int, wrap64: bool):
        import torch
        sym = torch.tensor([[int(symbol)]], dtype=torch.int32, device=enc.device)
        kind = _kind(predictor)
        if kind == "uniform":
            enc.encode_uniform(sym, predictor.n)
        elif kind == "logits":
            enc.encode_logits(predictor.logits_row().view(1, 1, -1), sym)
        else:
            dist = torch.as_tensor(np.asarray(predictor.dist, dtype=np.int64)).to(enc.device)
            minp = torch.tensor([int(predictor.minp)], dtype=torch.int64, device=enc.device)
            enc.encode_tables(dist, sym, minp, wrap64=wrap64)

    @staticmethod
    def decode(dec, predictor, wrap64: bool):
        """One symbol on both pseudo-streams; returns int32 [2] (device)."""
        import torch
        kind = _kind(predictor)
        if kind == "uniform":
            return dec.decode_uniform(predictor.n, 1, check_status=False)[:, 0]
        if kind == "logits":
            return dec.decode_logits(predictor.logits_row().view(1, 1, -1), check_status=False)[:, 0]
        dist = torch.as_tensor(np.asarray(predictor.dist, dtype=np.int64)).to(dec.device)
        minp = torch.tensor([int(predictor.minp)], dtype=torch.int64, device=dec.device)
        return dec.decode_tables(dist, minp, 1, wrap64=wrap64, check_status=False)[:, 0]


# ------------------------------------------------------------------ the coder pair
ternary = Predictor(3)  # arith_code.py:143


class AC:
    def __init__(self, predictor=ternary, prec: int = 16, wrap64: bool = False):
        self.predictor = predictor
        self.precision = prec
        self.wrap64 = wrap64  # reproduce Llama_AC's numpy-int64 overflow in fudged_dist (llama_compress.py:29)

    def __repr__(self) -> str:
        return f"AC({self.predictor!r} at {self.precision} bits)"

    @property
    def to_bin(self):
        return A_to_bin(self.predictor.copy(), self.precision, self.wrap64)

    @property
    def from_bin(self):
        return A_from_bin(self.predictor.copy(), self.precision, self.wrap64)


class A_to_bin:
    """Encoder (arith_code.py:156-246).  The interval (l, h) and the emitted-bit count live on the device; l, h and
    emitted_bits below are read-backs of that state."""

    def __init__(self, predictor=ternary, prec: int = 16, wrap64: bool = False):
        self.predictor = predictor
        self.precision = prec
        self.wrap64 = wrap64
        self.denom = 1 << prec
        self.decision = 1 << (prec - 1)
        self.l = 0
        self.h = self.denom - 1
        self.emitted_bits = 0
        self._enc = None
        self._cap = 1 << 12

    # ---- device state
    def _encoder(self):
        if self._enc is None:
            from . import coder
            self._enc = coder.StreamEncoder(1, prec=self.precision, capacity_bytes=self._cap)
        return self._enc

    def _grow(self):
        """Double the stream buffer (the incremental API has no length limit); state and bytes carry over."""
        import torch
        from . import coder
        old = self._enc
        self._cap *= 2
        new = coder.StreamEncoder(1, prec=self.precision, capacity_bytes=self._cap)
        new.state.copy_(old.state)
        new.out[:, : old.cap].copy_(old.out)
        self._enc = new

    def _sync(self):
        """Read (l, h, emitted_bits, status) back; raises on a coder error (unknown symbol: arith_code.py:100-101)."""
        from ._ffi import LacError, LAC_E_ARG, LAC_ST_SYMBOL, LAC_ST_TABLE
        st = self._enc.state.cpu().numpy().view(np.int64).reshape(-1)
        status = int(st[3]) & 0xFFFFFFFF
        if status & LAC_ST_SYMBOL:
            raise AssertionError("unknown symbol")
        if status & LAC_ST_TABLE:
            raise LacError(LAC_E_ARG, "unusable table (zero-width symbol)")
        self.l, self.h = int(st[0]), int(st[1])
        prev, self.emitted_bits = self.emitted_bits, int(st[2])
        return self.emitted_bits - prev

    def _appended(self, k: int, before: int) -> int:
        """The integer E the last kernel call added to the stream as its k new bits (carries / borrows into older
        bits included): N_after = N_before * 2^k + E on the bit strings, evaluated modulo 2^(k + 66) on the tail."""
        nb = self.emitted_bits
        m = k + 66
        first = max(0, nb - m) // 8
        tail = bytes(self._enc.out[0, first:(nb + 7) // 8].cpu().numpy())
        n_after = (int.from_bytes(tail, "big") >> ((8 - nb % 8) % 8)) if tail else 0
        mod = 1 << m
        e = (n_after - (before << k)) % mod
        return e - mod if e >= mod >> 1 else e

    def _tail_value(self) -> int:
        """Value of (up to) the last 66 emitted bits: what a later _appended() needs of N_before."""
        nb = self.emitted_bits
        if nb == 0:
            return 0
        first = max(0, nb - 66) // 8
        tail = bytes(self._enc.out[0, first:(nb + 7) // 8].cpu().numpy())
        return int.from_bytes(tail, "big") >> ((8 - nb % 8) % 8)

    @staticmethod
    def _digits(e: int, k: int):
        """E as the reference's digit string: first digit carries the overflow, the rest are plain bits."""
        if k == 0:
            return ()
        return (e >> (k - 1),) + tuple((e >> (k - 2 - i)) & 1 for i in range(k - 1))

    def __repr__(self):
        sl = bin(self.l + (self.denom << 1))[3:]
        sh = bin(self.h + (self.denom << 1))[3:]
        return f"A_to_bin([{sl[0]}.{sl[1:]},{sh[0]}.{sh[1:]}])"

    # ---- one symbol at a time (arith_code.py:187-206)
    def step(self, symbol):
        enc = self._encoder()
        if (self.emitted_bits + 2 * self.precision + 80) // 8 >= self._cap:
            self._grow()
            enc = self._enc
        before = self._tail_value()
        _Step.encode(enc, self.predictor, symbol, self.wrap64)
        self.predictor.accept(symbol)
        k = self._sync()
        yield from self._digits(self._appended(k, before), k)

    def flush(self):
        """Emit the shortest bit string that is fully within [l, h] (arith_code.py:193-202); resets the interval."""
        enc = self._encoder()
        before = self._tail_value()
        enc.finished = False
        enc.finish()
        k = self._sync()
        yield from self._digits(self._appended(k, before), k)

    def __call__(self, symbol):
        if symbol is None:
            return tuple(self.flush())
        return tuple(self.step(symbol))

    def run(self, symbols, stop=1):
        for s in symbols:
            yield from self.step(s)
        if stop:
            yield from self.flush()

    def encode(self, symbols, stop=1):
        """(r, length) with r the carry-resolved integer of the digits (arith_code.py:212-219)."""
        if hasattr(symbols, "__len__") and self._fresh():
            data, n = self._bulk(symbols, stop)          # a whole sequence from a fresh coder: one GPU call
            return (int.from_bytes(data, "big") >> (8 * len(data) - n)) if n else 0, n
        r = length = 0
        for v in self.run(symbols, stop):
            r = (r << 1) + v
            length += 1
        return r, length

    def _fresh(self) -> bool:
        return self._enc is None and self.emitted_bits == 0 and self.l == 0 and self.h == self.denom - 1

    @property
    def info(self):
        return -math.log2((self.h - self.l + 1) / self.denom)

    @property
    def total_encoded_entropy(self):
        return self.emitted_bits + self.info

    @property
    def certain(self):
        return 0 <= self.l and self.h < self.denom

    def bits(self, symbols, stop=1):
        """Carry-resolved bits, yielded as soon as no later carry can change them (arith_code.py:230-246).  The
        check is made after every token (the reference makes it after every digit), so the bits are the same and
        arrive in the same order, at most one token later."""
        if hasattr(symbols, "__len__") and self._fresh():
            data, n = self._bulk(symbols, stop)          # a whole sequence from a fresh coder: one GPU call
            yield from _bits_of(data, n)
            return
        pending, plen = 0, 0
        it = iter(symbols)
        done = False
        while not done:
            try:
                digits = self(next(it))
            except StopIteration:
                done = True
                digits = tuple(self.flush()) if stop else ()
            for v in digits:
                pending = (pending << 1) + v
                plen += 1
            if self.certain or done:
                while plen:
                    plen -= 1
                    yield (pending >> plen) & 1
                pending = 0

    # ---- whole sequences in one GPU call
    def _bulk(self, symbols, stop):
        import torch
        from . import coder
        symbols = [int(s) for s in symbols]
        T = len(symbols)
        enc = coder.StreamEncoder(1, prec=self.precision, capacity_bytes=T * 8 + 64)
        kind = _kind(self.predictor)
        if T == 0:
            if stop:
                enc.finish()
        elif kind == "uniform":
            enc.encode_uniform(torch.tensor([symbols], dtype=torch.int32, device="cuda"), self.predictor.n,
                               finish=bool(stop))
        elif kind == "logits":
            rows = []
            for s in symbols:
                rows.append(self.predictor.logits_row().clone())
                self.predictor.accept(s)
            enc.encode_logits(torch.stack(rows).unsqueeze(0), torch.tensor([symbols], dtype=torch.int32, device="cuda"),
                              finish=bool(stop))
        elif kind == "counts" and _counts_fit(self.predictor, T, self.wrap64):
            counts = _device_counts(self.predictor)
            enc.encode_adaptive(torch.tensor([symbols], dtype=torch.int32, device="cuda"), counts, finish=bool(stop))
            _take_counts(self.predictor, counts)
        else:
            dist, minp = materialise_tables(self.predictor, symbols)
            enc.encode_tables(torch.from_numpy(dist).cuda(), torch.tensor([symbols], dtype=torch.int32, device="cuda"),
                              torch.from_numpy(minp).cuda(), finish=bool(stop), wrap64=self.wrap64)
        streams, nbits = enc.bitstreams()
        st = enc.state.cpu().numpy().view(np.int64).reshape(-1)
        self.l, self.h, self.emitted_bits = int(st[0]), int(st[1]), int(nbits[0])
        return streams[0], int(nbits[0])

    def compress(self, symbols, stop=1) -> bytes:
        """bytes(group_bits(self.bits(symbols, stop))) without the Python bit loop (fresh coder only)."""
        return self._bulk(symbols, stop)[0]


class A_from_bin:
    """Decoder (arith_code.py:248-334).  (l, h) live on the device, in two decoder states that carry the two ends
    lb / hb of the bit window as their code values; lb, hb (the bit reader's state) are kept here."""

    def __init__(self, predictor=ternary, prec: int = 16, wrap64: bool = False):
        self.predictor = predictor
        self.precision = prec
        self.wrap64 = wrap64
        self.denom = 1 << prec
        self.decision = 1 << (prec - 1)
        self.l = 0
        self.h = self.denom - 1
        self.lb = 0
        self.hb = self.denom - 1
        self._dec = None

    def __repr__(self):
        sl = bin(self.l + (self.denom << 1))[3:]
        sh = bin(self.h + (self.denom << 1))[3:]
        return f"A_from_bin([{sl[0]}.{sl[1:]},{sh[0]}.{sh[1:]}],[{self.lb},{self.hb}])"

    # ---- the bit reader (host): arith_code.py:264-267
    def receive_bit(self, bit):
        w = (self.hb - self.lb + 1) // 2
        self.lb += w * bit
        self.hb = self.lb + w - 1

    # ---- the coder (device)
    def _decoder(self):
        if self._dec is None:
            from . import coder
            # pseudo-stream 0 continues with zeros (the low end of the window), pseudo-stream 1 with ones
            self._dec = coder.StreamDecoder([b"\x00" * 32, b"\xff" * 32], prec=self.precision)
        return self._dec

    def _push(self):
        """Device states := (l, h, value = lb | hb), reading position rewound onto the constant padding."""
        import torch
        st = np.zeros((2, 5), dtype=np.int64)
        st[:, 0], st[:, 1] = self.l, self.h
        st[0, 2], st[1, 2] = self.lb, self.hb
        st[:, 3] = self.precision
        self._dec.state.copy_(torch.from_numpy(st.view(np.uint8).reshape(2, -1)))

    def decide_symbol(self):
        """The next symbol if both ends of the bit window decode to it (arith_code.py:268-273); the kernel then
        has already done emit_symbol and the emit_bit loop (:274-291) on (l, h, lb, hb).  None otherwise."""
        dec = self._decoder()
        self._push()
        syms = _Step.decode(dec, self.predictor, self.wrap64).cpu().numpy()
        if int(syms[0]) != int(syms[1]):
            return None
        st = dec.state.cpu().numpy().view(np.int64).reshape(2, 5)
        if (int(st[0, 4]) | int(st[1, 4])) & 0xFFFFFFFF & 4:
            raise AssertionError("predictor range does not correspond to val", self, int(syms[0]))
        self.l, self.h = int(st[0, 0]), int(st[0, 1])
        self.lb, self.hb = int(st[0, 2]), int(st[1, 2])
        s = int(syms[0])
        self.predictor.accept(s)
        return s

    def step(self, bit):
        self.receive_bit(bit)
        r = self.decide_symbol()
        while r is not None:
            yield r
            r = self.decide_symbol()

    def flush(self):
        """The reference guesses further symbols here (arith_code.py:300-317); not reproduced (module docstring):
        nothing is yielded, the state is reset like the reference's."""
        self.l, self.h, self.lb, self.hb = 0, self.denom - 1, 0, self.denom - 1
        return
        yield  # pragma: no cover  (makes this a generator, like the reference's)

    def __call__(self, bit):
        if bit is None:
            return tuple(self.flush())
        return tuple(self.step(bit))

    def run(self, bits, stop=1, count: Optional[int] = None):
        """Symbols determined by the bits, as they become determined.  count=: decode exactly that many symbols
        from the whole bit string in one GPU call (zero-padded past its end)."""
        if count is not None:
            yield from self.decompress(bytes(group_bits(bits)), count)
            return
        for b in bits:
            yield from self.step(b)
        if stop:
            yield from self.flush()

    def decode(self, bits: int, length: int, stop=1, count: Optional[int] = None):
        def biter():
            n = length
            while n:
                n -= 1
                yield (bits >> n) & 1
        yield from self.run(biter(), stop, count)

    # ---- whole streams in one GPU call
    def decompress(self, data: bytes, count: int) -> List[int]:
        import torch
        from . import coder
        dec = coder.StreamDecoder([bytes(data)], prec=self.precision)
        kind = _kind(self.predictor)
        if kind == "uniform":
            return dec.decode_uniform(self.predictor.n, count).cpu().numpy()[0].astype(int).tolist()
        if kind == "counts" and _counts_fit(self.predictor, count, self.wrap64):
            counts = _device_counts(self.predictor)
            syms = dec.decode_adaptive(counts, count).cpu().numpy()[0].astype(int).tolist()
            _take_counts(self.predictor, counts)
            return syms
        out: List[int] = []
        static = kind == "tables" and (not hasattr(self.predictor, "dcache")
                                       or type(self.predictor).accept is Predictor.accept)
        if static:  # fixed table: one GPU call for all symbols
            dist = torch.as_tensor(np.asarray(self.predictor.dist, dtype=np.int64)).cuda()
            minp = torch.tensor([int(self.predictor.minp)], dtype=torch.int64, device="cuda")
            return dec.decode_tables(dist, minp, count, wrap64=self.wrap64).cpu().numpy()[0].astype(int).tolist()
        for _ in range(count):  # adaptive model: the next table depends on the symbol just decoded
            if kind == "logits":
                s = int(dec.decode_logits(self.predictor.logits_row().view(1, 1, -1)).cpu().numpy()[0, 0])
            else:
                dist = torch.as_tensor(np.asarray(self.predictor.dist, dtype=np.int64)).cuda()
                minp = torch.tensor([int(self.predictor.minp)], dtype=torch.int64, device="cuda")
                s = int(dec.decode_tables(dist, minp, 1, wrap64=self.wrap64).cpu().numpy()[0, 0])
            self.predictor.accept(s)
            out.append(s)
        return out


# ------------------------------------------------------------------ measure_compress (arith_code.py:401-420)
def measure_compress(comp, inp, print_every_out=100, print_every_inp=100, save_bits=None, inp_cb=lambda t: "",
                     out=None):
    """bytes(group_bits(comp.bits(inp))) with the reference's progress line (tokens -> bits, bits/token) written
    to `out` (default sys.stdout; pass a no-op writer to silence it)."""
    import sys
    write = (out or sys.stdout).write
    stats = [0, 0, 0]
    if save_bits is None:
        save_bits = []

    def report():
        info = comp.total_encoded_entropy
        write(f"{stats[0]} -> {info}     {info / max(stats[0], 1)}  bits/tok  {inp_cb(stats[2])}        \r")

    def ini():
        for v in inp:
            yield v
            stats[2] = v
            stats[0] += 1
            if stats[1] % print_every_inp == 0:
                report()

    def outi(it):
        for b in it:
            save_bits.append(b)
            yield b
            stats[1] += 1
            if stats[1] % print_every_out == 0:
                report()

    return bytes(group_bits(outi(comp.bits(ini()))))
