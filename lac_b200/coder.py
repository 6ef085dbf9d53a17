"""Batched GPU coder API: torch tensors in, torch tensors / bytes out, every operation a call
into liblac_b200.so through the C ABI (lac_b200/_ffi.py).  torch is used for device memory
and streams only.

Conventions
-----------
* uint32 values (LQ32 cumulative frequencies, pairs) are carried in torch.int32 tensors
  holding the same 32 bits; `u32(t)` widens them to int64 for arithmetic on the host side.
* Bitstreams are MSB-first bytes, byte-for-byte what the reference's
  bytes(group_bits(A_to_bin.bits(...))) (arith_code.py:336-347) / packbits
  (arithmetic_coding.py:212-225) produce.
* Workspace: the logits-driven calls take an optional `Workspace` (device scratch for the row summaries); with one
  they allocate nothing, which is what a per-token loop or a CUDA graph wants.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _ffi
from ._ffi import LacError, check, lib

DEFAULT_PREC = 48  # llama_compress.py:4 r(..., prec=48)


def _cur_stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _need_cuda(t: torch.Tensor, name: str, dtype=None):
    if not t.is_cuda:
        raise LacError(_ffi.LAC_E_ARG, f"{name} must be a CUDA tensor (lac_b200 has no CPU path)")
    if dtype is not None and t.dtype != dtype:
        raise LacError(_ffi.LAC_E_ARG, f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise LacError(_ffi.LAC_E_ARG, f"{name} must be contiguous")


class Workspace:
    """Device scratch for the logits-driven calls, sized for `rows` logits rows per call (lac_workspace_bytes)."""

    def __init__(self, rows: int, vocab: int, device="cuda"):
        self.nbytes = int(lib().lac_workspace_bytes(int(rows), int(vocab)))
        self.buf = torch.empty(max(self.nbytes, 16), dtype=torch.uint8, device=device)

    @property
    def ptr(self):
        return self.buf.data_ptr()


def _ws(ws: Optional["Workspace"]):
    return (ws.ptr, ws.nbytes) if ws is not None else (None, 0)


def u32(t: torch.Tensor) -> torch.Tensor:
    """int32-carried uint32 -> int64 values."""
    return t.to(torch.int64) & 0xFFFFFFFF


# ------------------------------------------------------------------------------------ (a) CDF
def cdf_build(logits: torch.Tensor, ws: Optional[Workspace] = None) -> torch.Tensor:
    """LQ32 exclusive cumulative table per row: int32-carried uint32 [rows, V]; total 2^32 implicit.

    Replaces Llama_AC.calc_dist (llama_compress.py:24-30) / ProbPredictor.calc_dist
    (arith_code.py:117-123)."""
    _need_cuda(logits, "logits", torch.float32)
    rows, V = logits.shape
    cum = torch.empty((rows, V), dtype=torch.int32, device=logits.device)
    check(lib().lac_cdf_build_f32(logits.data_ptr(), rows, V, V, cum.data_ptr(), *_ws(ws), _cur_stream()))
    return cum


def cdf_lookup(logits: torch.Tensor, syms: torch.Tensor, status: Optional[torch.Tensor] = None,
               ws: Optional[Workspace] = None) -> torch.Tensor:
    """(cum[sym], cum[sym+1]) per row, int32-carried uint32 [rows, 2]; hi == 0 means 2^32."""
    _need_cuda(logits, "logits", torch.float32)
    _need_cuda(syms, "syms", torch.int32)
    rows, V = logits.shape
    if syms.numel() != rows:
        raise LacError(_ffi.LAC_E_ARG, "syms must have one entry per logits row")
    pairs = torch.empty((rows, 2), dtype=torch.int32, device=logits.device)
    check(lib().lac_cdf_lookup_f32(logits.data_ptr(), rows, V, V, syms.data_ptr(), pairs.data_ptr(),
                                   status.data_ptr() if status is not None else None, *_ws(ws), _cur_stream()))
    return pairs


def cdf_to_dist(cum: torch.Tensor) -> np.ndarray:
    """Exclusive uint32 table(s) -> int64 inclusive cumulative tables as CDFPredictor.dist holds them."""
    c = u32(cum).cpu().numpy()
    out = np.empty_like(c)
    out[..., :-1] = c[..., 1:]
    out[..., -1] = 1 << 32
    return out


# ------------------------------------------------------------------------------------ (b) coder
class Counts:
    """Device-resident counts of an adaptive frequency model, int64 [n_streams, vocab]: prob(s) = counts[s], and
    every coded or decoded token adds `inc` to its symbol's count (the kernels update them in place).  `init` is
    None (all ones), [vocab] (the same for every stream) or [n_streams, vocab].  An encoder and a decoder each need
    their own Counts, started from the same values."""

    def __init__(self, n_streams: int, vocab: int, init=None, inc: int = 1, device="cuda"):
        self.n, self.vocab, self.inc = int(n_streams), int(vocab), int(inc)
        if not 1 <= self.vocab <= _ffi.LAC_ADAPTIVE_MAX_VOCAB:
            raise LacError(_ffi.LAC_E_ARG, f"vocab {self.vocab} out of range [1, {_ffi.LAC_ADAPTIVE_MAX_VOCAB}]")
        if self.inc < 0:
            raise LacError(_ffi.LAC_E_ARG, f"inc must be >= 0, got {self.inc}")
        self.device = torch.device(device)
        self.counts = torch.empty((self.n, self.vocab), dtype=torch.int64, device=self.device)
        self.reset(init)

    def reset(self, init=None):
        """Start again from `init` (None: all ones) in the same device buffer."""
        if init is None:
            self.counts.fill_(1)
            return
        a = torch.as_tensor(np.asarray(init, dtype=np.int64) if not torch.is_tensor(init) else init)
        if tuple(a.shape) not in ((self.vocab,), (self.n, self.vocab)):
            raise LacError(_ffi.LAC_E_ARG, f"init must be [{self.vocab}] or [{self.n}, {self.vocab}], "
                                           f"got {list(a.shape)}")
        self.counts.copy_(a.to(device=self.device, dtype=torch.int64).expand(self.n, self.vocab))

    @property
    def ptr(self):
        return self.counts.data_ptr()


def _check_counts(counts: "Counts", n: int):
    _need_cuda(counts.counts, "counts", torch.int64)
    if tuple(counts.counts.shape) != (n, counts.vocab):
        raise LacError(_ffi.LAC_E_ARG, f"counts hold {counts.counts.shape[0]} streams, the coder {n}")


def _collect_streams(out: torch.Tensor, state: torch.Tensor) -> Tuple[List[bytes], np.ndarray]:
    st = state.cpu().numpy().view(np.uint8).reshape(-1, _ffi.ENC_STATE_BYTES)
    nbits = st[:, 16:24].copy().view(np.uint64).reshape(-1)
    status = st[:, 24:28].copy().view(np.uint32).reshape(-1)
    if (status & _ffi.LAC_ST_CAP).any():
        raise LacError(_ffi.LAC_E_CAP, f"output capacity exceeded on streams {np.nonzero(status & 1)[0][:8].tolist()}")
    if (status & _ffi.LAC_ST_SYMBOL).any():
        raise LacError(_ffi.LAC_E_SYMBOL, f"symbol out of range on streams {np.nonzero(status & 2)[0][:8].tolist()}")
    if (status & _ffi.LAC_ST_TABLE).any():
        raise LacError(_ffi.LAC_E_ARG, f"unusable table (zero-width symbol) on streams {np.nonzero(status & 4)[0][:8].tolist()}")
    host = out.cpu().numpy()
    nbytes = (nbits + 7) // 8
    return [host[i, : int(nbytes[i])].tobytes() for i in range(host.shape[0])], nbits


class StreamEncoder:
    """n_streams independent A_to_bin coders (arith_code.py:156-246) living on the GPU.

    Feed tokens in slices (state persists between calls), then finish()."""

    def __init__(self, n_streams: int, prec: int = DEFAULT_PREC, capacity_bytes: int = 1 << 16, device="cuda"):
        self.n, self.prec, self.cap = int(n_streams), int(prec), int(capacity_bytes)
        self.device = torch.device(device)
        self.state = torch.zeros((self.n, _ffi.ENC_STATE_BYTES), dtype=torch.uint8, device=self.device)
        self.out = torch.zeros((self.n, self.cap), dtype=torch.uint8, device=self.device)
        self.reset()

    def reset(self):
        """Start n_streams new streams in the same device buffers (their addresses stay valid for CUDA graphs)."""
        check(lib().lac_enc_init(self.state.data_ptr(), self.n, self.prec, _cur_stream()))
        self.finished = False

    def status(self) -> int:
        """OR of the streams' status words (one 4-byte read)."""
        flag = torch.zeros(1, dtype=torch.int32, device=self.device)
        check(lib().lac_enc_status(self.state.data_ptr(), self.n, flag.data_ptr(), _cur_stream()))
        return int(flag.item()) & 0xFFFFFFFF

    def _ntok(self, ntok):
        if ntok is None:
            return None
        _need_cuda(ntok, "ntok", torch.int32)
        return ntok.data_ptr()

    def encode_pairs(self, pairs: torch.Tensor, ntok: Optional[torch.Tensor] = None, finish: bool = False):
        """pairs: int32-carried uint32 [n_streams, T, 2] from cdf_lookup."""
        _need_cuda(pairs, "pairs", torch.int32)
        S, T, two = pairs.shape
        if S != self.n or two != 2:
            raise LacError(_ffi.LAC_E_ARG, "pairs must be [n_streams, T, 2]")
        check(lib().lac_ac_encode_pairs(pairs.data_ptr(), S, T, T, 1, self._ntok(ntok), self.state.data_ptr(),
                                        self.out.data_ptr(), self.cap, int(finish), self.prec, _cur_stream()))
        self.finished = self.finished or finish

    def encode_logits(self, logits: torch.Tensor, syms: torch.Tensor, ntok: Optional[torch.Tensor] = None,
                      finish: bool = False, ws: Optional[Workspace] = None):
        """logits [n_streams, T, V] fp32, syms [n_streams, T] int32: one pass over the logits (row summaries), then
        ONE kernel that looks up the coded symbols' ranges and runs the coder (lac_ac_encode_logits_f32)."""
        _need_cuda(logits, "logits", torch.float32)
        _need_cuda(syms, "syms", torch.int32)
        S, T, V = logits.shape
        if S != self.n or tuple(syms.shape) != (S, T):
            raise LacError(_ffi.LAC_E_ARG, "logits must be [n_streams, T, V] and syms [n_streams, T]")
        check(lib().lac_ac_encode_logits_f32(logits.data_ptr(), S, T, T * V, V, V, syms.data_ptr(), T,
                                             self._ntok(ntok), self.state.data_ptr(), self.out.data_ptr(), self.cap,
                                             int(finish), self.prec, *_ws(ws), _cur_stream()))
        self.finished = self.finished or finish

    def encode_step(self, logits: torch.Tensor, syms: torch.Tensor, live: Optional[torch.Tensor] = None,
                    ws: Optional[Workspace] = None):
        """One model-in-the-loop step: logits [n_streams, V], syms [n_streams]; live [n_streams] int32 0 / 1."""
        self.encode_logits(logits.unsqueeze(1), syms.unsqueeze(1), live, False, ws)

    def encode_tables(self, dist: torch.Tensor, syms: torch.Tensor, minp: torch.Tensor,
                      ntok: Optional[torch.Tensor] = None, finish: bool = False, wrap64: bool = False):
        """General int64 inclusive cumulative tables (CDFPredictor.dist): [V] shared, [T, V] per position,
        or [n_streams, T, V].  minp: matching [1] / [T] / [n_streams, T] int64 (predictor.minp)."""
        _need_cuda(dist, "dist", torch.int64)
        _need_cuda(minp, "minp", torch.int64)
        _need_cuda(syms, "syms", torch.int32)
        S, T = syms.shape
        V, ss, ts, mss, mts = _table_strides(dist, minp, S, T)
        check(lib().lac_ac_encode_tables(dist.data_ptr(), V, ss, ts, minp.data_ptr(), mss, mts, syms.data_ptr(), T, S, T,
                                         self._ntok(ntok), self.state.data_ptr(), self.out.data_ptr(), self.cap,
                                         int(finish), self.prec, _ffi.LAC_F_WRAP64 if wrap64 else 0, _cur_stream()))
        self.finished = self.finished or finish

    def encode_uniform(self, syms: torch.Tensor, n_symbols: int, ntok: Optional[torch.Tensor] = None,
                       finish: bool = False):
        """The reference's uniform base class Predictor(n) (arith_code.py:64-74, floor-mapped ranges)."""
        _need_cuda(syms, "syms", torch.int32)
        S, T = syms.shape
        check(lib().lac_ac_encode_uniform(syms.data_ptr(), S, T, T, self._ntok(ntok), int(n_symbols),
                                          self.state.data_ptr(), self.out.data_ptr(), self.cap, int(finish),
                                          self.prec, _cur_stream()))
        self.finished = self.finished or finish

    def acs_encode_tables(self, cdf: torch.Tensor, syms: torch.Tensor, ntok: Optional[torch.Tensor] = None,
                          finish=False):
        """ACSampler semantics (arithmetic_coding.py:73-95): int64-carried uint64 inclusive tables.
        finish=True: the reference's flush_compress (bit-exact; tail tokens may be undecodable);
        finish="safe": A_to_bin-style termination, always decodable."""
        _need_cuda(cdf, "cdf", torch.int64)
        _need_cuda(syms, "syms", torch.int32)
        S, T = syms.shape
        V, ss, ts, _, _ = _table_strides(cdf, None, S, T)
        check(lib().lac_acs_encode_tables(cdf.data_ptr(), V, ss, ts, syms.data_ptr(), T, S, T, self._ntok(ntok),
                                          self.state.data_ptr(), self.out.data_ptr(), self.cap,
                                          2 if finish == "safe" else int(bool(finish)), self.prec, _cur_stream()))
        self.finished = self.finished or bool(finish)

    def encode_adaptive(self, syms: torch.Tensor, counts: Counts, ntok: Optional[torch.Tensor] = None,
                        finish: bool = False):
        """Adaptive frequency model under A_to_bin: CDFPredictor on dist = cumsum(counts) before each token, then
        counts[sym] += counts.inc (lac_ac_encode_adaptive).  syms [n_streams, T] int32; `counts` carries over
        between calls like the coder state."""
        _need_cuda(syms, "syms", torch.int32)
        S, T = syms.shape
        _check_counts(counts, self.n)
        if S != self.n:
            raise LacError(_ffi.LAC_E_ARG, "syms must be [n_streams, T]")
        check(lib().lac_ac_encode_adaptive(counts.ptr, counts.vocab, counts.inc, syms.data_ptr(), T, S, T,
                                           self._ntok(ntok), self.state.data_ptr(), self.out.data_ptr(), self.cap,
                                           int(finish), self.prec, _cur_stream()))
        self.finished = self.finished or finish

    def acs_encode_adaptive(self, syms: torch.Tensor, counts: Counts, ntok: Optional[torch.Tensor] = None,
                            finish=False):
        """The same model under ACSampler (cdf = cumsum(counts)); finish as acs_encode_tables."""
        _need_cuda(syms, "syms", torch.int32)
        S, T = syms.shape
        _check_counts(counts, self.n)
        if S != self.n:
            raise LacError(_ffi.LAC_E_ARG, "syms must be [n_streams, T]")
        check(lib().lac_acs_encode_adaptive(counts.ptr, counts.vocab, counts.inc, syms.data_ptr(), T, S, T,
                                            self._ntok(ntok), self.state.data_ptr(), self.out.data_ptr(), self.cap,
                                            2 if finish == "safe" else int(bool(finish)), self.prec, _cur_stream()))
        self.finished = self.finished or bool(finish)

    def acs_flush(self, safe: bool = False):
        """ACSampler.flush_compress (arithmetic_coding.py:50-56) on every stream, no token coded."""
        one = torch.ones(1, dtype=torch.int64, device=self.device)
        none = torch.empty((self.n, 0), dtype=torch.int32, device=self.device)
        check(lib().lac_acs_encode_tables(one.data_ptr(), 1, 0, 0, none.data_ptr(), 0, self.n, 0, None,
                                          self.state.data_ptr(), self.out.data_ptr(), self.cap, 2 if safe else 1,
                                          self.prec, _cur_stream()))

    def finish(self):
        if not self.finished:
            empty = torch.empty((self.n, 0, 2), dtype=torch.int32, device=self.device)
            if self.prec >= 34:
                self.encode_pairs(empty, finish=True)
            else:  # pairs entry point needs prec >= 34; an empty table call flushes any precision
                dist = torch.ones(1, dtype=torch.int64, device=self.device)
                syms = torch.empty((self.n, 0), dtype=torch.int32, device=self.device)
                self.encode_tables(dist, syms, dist, finish=True)

    def nbits(self) -> np.ndarray:
        st = self.state.cpu().numpy().view(np.uint8).reshape(-1, _ffi.ENC_STATE_BYTES)
        return st[:, 16:24].copy().view(np.uint64).reshape(-1)

    def bitstreams(self) -> Tuple[List[bytes], np.ndarray]:
        """(bytes per stream, bit length per stream); raises on capacity / symbol errors."""
        return _collect_streams(self.out, self.state)


def _table_strides(tab: torch.Tensor, minp: Optional[torch.Tensor], S: int, T: int):
    if tab.dim() == 1:
        V, ss, ts, mss, mts = tab.shape[0], 0, 0, 0, 0
    elif tab.dim() == 2:
        if tab.shape[0] < T:
            raise LacError(_ffi.LAC_E_ARG, "per-position tables need at least T rows")
        V, ss, ts, mss, mts = tab.shape[1], 0, tab.shape[1], 0, 1
    elif tab.dim() == 3:
        if tab.shape[0] != S or tab.shape[1] < T:
            raise LacError(_ffi.LAC_E_ARG, "tables must be [n_streams, >=T, V]")
        V, ss, ts, mss, mts = tab.shape[2], tab.shape[1] * tab.shape[2], tab.shape[2], tab.shape[1], 1
    else:
        raise LacError(_ffi.LAC_E_ARG, "tables must be 1-, 2- or 3-dimensional")
    if minp is not None:
        need = 1 if tab.dim() == 1 else (tab.shape[0] if tab.dim() == 2 else tab.shape[0] * tab.shape[1])
        if minp.numel() != need:
            raise LacError(_ffi.LAC_E_ARG, f"minp needs {need} entries, got {minp.numel()}")
    return V, ss, ts, mss, mts


def pack_streams(streams: Sequence[bytes], device="cuda") -> Tuple[torch.Tensor, torch.Tensor]:
    """Concatenate bitstreams into one device buffer + int64 offsets [n + 1] (padded so reads stay in bounds)."""
    offs = np.zeros(len(streams) + 1, dtype=np.int64)
    for i, s in enumerate(streams):
        offs[i + 1] = offs[i] + len(s)
    buf = np.frombuffer(b"".join(streams) + b"\0" * 16, dtype=np.uint8).copy()
    return torch.from_numpy(buf).to(device), torch.from_numpy(offs).to(device)


class StreamDecoder:
    """n_streams independent A_from_bin decoders (arith_code.py:248-334) on the GPU, decoding a
    known number of tokens (the reference has no length framing; the container supplies it)."""

    def __init__(self, streams: Sequence[bytes], prec: int = DEFAULT_PREC, device="cuda",
                 capacity_bytes: Optional[int] = None):
        self.n, self.prec = len(streams), int(prec)
        self.device = torch.device(device)
        total = sum(len(s) for s in streams) + 16
        self.bytes = torch.zeros(max(total, int(capacity_bytes or 0)), dtype=torch.uint8, device=self.device)
        self.offsets = torch.zeros(self.n + 1, dtype=torch.int64, device=self.device)
        self.state = torch.zeros((self.n, _ffi.DEC_STATE_BYTES), dtype=torch.uint8, device=self.device)
        self.reset(streams)

    def reset(self, streams: Sequence[bytes]):
        """Start decoding a new set of n_streams streams in the same device buffers (addresses stay valid for CUDA
        graphs); they must fit the byte capacity given at construction."""
        if len(streams) != self.n:
            raise LacError(_ffi.LAC_E_ARG, f"expected {self.n} streams, got {len(streams)}")
        offs = np.zeros(self.n + 1, dtype=np.int64)
        np.cumsum([len(s) for s in streams], out=offs[1:])
        if int(offs[-1]) + 16 > self.bytes.numel():
            raise LacError(_ffi.LAC_E_CAP, f"{int(offs[-1])} stream bytes exceed the decoder's capacity "
                                           f"({self.bytes.numel() - 16}); construct it with capacity_bytes=")
        buf = np.frombuffer(b"".join(streams) + b"\0" * 16, dtype=np.uint8)
        self.bytes[: len(buf)].copy_(torch.from_numpy(buf.copy()))
        self.offsets.copy_(torch.from_numpy(offs))
        check(lib().lac_dec_init(self.state.data_ptr(), self.n, self.prec, self.bytes.data_ptr(),
                                 self.offsets.data_ptr(), _cur_stream()))

    def decode_logits(self, logits: torch.Tensor, ntok: Optional[torch.Tensor] = None,
                      ws: Optional[Workspace] = None, out: Optional[torch.Tensor] = None,
                      check_status: bool = True) -> torch.Tensor:
        """logits [n_streams, T, V] fp32 -> symbols int32 [n_streams, T] (row summaries, then search + update).
        logits [1, T, V] is shared by all streams (stream stride 0).
        Raises LacError(LAC_E_STREAM) for a truncated / foreign stream unless check_status=False (a per-token loop
        checks once at the end with status())."""
        _need_cuda(logits, "logits", torch.float32)
        S, T, V = logits.shape
        if S != self.n and S != 1:
            raise LacError(_ffi.LAC_E_ARG, "logits must be [n_streams, T, V] (or [1, T, V], shared)")
        stream_stride = T * V if S == self.n else 0
        S = self.n
        syms = out if out is not None else torch.zeros((S, T), dtype=torch.int32, device=self.device)
        check(lib().lac_ac_decode_logits_f32(logits.data_ptr(), S, T, stream_stride, V, V,
                                             ntok.data_ptr() if ntok is not None else None, self.state.data_ptr(),
                                             self.bytes.data_ptr(), self.offsets.data_ptr(), syms.data_ptr(),
                                             syms.stride(0), self.prec, *_ws(ws), _cur_stream()))
        if check_status:
            self._check_status()
        return syms

    def decode_step(self, logits: torch.Tensor, live: Optional[torch.Tensor] = None, ws: Optional[Workspace] = None,
                    out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """One model-in-the-loop step: logits [n_streams, V] -> symbols [n_streams] (status checked by the caller
        at the end of the loop: status())."""
        o = out.unsqueeze(1) if out is not None else None
        return self.decode_logits(logits.unsqueeze(1), live, ws, o, check_status=False).squeeze(1)

    def status(self) -> int:
        """OR of the streams' status words (one 4-byte read)."""
        flag = torch.zeros(1, dtype=torch.int32, device=self.device)
        check(lib().lac_dec_status(self.state.data_ptr(), self.n, flag.data_ptr(), _cur_stream()))
        return int(flag.item()) & 0xFFFFFFFF

    def decode_tables(self, dist: torch.Tensor, minp: torch.Tensor, T: int, ntok: Optional[torch.Tensor] = None,
                      wrap64: bool = False, check_status: bool = True) -> torch.Tensor:
        _need_cuda(dist, "dist", torch.int64)
        _need_cuda(minp, "minp", torch.int64)
        V, ss, ts, mss, mts = _table_strides(dist, minp, self.n, T)
        syms = torch.zeros((self.n, T), dtype=torch.int32, device=self.device)
        check(lib().lac_ac_decode_tables(dist.data_ptr(), V, ss, ts, minp.data_ptr(), mss, mts, self.n, T,
                                         ntok.data_ptr() if ntok is not None else None, self.state.data_ptr(),
                                         self.bytes.data_ptr(), self.offsets.data_ptr(), syms.data_ptr(), T,
                                         self.prec, _ffi.LAC_F_WRAP64 if wrap64 else 0, _cur_stream()))
        if check_status:
            self._check_status()
        return syms

    def decode_uniform(self, n_symbols: int, T: int, ntok: Optional[torch.Tensor] = None,
                       check_status: bool = True) -> torch.Tensor:
        """Decoder for encode_uniform streams: the symbol whose floor-mapped range holds the code value."""
        syms = torch.zeros((self.n, T), dtype=torch.int32, device=self.device)
        check(lib().lac_ac_decode_uniform(self.n, T, ntok.data_ptr() if ntok is not None else None, int(n_symbols),
                                          self.state.data_ptr(), self.bytes.data_ptr(), self.offsets.data_ptr(),
                                          syms.data_ptr(), T, self.prec, _cur_stream()))
        if check_status:
            self._check_status()
        return syms

    def acs_decode_tables(self, cdf: torch.Tensor, T: int, ntok: Optional[torch.Tensor] = None,
                          check_status: bool = True) -> torch.Tensor:
        _need_cuda(cdf, "cdf", torch.int64)
        V, ss, ts, _, _ = _table_strides(cdf, None, self.n, T)
        syms = torch.zeros((self.n, T), dtype=torch.int32, device=self.device)
        check(lib().lac_acs_decode_tables(cdf.data_ptr(), V, ss, ts, self.n, T,
                                          ntok.data_ptr() if ntok is not None else None, self.state.data_ptr(),
                                          self.bytes.data_ptr(), self.offsets.data_ptr(), syms.data_ptr(), T,
                                          self.prec, _cur_stream()))
        if check_status:
            self._check_status()
        return syms

    def decode_adaptive(self, counts: Counts, T: int, ntok: Optional[torch.Tensor] = None,
                        check_status: bool = True) -> torch.Tensor:
        """Decoder for encode_adaptive streams: T symbols per stream from the bits alone, `counts` (the decoder's
        own, started where the encoder's started) updated after every symbol."""
        _check_counts(counts, self.n)
        syms = torch.zeros((self.n, T), dtype=torch.int32, device=self.device)
        check(lib().lac_ac_decode_adaptive(counts.ptr, counts.vocab, counts.inc, self.n, T,
                                           ntok.data_ptr() if ntok is not None else None, self.state.data_ptr(),
                                           self.bytes.data_ptr(), self.offsets.data_ptr(), syms.data_ptr(), T,
                                           self.prec, _cur_stream()))
        if check_status:
            self._check_status()
        return syms

    def acs_decode_adaptive(self, counts: Counts, T: int, ntok: Optional[torch.Tensor] = None,
                            check_status: bool = True) -> torch.Tensor:
        """Decoder for acs_encode_adaptive streams."""
        _check_counts(counts, self.n)
        syms = torch.zeros((self.n, T), dtype=torch.int32, device=self.device)
        check(lib().lac_acs_decode_adaptive(counts.ptr, counts.vocab, counts.inc, self.n, T,
                                            ntok.data_ptr() if ntok is not None else None, self.state.data_ptr(),
                                            self.bytes.data_ptr(), self.offsets.data_ptr(), syms.data_ptr(), T,
                                            self.prec, _cur_stream()))
        if check_status:
            self._check_status()
        return syms

    def _check_status(self):
        if self.status() == 0:
            return
        st = self.state.cpu().numpy().view(np.uint8).reshape(-1, _ffi.DEC_STATE_BYTES)
        status = st[:, 32:36].copy().view(np.uint32).reshape(-1)
        if (status & _ffi.LAC_ST_TRUNC).any():
            bad = np.nonzero(status & _ffi.LAC_ST_TRUNC)[0][:8].tolist()
            raise LacError(_ffi.LAC_E_STREAM, f"truncated or foreign bitstream on streams {bad} "
                                              "(more bits consumed than the stream holds)")
        raise LacError(_ffi.LAC_E_ARG, f"unusable table on streams {np.nonzero(status)[0][:8].tolist()}")


# ------------------------------------------------------------------------------------ host-buffer calls
def encode_logits_host(logits: np.ndarray, syms: np.ndarray, prec: int = DEFAULT_PREC,
                       capacity_bytes: Optional[int] = None, out: Optional[np.ndarray] = None):
    """HOST numpy buffers in, HOST buffers out (copies inside): what bench.py's e2e leg times.
    Returns (out [n_streams, capacity] uint8, nbits [n_streams] uint64)."""
    logits = np.ascontiguousarray(logits, dtype=np.float32)
    syms = np.ascontiguousarray(syms, dtype=np.int32)
    S, T, V = logits.shape
    cap = int(capacity_bytes or (T * 8 + 64))
    if out is None:
        out = np.zeros((S, cap), dtype=np.uint8)
    nbits = np.zeros(S, dtype=np.uint64)
    check(lib().lac_encode_logits_host(logits.ctypes.data, syms.ctypes.data, S, T, V, out.ctypes.data, cap,
                                       nbits.ctypes.data, prec))
    return out, nbits


def decode_logits_host(logits: np.ndarray, data: np.ndarray, offsets: np.ndarray, prec: int = DEFAULT_PREC,
                       out: Optional[np.ndarray] = None) -> np.ndarray:
    logits = np.ascontiguousarray(logits, dtype=np.float32)
    data = np.ascontiguousarray(data, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    S, T, V = logits.shape
    if out is None:
        out = np.zeros((S, T), dtype=np.int32)
    check(lib().lac_decode_logits_host(logits.ctypes.data, S, T, V, data.ctypes.data, offsets.ctypes.data,
                                       out.ctypes.data, prec))
    return out
