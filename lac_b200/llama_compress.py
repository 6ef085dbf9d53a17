"""The llama_compress.py path (reference llama_compress.py:1-61) on the GPU: an autoregressive model
predicts every token, the logits go through LQ32 and the batched range coder, independent chunks are
independent streams, batches of chunks shard over the GPUs of a box.

Reference behaviour kept:
  * every chunk starts from a reset model that has seen the BOS token 1 (Llama_AC.reset, :20-23);
  * the table for position t is computed from the logits after tokens < t (calc_dist, :24-30);
  * coder precision 48 (r(..., prec=48), :4);
  * an unknown token raises AssertionError("unknown symbol") (:51-52).
Reference behaviour replaced: tables are LQ32 (total 2^32) instead of cumsum(clip(softmax * 2^60, 2)) --
bound in DESIGN.md section 3 -- and chunks carry their token counts in the LACB container.  The reference's
context roll-over at n_ctx (accept, :31-39) does not arise: a chunk is at most max_len tokens.

Losslessness needs bit-identical logits when compressing and decompressing.  The reference gets that by
evaluating llama.cpp token by token in both directions; here both directions replay the SAME captured CUDA graph
of `model.step` with the same batch shape (chunks are coded in batches of exactly `batch_streams` streams), so
the same kernels run in the same order whether a file is written on one GPU and read on eight or the other way
round.

With LlamaModel(..., batch_invariant=True) the model runs the batch-invariant kernels of liblac_b200.so (DESIGN.md
section 13): a row's logits do not depend on how many rows or positions a launch covers, so the encoder computes a
whole block of positions in one prefill pass (StepEngine.prefill_encode_batch) and the stepwise decoder still
reproduces its logits bit for bit.

The per-token step -- model forward, LQ32 row summaries, fused symbol-range + range-coder kernel (or the decoder's
serial pass), position update -- is ONE CUDA graph replay with no host-fed inputs: the tokens of the step are
gathered on the device from the token matrix with the device-side position.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Optional

import numpy as np
import torch

from . import _ffi, coder, container, sharding

BOS = 1  # llama_compress.py:21 self.past = [1]


@dataclass(frozen=True)
class LlamaConfig:
    name: str
    vocab: int
    dim: int
    layers: int
    heads: int
    kv_heads: int
    ffn: int
    max_len: int = 2048

    def describe(self) -> str:
        return (f"{self.name}:v{self.vocab}:d{self.dim}:l{self.layers}:h{self.heads}:kv{self.kv_heads}:f{self.ffn}:"
                f"n{self.max_len}")

    @property
    def params(self) -> int:
        hd = self.dim // self.heads
        per_layer = self.dim * (self.heads + 2 * self.kv_heads) * hd + self.dim * self.dim + 3 * self.dim * self.ffn
        return self.layers * per_layer + 2 * self.vocab * self.dim


CONFIGS: Dict[str, LlamaConfig] = {
    # miniature for tests
    "tiny": LlamaConfig("tiny", 32000, 256, 2, 4, 2, 512, 2048),
    # configs[2]: "Llama-style ~1B random-init model (vocab 32000)" -- TinyLlama-1.1B geometry
    "1b": LlamaConfig("1b", 32000, 2048, 22, 32, 4, 5632, 2048),
    # configs[3]: Llama-3 8B geometry (vocab 128256)
    "8b": LlamaConfig("8b", 128256, 4096, 32, 32, 8, 14336, 2048),
    # configs[4]: a 1B-class predictor with the 128256 vocabulary (Llama-3.2-1B geometry) for 8192 concurrent streams
    "1b-128k": LlamaConfig("1b-128k", 128256, 2048, 16, 32, 8, 8192, 2048),
}

_BUCKETS = (128, 256, 512, 1024, 2048, 4096, 8192)


class LlamaModel(torch.nn.Module):
    """Llama-style decoder (RMSNorm, rotary GQA attention with a KV cache, SwiGLU), random-init, bf16 weights.
    step(tokens int64 [S]) -> fp32 logits [S, vocab] for the next position; the position lives on the device.
    All shapes are static for a given attention bucket, so a step can be captured into a CUDA graph.

    batch_invariant=True runs every layer on the lac_model_* kernels instead of torch ops (same weights, same
    function up to rounding), and adds prefill(): logits of a whole block of positions whose bits equal step()'s.
    In that mode step() and prefill() also take n <= S streams (the tokens' shape): they run on the first n slots of
    the KV cache, and a stream's logits are the same bits whatever n is."""

    def __init__(self, cfg: LlamaConfig, n_streams: int, max_len: Optional[int] = None, seed: int = 0,
                 device="cuda", dtype=torch.bfloat16, batch_invariant: bool = False):
        super().__init__()
        self.cfg, self.S = cfg, int(n_streams)
        self.batch_invariant = bool(batch_invariant)
        if self.batch_invariant and dtype != torch.bfloat16:
            raise ValueError("the batch-invariant kernels are bf16")
        self.max_len = int(max_len or cfg.max_len)
        self.device, self.dtype = torch.device(device), dtype
        g = torch.Generator(device=self.device).manual_seed(seed)
        hd = cfg.dim // cfg.heads
        self.hd = hd

        def w(*shape, scale):
            return (torch.randn(*shape, generator=g, device=self.device, dtype=torch.float32) * scale).to(dtype)
        d = cfg.dim
        self.emb = w(cfg.vocab, d, scale=1.0)
        self.wqkv = [w(d, (cfg.heads + 2 * cfg.kv_heads) * hd, scale=d ** -0.5) for _ in range(cfg.layers)]
        self.wo = [w(d, d, scale=d ** -0.5) for _ in range(cfg.layers)]
        self.w13 = [w(d, 2 * cfg.ffn, scale=d ** -0.5) for _ in range(cfg.layers)]
        self.w2 = [w(cfg.ffn, d, scale=cfg.ffn ** -0.5) for _ in range(cfg.layers)]
        self.head = w(d, cfg.vocab, scale=d ** -0.5 * 3.0)   # logit std ~3: a peaked, LLM-like next-token law
        inv = 1.0 / (10000 ** (torch.arange(0, hd, 2, device=self.device).float() / hd))
        ang = torch.arange(self.max_len, device=self.device).float()[:, None] * inv[None]
        self.cos = torch.cat([ang.cos(), ang.cos()], -1).to(dtype)    # rotate-half form, [max_len, hd]
        self.sin = torch.cat([ang.sin(), ang.sin()], -1).to(dtype)
        # KV cache [layer][S, kv_heads, max_len, hd]
        self.kc = [torch.zeros((self.S, cfg.kv_heads, self.max_len, hd), device=self.device, dtype=dtype)
                   for _ in range(cfg.layers)]
        self.vc = [torch.zeros_like(k) for k in self.kc]
        self.pos = torch.zeros(1, dtype=torch.int64, device=self.device)
        self.ar = torch.arange(self.max_len, device=self.device)

    def describe(self) -> str:
        """The predictor configuration a file records (its LACB model tag): the two modes round differently."""
        return self.cfg.describe() + (":bi" if self.batch_invariant else "")

    def reset(self):
        self.pos.zero_()

    def _norm(self, x):
        return torch.nn.functional.rms_norm(x, (x.shape[-1],), eps=1e-6)

    @staticmethod
    def _rope(x, c, s):  # x [S, heads, hd]; c, s [1, 1, hd]
        half = x.shape[-1] // 2
        rot = torch.cat([-x[..., half:], x[..., :half]], -1)
        return x * c + rot * s

    @torch.no_grad()
    def step(self, tokens: torch.Tensor, bucket: int) -> torch.Tensor:
        """One position for all S streams; attends over the first `bucket` cache slots (bucket > pos).  The
        attention is torch's scaled_dot_product_attention over the KV-cache slice with a position mask (measured
        against a bmm formulation and flash_attn_with_kvcache in tools/attn_bench.py: 0.10 vs 0.29 / 0.19 ms per
        layer at 256 streams x 2048 positions, deterministic).  Batch-invariant: tokens [n], 1 <= n <= S, streams
        0 .. n - 1, logits [n, vocab]."""
        if self.batch_invariant:
            n = tokens.shape[0]
            if not 1 <= n <= self.S:
                raise ValueError(f"step over {n} streams; this model holds 1 .. {self.S}")
            return self._forward_bi(tokens, self.pos, 0, 1)
        if tokens.shape[0] != self.S:
            raise ValueError(f"a torch-mode step runs exactly {self.S} streams, got {tokens.shape[0]}")
        cfg, S, hd = self.cfg, self.S, self.hd
        H, K = cfg.heads, cfg.kv_heads
        pos = self.pos
        c = self.cos.index_select(0, pos).view(1, 1, hd)
        s = self.sin.index_select(0, pos).view(1, 1, hd)
        mask = (self.ar[:bucket] <= pos).view(1, 1, 1, bucket)
        x = self.emb.index_select(0, tokens)
        for l in range(cfg.layers):
            qkv = (self._norm(x) @ self.wqkv[l]).view(S, H + 2 * K, hd)
            qk = self._rope(qkv[:, :H + K], c, s)
            self.kc[l].index_copy_(2, pos, qk[:, H:].unsqueeze(2))
            self.vc[l].index_copy_(2, pos, qkv[:, H + K:].unsqueeze(2))
            o = torch.nn.functional.scaled_dot_product_attention(
                qk[:, :H].unsqueeze(2), self.kc[l][:, :, :bucket], self.vc[l][:, :, :bucket], attn_mask=mask,
                enable_gqa=True)
            x = x + o.reshape(S, H * hd) @ self.wo[l]
            h13 = self._norm(x) @ self.w13[l]
            x = x + (torch.nn.functional.silu(h13[:, :cfg.ffn]) * h13[:, cfg.ffn:]) @ self.w2[l]
        return (self._norm(x) @ self.head).float()

    @torch.no_grad()
    def prefill(self, tokens: torch.Tensor, p0: int) -> torch.Tensor:
        """tokens [T_blk, n] (position-major: row t holds every stream's input at position p0 + t; n <= S streams)
        -> fp32 logits [T_blk, n, vocab].  Writes the KV cache at positions p0 .. p0 + T_blk - 1 and leaves `pos`
        alone.  Row (t, s) equals, bit for bit, what step() returns for stream s at position p0 + t after the same
        inputs."""
        if not self.batch_invariant:
            raise ValueError("prefill() needs LlamaModel(..., batch_invariant=True)")
        Tb, n = tokens.shape
        if not 1 <= n <= self.S or p0 < 0 or p0 + Tb > self.max_len:
            raise ValueError(f"prefill block [{Tb}, {n}] at p0={p0} does not fit [*, <= {self.S}] x {self.max_len}")
        return self._forward_bi(tokens.reshape(-1), None, int(p0), Tb).view(Tb, n, self.cfg.vocab)

    def _forward_bi(self, tokens, d_pos, p0, n_q):
        """The model on the lac_model_* kernels over n_q positions x S streams (rows position-major), S the
        tokens' stream count: the first S slots of the KV cache."""
        cfg, hd = self.cfg, self.hd
        S = tokens.numel() // n_q
        H, K, d, M = cfg.heads, cfg.kv_heads, cfg.dim, tokens.numel()
        L, st = _ffi.lib(), torch.cuda.current_stream(self.device).cuda_stream
        pos_p = d_pos.data_ptr() if d_pos is not None else None
        x = self.emb.index_select(0, tokens)
        h = torch.empty_like(x)
        qkv = torch.empty((M, (H + 2 * K) * hd), device=self.device, dtype=self.dtype)
        o = torch.empty((M, H * hd), device=self.device, dtype=self.dtype)
        h13 = torch.empty((M, 2 * cfg.ffn), device=self.device, dtype=self.dtype)
        f = torch.empty((M, cfg.ffn), device=self.device, dtype=self.dtype)
        logits = torch.empty((M, cfg.vocab), device=self.device, dtype=torch.float32)

        def gemm(a, w, epi, y, res=None):
            _ffi.check(L.lac_model_gemm(a.data_ptr(), w.data_ptr(), M, w.shape[1], w.shape[0], epi,
                                        None if res is None else res.data_ptr(), y.data_ptr(), st))

        def norm(a, y):
            _ffi.check(L.lac_model_rmsnorm(a.data_ptr(), M, d, 1e-6, y.data_ptr(), st))
        for l in range(cfg.layers):
            norm(x, h)
            gemm(h, self.wqkv[l], _ffi.LAC_MODEL_OUT_BF16, qkv)
            _ffi.check(L.lac_model_rope_kv(qkv.data_ptr(), M, S, H, K, hd, self.cos.data_ptr(), self.sin.data_ptr(),
                                           pos_p, p0, self.kc[l].data_ptr(), self.vc[l].data_ptr(), self.max_len, st))
            _ffi.check(L.lac_model_attention(qkv.data_ptr(), S, n_q, H, K, hd, pos_p, p0, self.kc[l].data_ptr(),
                                             self.vc[l].data_ptr(), self.max_len, o.data_ptr(), st))
            gemm(o, self.wo[l], _ffi.LAC_MODEL_OUT_BF16_ADD, x, res=x)
            norm(x, h)
            gemm(h, self.w13[l], _ffi.LAC_MODEL_OUT_BF16, h13)
            _ffi.check(L.lac_model_swiglu(h13.data_ptr(), M, cfg.ffn, f.data_ptr(), st))
            gemm(f, self.w2[l], _ffi.LAC_MODEL_OUT_BF16_ADD, x, res=x)
        norm(x, h)
        gemm(h, self.head, _ffi.LAC_MODEL_OUT_F32, logits)
        return logits


# Logits of one prefill block (fp32 [T_blk, S, vocab]) stay within this many bytes: T_blk = budget // (4 S vocab).
PREFILL_LOGITS_BYTES = 1 << 31


def prefill_block(model: "LlamaModel") -> int:
    """Positions per prefill block for this model's batch shape."""
    return max(1, PREFILL_LOGITS_BYTES // (4 * model.S * model.cfg.vocab))


def _bucket_for(pos: int, max_len: int) -> int:
    for b in _BUCKETS:
        if pos < b:
            return min(b, max_len)
    return max_len


def active_streams(count: int, S: int) -> int:
    """The stream count a batch-invariant decode of `count` streams runs at: the smallest rung >= count of the
    ladder 1, 2, 4, ... (powers of two below S), S.  A fixed ladder bounds the graphs to about log2(S) + 1 per
    direction."""
    if not 1 <= count <= S:
        raise ValueError(f"{count} streams do not fit a batch of {S}")
    n = 1
    while n < count:
        n *= 2
    return min(n, S)


class StepEngine:
    """The per-token loop of one batch: holds the model, the static device buffers and one captured CUDA graph per
    (direction, attention bucket, active streams).  A step is `graph.replay()`; nothing is fed from the host.

    A torch-mode model always runs its S streams.  A batch-invariant model decodes a batch of any size <= S at the
    active stream count active_streams(): the first n rows of the buffers and of the KV cache, one decoder per n,
    the workspace sized for S.  Its attention reads the position itself, so that is one graph per (direction, n)."""

    def __init__(self, model: LlamaModel, chunk_tokens: int, prec: int, use_graphs: bool = True):
        self.m, self.T, self.prec, self.use_graphs = model, int(chunk_tokens), int(prec), use_graphs
        S, V, dev = model.S, model.cfg.vocab, model.device
        if self.T > model.max_len:
            raise ValueError("chunk_tokens exceeds the model's max_len")
        self.tok = torch.zeros((S, self.T), dtype=torch.int32, device=dev)      # encode: input; decode: output
        self.ntok = torch.zeros(S, dtype=torch.int32, device=dev)
        self.live = torch.zeros(S, dtype=torch.int32, device=dev)
        self.sym = torch.zeros(S, dtype=torch.int32, device=dev)
        self.ws = coder.Workspace(S, V, dev)
        self.cap = self.T * 8 + 64
        self.enc: Optional[coder.StreamEncoder] = None
        self.dec: Optional[coder.StreamDecoder] = None
        self.decs: Dict[int, coder.StreamDecoder] = {}   # decoder per active stream count
        self.n = S                                       # active streams of the batch being coded
        self.graphs: Dict = {}
        self.stream = torch.cuda.Stream(device=dev)

    # ---- one step, expressed on device tensors only
    def _prev_tokens(self):
        pos = self.m.pos
        prev = self.tok[:self.n].index_select(1, (pos - 1).clamp_(min=0)).squeeze(1).to(torch.int64)
        return torch.where(pos > 0, prev, torch.full_like(prev, BOS))

    def _enc_step(self, bucket):
        logits = self.m.step(self._prev_tokens(), bucket)
        pos = self.m.pos
        self.sym.copy_(self.tok.index_select(1, pos).squeeze(1))
        self.live.copy_((self.ntok > pos).to(torch.int32))
        self.enc.encode_step(logits, self.sym, self.live, self.ws)
        pos.add_(1)

    def _dec_step(self, bucket):
        n = self.n
        tok, live, sym = self.tok[:n], self.live[:n], self.sym[:n]
        logits = self.m.step(self._prev_tokens(), bucket)
        pos = self.m.pos
        live.copy_((self.ntok[:n] > pos).to(torch.int32))
        self.dec.decode_step(logits, live, self.ws, out=sym)
        tok.index_copy_(1, pos, torch.where(live > 0, sym, torch.zeros_like(sym)).unsqueeze(1))
        pos.add_(1)

    def _run(self, kind, n_steps):
        fn = self._enc_step if kind == "enc" else self._dec_step
        cur = torch.cuda.current_stream(self.m.device)
        self.stream.wait_stream(cur)
        with torch.cuda.stream(self.stream):
            for t in range(n_steps):
                # the batch-invariant attention reads the position itself: one graph per direction
                bucket = self.m.max_len if self.m.batch_invariant else _bucket_for(t, self.m.max_len)
                if not self.use_graphs:
                    fn(bucket)
                    continue
                key = (kind, bucket, self.n)
                if key not in self.graphs:
                    # warm-up run outside capture (cuBLAS handles / workspaces), then rewind what it changed
                    snap = self._snapshot(kind)
                    fn(bucket)
                    self._restore(kind, snap)
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=self.stream):
                        fn(bucket)
                    self._restore(kind, snap)
                    self.graphs[key] = g
                self.graphs[key].replay()
        cur.wait_stream(self.stream)

    def _snapshot(self, kind):
        """Everything a step changes that the next step reads: position, coder state, decoded tokens, and -- encode
        side -- the stream bytes (a carry ripples into bytes already written, so a repeated step would add it twice)."""
        st = self.enc.state if kind == "enc" else self.dec.state
        out = self.enc.out.clone() if kind == "enc" else None
        return (self.m.pos.clone(), st.clone(), self.tok.clone(), out)

    def _restore(self, kind, snap):
        st = self.enc.state if kind == "enc" else self.dec.state
        self.m.pos.copy_(snap[0])
        st.copy_(snap[1])
        self.tok.copy_(snap[2])
        if snap[3] is not None:
            self.enc.out.copy_(snap[3])

    # ---- whole batches
    def encode_batch(self, tokens: np.ndarray, ntok: np.ndarray):
        S = self.n = self.m.S
        assert tokens.shape == (S, self.T) and ntok.shape == (S,)
        self.tok.copy_(torch.from_numpy(np.ascontiguousarray(tokens, dtype=np.int32)))
        self.ntok.copy_(torch.from_numpy(np.ascontiguousarray(ntok, dtype=np.int32)))
        if self.enc is None:
            self.enc = coder.StreamEncoder(S, prec=self.prec, capacity_bytes=self.cap, device=self.m.device)
        else:
            self.enc.reset()
        self.m.reset()
        self._run("enc", int(ntok.max()) if len(ntok) else 0)
        self.enc.finish()
        return self.enc.bitstreams()

    def prefill_encode_batch(self, tokens: np.ndarray, ntok: np.ndarray):
        """encode_batch through model.prefill (batch-invariant models): the chunk in blocks of prefill_block()
        positions, one prefill and one encode call per block.  The same bitstreams as encode_batch."""
        S, T, V = self.m.S, self.T, self.m.cfg.vocab
        assert tokens.shape == (S, T) and ntok.shape == (S,)
        self.tok.copy_(torch.from_numpy(np.ascontiguousarray(tokens, dtype=np.int32)))
        self.ntok.copy_(torch.from_numpy(np.ascontiguousarray(ntok, dtype=np.int32)))
        if self.enc is None:
            self.enc = coder.StreamEncoder(S, prec=self.prec, capacity_bytes=self.cap, device=self.m.device)
        else:
            self.enc.reset()
        self.m.reset()
        n = int(ntok.max()) if len(ntok) else 0
        tb = prefill_block(self.m)
        L, st = _ffi.lib(), torch.cuda.current_stream(self.m.device).cuda_stream
        inp = torch.cat([torch.full((S, 1), BOS, dtype=torch.int64, device=self.m.device),
                         self.tok[:, :T - 1].to(torch.int64)], 1)        # the model's input at every position
        ws = coder.Workspace(S * tb, V, self.m.device)
        for p0 in range(0, n, tb):
            nb = min(tb, n - p0)
            logits = self.m.prefill(inp[:, p0:p0 + nb].t().contiguous(), p0)
            cnt = (self.ntok - p0).clamp_(0, nb).to(torch.int32)
            _ffi.check(L.lac_ac_encode_logits_f32(logits.data_ptr(), S, nb, V, S * V, V, self.tok[:, p0:].data_ptr(),
                                                  T, cnt.data_ptr(), self.enc.state.data_ptr(),
                                                  self.enc.out.data_ptr(), self.cap, 0, self.prec, ws.ptr, ws.nbytes,
                                                  st))
        self.enc.finish()
        return self.enc.bitstreams()

    def decode_batch(self, streams: List[bytes], ntok: np.ndarray) -> np.ndarray:
        """Decode ntok[i] tokens of streams[i] -> int32 [len(streams), chunk_tokens].  A torch-mode model takes
        exactly S streams; a batch-invariant one any 1 .. S, run at active_streams() with empty padding streams."""
        S, B = self.m.S, len(streams)
        assert ntok.shape == (B,) and (B == S or (self.m.batch_invariant and 1 <= B <= S))
        n = self.n = active_streams(B, S) if self.m.batch_invariant else S
        streams = list(streams) + [b""] * (n - B)
        self.ntok.zero_()
        self.ntok[:B].copy_(torch.from_numpy(np.ascontiguousarray(ntok, dtype=np.int32)))
        self.tok.zero_()
        self.dec = self.decs.get(n)
        if self.dec is None:
            self.dec = self.decs[n] = coder.StreamDecoder(streams, prec=self.prec, device=self.m.device,
                                                          capacity_bytes=n * self.cap)
        else:
            self.dec.reset(streams)
        self.m.reset()
        self._run("dec", int(ntok.max()) if len(ntok) else 0)
        st = self.dec.status()
        if st & _ffi.LAC_ST_TRUNC:
            raise _ffi.LacError(_ffi.LAC_E_STREAM, "truncated or foreign bitstream (wrong model for this file?)")
        return self.tok[:B].cpu().numpy()


class LlamaCompressor:
    """compress(token ids) -> LACB bytes, decompress(bytes[, start, stop]) -> token ids.  With torch.distributed
    initialised every rank calls both with the same arguments; rank 0 gets the result, the others None."""

    def __init__(self, model: LlamaModel, chunk_tokens: int = 2048, prec: int = coder.DEFAULT_PREC,
                 use_graphs: bool = True, group=None):
        self.model, self.chunk, self.prec, self.group = model, int(chunk_tokens), int(prec), group
        self.vocab = model.cfg.vocab
        self.engine = StepEngine(model, chunk_tokens, prec, use_graphs)
        self.tag = container.model_tag(model.describe())

    def compress(self, tokens) -> Optional[bytes]:
        toks = np.ascontiguousarray(tokens, dtype=np.int32)
        if toks.size and (int(toks.min()) < 0 or int(toks.max()) >= self.vocab):
            bad = int(toks.max()) if int(toks.max()) >= self.vocab else int(toks.min())
            raise AssertionError("unknown symbol", bad)  # llama_compress.py:51-52
        encode = self.engine.prefill_encode_batch if self.model.batch_invariant else self.engine.encode_batch
        return sharding.compress_sharded(toks, self.chunk, self.model.S, encode, self.prec, self.vocab,
                                         self.model.device, self.tag, self.group)

    def decompress(self, blob: bytes, start: Optional[int] = None, stop: Optional[int] = None) -> Optional[np.ndarray]:
        """The tokens of the file, or tokens[start:stop] (0 <= start <= stop <= total, no negative indices).

        A torch-mode file decodes in the batches it was written in (the header's batch_streams must be this model's
        S): only the batches that hold the range, each for as many steps as its needed chunks reach into it.  A file
        written by this batch-invariant predictor (its tag ends in :bi) decodes at any S: only the needed chunks,
        packed into batches of similar length (sharding.decompress_packed); its batch_streams is informational."""
        c = container.unpack(blob)
        if c.vocab != self.vocab or c.quantiser != container.QUANT_LQ32:
            raise ValueError("container was written for a different vocabulary / quantiser")
        packed = self.model.batch_invariant and c.tag == self.tag
        if (not packed and c.batch_streams != self.model.S) or c.chunk_tokens != self.chunk:
            raise ValueError(f"container was written with batches of {c.batch_streams} streams x {c.chunk_tokens} "
                             f"tokens; this compressor runs {self.model.S} x {self.chunk}")
        if c.tag and c.tag != self.tag:
            raise ValueError("container was written with a different predictor configuration")
        start = 0 if start is None else start
        if packed:
            return sharding.decompress_packed(blob, self.engine.decode_batch, self.model.S, self.model.device,
                                              self.group, start, stop)
        return sharding.decompress_sharded(blob, self.engine.decode_batch, self.model.device, self.group, start, stop)


# ------------------------------------------------------------------ the reference's own entry points
from .arith_code import AC, ProbPredictor  # noqa: E402


class Llama_AC(ProbPredictor):
    """Drop-in for the reference's Llama_AC (llama_compress.py:14-61): a predictor around a llama_cpp.Llama-like
    object -- anything with reset(), eval(tokens), n_ctx() and _scores[-1] (the fp32 logits row of the current
    position, numpy or torch).  AC(Llama_AC(llm), 48).to_bin / .from_bin then code through the LQ32 kernels: the
    row goes to the device once per token (logits_row) and lac_ac_encode_logits_f32 / lac_ac_decode_logits_f32 do
    calc_dist + symbol_to_range / val_to_symbol + the coder step.  The tables are LQ32's, not the reference's
    cumsum(clip(softmax * 2^60, 2)) (whose re-scaling wraps int64, DESIGN.md section 1), so the bitstreams are not
    interchangeable with the reference's; calc_dist() returns the LQ32 table in the reference's layout (inclusive
    cumulative, total 2^32) for callers that look at it."""

    def __init__(self, llm, maxtoks=2048):
        super().__init__(0)
        self.llm = llm
        self.overlap = 2
        self.reset()

    def reset(self):                                       # :20-23
        self.past = [BOS]
        self.llm.reset()
        self.llm.eval([BOS])
        self.dcache = None

    def logits_row(self) -> torch.Tensor:
        row = self.llm._scores[-1]
        if not isinstance(row, torch.Tensor):
            row = torch.from_numpy(np.ascontiguousarray(row, dtype=np.float32))
        return row.to(device="cuda", dtype=torch.float32).contiguous().view(-1)

    def calc_dist(self):                                   # :24-30, LQ32 instead of the float cumsum
        cum = coder.cdf_build(self.logits_row().view(1, -1))
        self.dcache = coder.cdf_to_dist(cum)[0]
        return self.dcache

    @property
    def minp(self):                                        # :43-45
        d = self.dist
        return int(min(int(d[0]), int(np.min(np.diff(d)))))

    def accept(self, symbol):                              # :31-39
        self.past.append(symbol)
        if len(self.past) == self.llm.n_ctx():
            self.past = self.past[self.llm.n_ctx() - self.llm.n_ctx() // self.overlap:]
            self.llm.reset()
            self.llm.eval(self.past)
        else:
            self.llm.eval([symbol])
        return super().accept(symbol)

    def copy(self):                                        # :40-41
        return Llama_AC(self.llm)


_llm = None


def r(model_path="../../llama.cpp/models/llama-2-7b.ggmlv3.q5_1.bin", prec=48):
    """llama_compress.py:4-10: AC(Llama_AC(llama_cpp.Llama(model_path, n_ctx=512)), prec)."""
    import llama_cpp
    global _llm
    if _llm is None:
        _llm = llama_cpp.Llama(model_path=model_path, n_ctx=512)
    return AC(Llama_AC(_llm), prec)
