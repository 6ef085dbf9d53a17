"""Prefill compression against stepwise compression, on one GPU.

    python tools/prefill_bench.py [--streams 256] [--chunk-tokens 2048] [--streams-8b 64] [--chunk-tokens-8b 512]

For the `1b` model one batch of --streams chunks x --chunk-tokens tokens (the configs[2] shape), and for the `8b`
model one smaller batch, it compresses and decompresses the same tokens (uniform random ids, as bench.py --workload
llama) with LlamaCompressor in torch mode and in batch-invariant mode.  Each call runs once as a warm-up (graph
capture) and once timed by the host clock, ending in a device synchronise; every decode is compared with the source.

For `1b` it also times, with CUDA events (median of 5 after a warm-up):
  * lac_model_gemm at each weight shape, for one prefill block (M = T_blk x streams) and one step (M = streams), as
    TFLOP/s and as a share of the NVIDIA data-sheet dense-BF16 rate for one B200 (2,250 TFLOP/s, not a measured peak);
  * one model.prefill block, and the attention launches inside it (their share of the block);
  * one model step in each mode (the decode step's model part, without the coder, launched eagerly), and the
    attention launches of a batch-invariant step.
The card's name, power limit and max SM clock are read in the same run.  Prints one JSON line; writes nothing.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

from adaptive_bench import card  # noqa: E402
from lac_b200 import _ffi, llama_compress as lc  # noqa: E402

DATASHEET_BF16_TFLOPS = 2250.0


def ev_time(fn, reps=5):
    fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def compress_roundtrip(cfg, S, T, bi, toks):
    model = lc.LlamaModel(cfg, n_streams=S, max_len=T, seed=0, batch_invariant=bi)
    comp = lc.LlamaCompressor(model, chunk_tokens=T)
    comp.compress(toks)
    tc, blob = wall(lambda: comp.compress(toks))
    comp.decompress(blob)
    td, back = wall(lambda: comp.decompress(blob))
    res = {"compress_s": round(tc, 3), "decompress_s": round(td, 3), "bytes": len(blob),
           "lossless": bool(np.array_equal(back, toks))}
    del comp, model
    torch.cuda.empty_cache()
    return res, blob


def kernel_times(cfg, S, T):
    m = lc.LlamaModel(cfg, n_streams=S, max_len=T, seed=0, batch_invariant=True)
    tb = lc.prefill_block(m)
    L, st = _ffi.lib(), torch.cuda.current_stream().cuda_stream
    gemms = {"wqkv": m.wqkv[0], "wo": m.wo[0], "w13": m.w13[0], "w2": m.w2[0], "head": m.head}
    out = {"prefill_block_positions": tb, "gemm": {}}
    for name, w in gemms.items():
        K, N = w.shape
        epi = _ffi.LAC_MODEL_OUT_F32 if name == "head" else _ffi.LAC_MODEL_OUT_BF16
        row = {"K": K, "N": N}
        for kind, M in (("prefill", tb * S), ("step", S)):
            x = torch.randn((M, K), device="cuda").to(torch.bfloat16)
            y = torch.empty((M, N), device="cuda", dtype=torch.float32 if epi == _ffi.LAC_MODEL_OUT_F32
                            else torch.bfloat16)
            ms = ev_time(lambda: _ffi.check(L.lac_model_gemm(x.data_ptr(), w.data_ptr(), M, N, K, epi, None,
                                                             y.data_ptr(), st)))
            tf = 2.0 * M * N * K / (ms * 1e-3) / 1e12
            row[kind] = {"M": M, "ms": round(ms, 4), "tflops": round(tf, 1),
                         "share_of_datasheet_bf16": round(tf / DATASHEET_BF16_TFLOPS, 3)}
        out["gemm"][name] = row
    # one prefill block in the middle of the chunk, and its attention launches alone
    p0 = (T // 2 // tb) * tb
    inp = torch.randint(0, cfg.vocab, (tb, S), device="cuda")
    block_ms = ev_time(lambda: m.prefill(inp, p0))
    H, KV, hd = cfg.heads, cfg.kv_heads, m.hd
    qkv = torch.randn((tb * S, (H + 2 * KV) * hd), device="cuda").to(torch.bfloat16)
    o = torch.empty((tb * S, H * hd), device="cuda", dtype=torch.bfloat16)

    def attn_all():
        for l in range(cfg.layers):
            _ffi.check(L.lac_model_attention(qkv.data_ptr(), S, tb, H, KV, hd, None, p0, m.kc[l].data_ptr(),
                                             m.vc[l].data_ptr(), m.max_len, o.data_ptr(), st))
    attn_ms = ev_time(attn_all)
    out["prefill_block"] = {"p0": p0, "ms": round(block_ms, 3), "attention_ms": round(attn_ms, 3),
                            "attention_share": round(attn_ms / block_ms, 3)}
    # the model part of one decode step at the same position, both modes, and the step's attention launches
    m.pos.fill_(p0)
    tok = torch.randint(0, cfg.vocab, (S,), device="cuda")
    out["model_step_ms"] = {"batch_invariant": round(ev_time(lambda: m.step(tok, T)), 3)}

    def attn_step():
        for l in range(cfg.layers):
            _ffi.check(L.lac_model_attention(qkv.data_ptr(), S, 1, H, KV, hd, m.pos.data_ptr(), 0,
                                             m.kc[l].data_ptr(), m.vc[l].data_ptr(), m.max_len, o.data_ptr(), st))
    out["model_step_ms"]["batch_invariant_attention"] = round(ev_time(attn_step), 3)
    del m
    torch.cuda.empty_cache()
    tm = lc.LlamaModel(cfg, n_streams=S, max_len=T, seed=0)
    tm.pos.fill_(p0)
    out["model_step_ms"]["torch"] = round(ev_time(lambda: tm.step(tok, lc._bucket_for(p0, T))), 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=256)
    ap.add_argument("--chunk-tokens", type=int, default=2048)
    ap.add_argument("--streams-8b", type=int, default=64)
    ap.add_argument("--chunk-tokens-8b", type=int, default=512)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prefill_bench needs a GPU")
    torch.cuda.set_device(0)
    line = {"tool": "prefill_bench", "card": card(), "runs": {}}
    for name, S, T in (("1b", args.streams, args.chunk_tokens), ("8b", args.streams_8b, args.chunk_tokens_8b)):
        cfg = lc.CONFIGS[name]
        toks = np.random.default_rng(0).integers(0, cfg.vocab, S * T).astype(np.int32)
        torch_mode, _ = compress_roundtrip(cfg, S, T, False, toks)
        bi_mode, _ = compress_roundtrip(cfg, S, T, True, toks)
        line["runs"][name] = {
            "model": cfg.describe(), "streams": S, "chunk_tokens": T,
            "torch": torch_mode, "batch_invariant": bi_mode,
            "compress_speedup": round(torch_mode["compress_s"] / bi_mode["compress_s"], 2),
            "decode_step_ms": {"torch": round(torch_mode["decompress_s"] / T * 1e3, 3),
                               "batch_invariant": round(bi_mode["decompress_s"] / T * 1e3, 3)}}
        if name == "1b":
            line["runs"][name]["kernels"] = kernel_times(cfg, S, T)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
