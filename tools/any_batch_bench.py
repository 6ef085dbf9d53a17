"""Decoding batch-invariant files at any batch size, on one GPU (`1b` model, batch-invariant mode).

    python tools/any_batch_bench.py [--baseline-lib PATH] [--reps 3] [--sections gemm,steps,reads] [--reads a,b]

Three sections, one JSON line, nothing written to disk; the card's name, power limit and max SM clock are read in
the same run.
  * gemm: lac_model_gemm at M in {1, 8, 32, 128, 256} on each `1b` weight shape (bf16 epilogue; fp32 for the head):
    time (CUDA events, median of 5 windows of 20 launches after a warm-up) and weight bytes per second.  Each launch
    reads another copy of the weight, the copies together >= 512 MB, so the weights come from HBM as in a model step,
    not from the 126 MB L2.  With --baseline-lib (another build of liblac_b200.so, e.g. of an earlier commit) the
    same launches run on that library too, alternating with this one, so both are timed under the same conditions.
  * steps: one model step (the model part of a decode step, replayed from a CUDA graph) at active stream counts n in
    {1, 4, 16, 64, 256} and positions 64 and 1000; CUDA events, median of 5 windows of 20 replays.
  * reads: a file of 257 chunks x 2048 tokens written at S = 256 by prefill -- two batches, the second holding one
    chunk (uniform random token ids, as bench.py --workload llama).  Token-range reads the old way
    (sharding.decompress_sharded: the file's batches at full S, other slots empty) and the new way
    (LlamaCompressor.decompress: needed chunks packed, sharding.decompress_packed): 64 tokens at a chunk start, one
    full chunk, 64 tokens across the boundary of the two batches, the first 256 chunks plus 64 tokens of the last
    one, and the whole file, the new way also with a decoder of S = 512.  --reads picks a subset by name.  Host
    wall clock ending in a device synchronise, median of --reps after a warm-up read; every read is compared with
    the source.
"""
import argparse
import ctypes as C
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
from lac_b200 import _ffi, sharding, llama_compress as lc  # noqa: E402

GEMM_M = (1, 8, 32, 128, 256)
STEP_N = (1, 4, 16, 64, 256)
STEP_POS = (64, 1000)


def ev_windows(fn, launches=20, windows=5):
    """Median ms per call over `windows` event-timed windows of `launches` calls, after one warm-up window."""
    for _ in range(launches):
        fn()
    ts = []
    for _ in range(windows):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(launches):
            fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) / launches)
    return float(np.median(ts))


def load_gemm(path):
    L = C.CDLL(path)
    L.lac_model_gemm.argtypes = _ffi.SIGNATURES["lac_model_gemm"]
    L.lac_model_gemm.restype = C.c_int
    return L


def gemm_section(m, baseline):
    libs = {"this": _ffi.lib()}
    if baseline:
        libs["baseline"] = load_gemm(baseline)
    st = torch.cuda.current_stream().cuda_stream
    out = {}
    for name, w in (("wqkv", m.wqkv[0]), ("wo", m.wo[0]), ("w13", m.w13[0]), ("w2", m.w2[0]), ("head", m.head)):
        K, N = w.shape
        wbytes = K * N * 2
        copies = [w] + [w.clone() for _ in range(max(1, -(-(512 << 20) // wbytes)) - 1)]
        epi = _ffi.LAC_MODEL_OUT_F32 if name == "head" else _ffi.LAC_MODEL_OUT_BF16
        row = {"K": K, "N": N, "weight_copies": len(copies)}
        for M in GEMM_M:
            x = torch.randn((M, K), device="cuda").to(torch.bfloat16)
            y = torch.empty((M, N), device="cuda",
                            dtype=torch.float32 if epi == _ffi.LAC_MODEL_OUT_F32 else torch.bfloat16)
            ring = [0]

            def launch(L):
                c = copies[ring[0] % len(copies)]
                ring[0] += 1
                rc = L.lac_model_gemm(x.data_ptr(), c.data_ptr(), M, N, K, epi, None, y.data_ptr(), st)
                if rc:
                    raise RuntimeError(f"lac_model_gemm returned {rc}")
            res = {}
            for _ in range(2):              # alternate the libraries twice; keep each one's best median
                for tag, L in libs.items():
                    ms = ev_windows(lambda: launch(L))
                    res[tag] = min(res.get(tag, ms), ms)
            cell = {t: {"us": round(ms * 1e3, 2), "weight_GBps": round(wbytes / (ms * 1e-3) / 1e9, 1)}
                    for t, ms in res.items()}
            if baseline:
                cell["speedup"] = round(res["baseline"] / res["this"], 2)
            row[f"M{M}"] = cell
        out[name] = row
        del copies
        torch.cuda.empty_cache()
    return out


def step_section(m):
    out = {}
    for n in STEP_N:
        tok = torch.randint(0, m.cfg.vocab, (n,), device="cuda")
        for p in STEP_POS:
            m.pos.fill_(p)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                m.step(tok, m.max_len)
            torch.cuda.current_stream().wait_stream(side)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                m.step(tok, m.max_len)
            out[f"n{n}_pos{p}"] = {"n": n, "pos": p, "ms": round(ev_windows(g.replay), 3)}
            del g
    return out


def timed(fn, want, reps):
    times, ok = [], True
    for i in range(reps + 1):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        got = fn()
        torch.cuda.synchronize()
        if i:
            times.append(time.perf_counter() - t0)
        ok = ok and got.dtype == np.int32 and np.array_equal(got, want)
    return {"s": round(float(np.median(times)), 4), "s_min": round(float(min(times)), 4), "lossless": ok}


READS = ("64_at_chunk_start", "one_chunk", "64_across_batch_boundary", "S_chunks_plus_64", "whole_file")


def read_section(cfg, reps, names):
    S, T = 256, 2048
    n_chunks = S + 1
    toks = np.random.default_rng(2024).integers(0, cfg.vocab, n_chunks * T).astype(np.int32)
    comp = lc.LlamaCompressor(lc.LlamaModel(cfg, n_streams=S, max_len=T, seed=0, batch_invariant=True),
                              chunk_tokens=T)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    blob = comp.compress(toks)
    torch.cuda.synchronize()
    out = {"file": {"chunks": n_chunks, "chunk_tokens": T, "written_at_S": S, "bytes": len(blob),
                    "compress_s": round(time.perf_counter() - t0, 3)}}
    c0 = (S // 2) * T
    reads = {"64_at_chunk_start": (c0, c0 + 64), "one_chunk": (c0, c0 + T),
             "64_across_batch_boundary": (S * T - 32, S * T + 32), "S_chunks_plus_64": (0, S * T + 64),
             "whole_file": (0, n_chunks * T)}
    reads = {k: v for k, v in reads.items() if k in names}

    def old(a, b):
        return sharding.decompress_sharded(blob, comp.engine.decode_batch, comp.model.device, None, a, b)
    for name, (a, b) in reads.items():
        out[name] = {"start": a, "stop": b, "old_S256": timed(lambda: old(a, b), toks[a:b], reps),
                     "new_S256": timed(lambda: comp.decompress(blob, a, b), toks[a:b], reps)}
        out[name]["speedup"] = round(out[name]["old_S256"]["s"] / out[name]["new_S256"]["s"], 2)
    del comp
    torch.cuda.empty_cache()
    if "whole_file" in reads:
        big = lc.LlamaCompressor(lc.LlamaModel(cfg, n_streams=2 * S, max_len=T, seed=0, batch_invariant=True),
                                 chunk_tokens=T)
        out["whole_file"]["new_S512"] = timed(lambda: big.decompress(blob), toks, reps)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline-lib", default=None, help="another liblac_b200.so to time lac_model_gemm against")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--sections", default="gemm,steps,reads", help="comma-separated subset of gemm,steps,reads")
    ap.add_argument("--reads", default=",".join(READS), help="comma-separated subset of " + ",".join(READS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("any_batch_bench.py needs a GPU")
    torch.cuda.set_device(0)
    cfg = lc.CONFIGS["1b"]
    sections = set(args.sections.split(","))
    line = {"tool": "any_batch_bench", "card": card(), "model": cfg.describe() + ":bi"}
    if sections & {"gemm", "steps"}:
        m = lc.LlamaModel(cfg, n_streams=max(STEP_N), max_len=cfg.max_len, seed=0, batch_invariant=True)
        if "gemm" in sections:
            line["gemm"] = gemm_section(m, args.baseline_lib)
        if "steps" in sections:
            line["steps"] = step_section(m)
        del m
        torch.cuda.empty_cache()
    if "reads" in sections:
        line["reads"] = read_section(cfg, args.reps, set(args.reads.split(",")))
        line["lossless"] = all(v["lossless"] for r in line["reads"].values() if isinstance(r, dict)
                               for k, v in r.items() if isinstance(v, dict) and "lossless" in v)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
