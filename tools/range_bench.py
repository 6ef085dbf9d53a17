"""Token-range reads of an LACB file written by the model in the loop, on one GPU.

    python tools/range_bench.py [--model 1b] [--batches 4] [--batch-streams 256] [--chunk-tokens 2048] [--reps 3]

Writes one file of --batches x --batch-streams chunks x --chunk-tokens tokens (synthetic text: uniform random token
ids, as bench.py --workload llama) with LlamaCompressor, then times LlamaCompressor.decompress(blob, start, stop) for:
  * the whole file;
  * one full chunk of the middle batch;
  * 64 tokens at the start of that chunk;
  * 64 tokens ending at that chunk's last position;
  * 2 x chunk-tokens across the boundary in front of the middle batch.
Each read: one warm-up, then the median (and min) of --reps host wall-clock times, each ending in a device
synchronise; every read is compared with the source tokens.  `model_steps` is the sum over the decoded batches of
the furthest position a needed chunk is read to, which is what a read costs.  The card's name, power limit and max
SM clock are read in the same run.  Prints one JSON line and writes nothing to disk.
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
from lac_b200 import llama_compress as lc  # noqa: E402


def timed_read(comp, blob, toks, start, stop, reps):
    want = toks[start:stop]
    times, lossless = [], True
    for i in range(reps + 1):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        got = comp.decompress(blob, start, stop)
        torch.cuda.synchronize()
        if i:
            times.append(time.perf_counter() - t0)
        lossless = lossless and got.dtype == np.int32 and np.array_equal(got, want)
    return float(np.median(times)), float(min(times)), lossless


def model_steps(chunk, B, n_chunks, start, stop):
    steps = {}
    for i in range(n_chunks):
        if max(i * chunk, start) < min((i + 1) * chunk, stop):
            steps[i // B] = max(steps.get(i // B, 0), min(chunk, stop - i * chunk))
    return sum(steps.values()), len(steps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", default="1b", help="lac_b200.llama_compress.CONFIGS key")
    ap.add_argument("--batches", type=int, default=4)
    ap.add_argument("--batch-streams", type=int, default=256)
    ap.add_argument("--chunk-tokens", type=int, default=2048)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("range_bench.py needs a GPU")
    torch.cuda.set_device(0)
    cfg, B, T = lc.CONFIGS[args.model], args.batch_streams, args.chunk_tokens
    n_chunks = args.batches * B
    n_tokens = n_chunks * T
    toks = np.random.default_rng(2024).integers(0, cfg.vocab, n_tokens).astype(np.int32)
    comp = lc.LlamaCompressor(lc.LlamaModel(cfg, n_streams=B, max_len=T, seed=0), chunk_tokens=T)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    blob = comp.compress(toks)
    torch.cuda.synchronize()
    compress_s = time.perf_counter() - t0        # includes capturing the encode graphs
    mid = args.batches // 2                      # the middle batch, and its middle chunk
    c0 = (mid * B + B // 2) * T
    reads = {
        "whole_file": (0, n_tokens),
        "one_chunk": (c0, c0 + T),
        "64_at_chunk_start": (c0, c0 + 64),
        "64_at_chunk_end": (c0 + T - 64, c0 + T),
        "across_batch_boundary": (mid * B * T - T, mid * B * T + T),
    }
    res = {}
    for name, (start, stop) in reads.items():
        med, mn, ok = timed_read(comp, blob, toks, start, stop, args.reps)
        steps, batches = model_steps(T, B, n_chunks, start, stop)
        res[name] = {"start": start, "stop": stop, "tokens": stop - start, "batches_decoded": batches,
                     "model_steps": steps, "s": med, "s_min": mn, "ms_per_model_step": 1e3 * med / steps,
                     "lossless": ok}
    line = {"tool": "range_bench", "card": card(), "model": cfg.describe(),
            "params_b": round(cfg.params / 1e9, 3), "file": {"batches": args.batches, "batch_streams": B,
                                                             "chunk_tokens": T, "tokens": n_tokens,
                                                             "bytes": len(blob), "compress_s": compress_s},
            "reps": args.reps, "reads": res, "lossless": all(r["lossless"] for r in res.values())}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
