"""Speed of the adaptive count models (prob(s) = 1 + occurrences of s so far, 256 byte symbols) on one GPU.

    python tools/adaptive_bench.py [--streams 8192] [--reps 3]

Prints one JSON line:
  * config0: BASELINE configs[0], the 64 KB golden byte stream (tests/golden/acs_64k.npz) under ACSampler at prec 48:
    the acs_encode_adaptive and acs_decode_adaptive call times (CUDA events, median of --reps after a warm-up call),
    next to the table path it replaces: materialise_tables on the host, the [65536, 256] int64 copy to the device
    and acs_encode_tables.  The table path has no decoder.
  * batch: --streams independent 64 KB streams of synthetic text (a word-salad pool like the goldens', each stream at
    its own offset), for both models (ac: A_to_bin at prec 32, acs: ACSampler at prec 48): input bytes per second of
    one encode call and of one decode call, each direction timed on its own (median of --reps after a warm-up call),
    and whether every stream decoded back.
The card's name and power limit are read in the same run.  Writes nothing to disk.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from lac_b200 import arith_code as ac  # noqa: E402
from lac_b200 import coder  # noqa: E402

N = 65536


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30)
        pl, clk = [x.strip() for x in q.stdout.strip().split(",")[:2]]
        info.update(power_limit_w=float(pl), max_sm_clock_mhz=float(clk))
    except Exception as e:  # the numbers stay without it; say so
        info["power_limit_w"] = f"not read: {e}"
    return info


def timed(fn, prep, reps):
    """fn() after prep() (outside the window): one warm-up, then the median and min of `reps` CUDA-event times (ms)."""
    prep()
    fn()
    out = []
    for _ in range(reps):
        prep()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return float(np.median(out)), float(min(out))


def config0(reps):
    g = np.load(os.path.join(ROOT, "tests", "golden", "acs_64k.npz"))
    data, prec = g["data"], int(g["prec"])
    syms = torch.from_numpy(data.astype(np.int32)[None]).cuda()
    enc = coder.StreamEncoder(1, prec=prec, capacity_bytes=N)
    counts = coder.Counts(1, 256)

    def prep_enc():
        enc.reset()
        counts.reset()

    enc_ms = timed(lambda: enc.acs_encode_adaptive(syms, counts, finish="safe"), prep_enc, reps)
    streams, _ = enc.bitstreams()
    dec = coder.StreamDecoder(streams, prec=prec)
    dcounts = coder.Counts(1, 256)
    out = {}

    def prep_dec():
        dec.reset(streams)
        dcounts.reset()

    def run_dec():
        out["syms"] = dec.acs_decode_adaptive(dcounts, N, check_status=False)

    dec_ms = timed(run_dec, prep_dec, reps)
    lossless = bool(np.array_equal(out["syms"].cpu().numpy()[0], data))
    # the table path: host tables, one copy, one table-driven encode call
    t0 = time.perf_counter()
    dist, _ = ac.materialise_tables(ac.CountPredictor(256), data.tolist())
    host_s = time.perf_counter() - t0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    d_dist = torch.from_numpy(dist).cuda()
    torch.cuda.synchronize()
    copy_s = time.perf_counter() - t0
    enc2 = coder.StreamEncoder(1, prec=prec, capacity_bytes=N)
    tab_ms = timed(lambda: enc2.acs_encode_tables(d_dist, syms, finish="safe"), enc2.reset, reps)
    same = enc2.bitstreams()[0] == streams
    return {"bytes": N, "prec": prec, "model": "acs",
            "adaptive": {"encode_ms": enc_ms[0], "encode_ms_min": enc_ms[1], "decode_ms": dec_ms[0],
                         "decode_ms_min": dec_ms[1], "lossless": lossless},
            "tables": {"materialise_s": host_s, "table_mb": dist.nbytes / 2 ** 20, "h2d_s": copy_s,
                       "encode_ms": tab_ms[0], "decode_ms": "no equivalent", "same_bytes": same}}


def pool(rng, n):
    """Word-salad text like tests/golden/make_golden.py's synth_bytes, generated with numpy."""
    letters = np.frombuffer(b"abcdefghijklmnopqrstuvwxyz", dtype=np.uint8)
    words = [letters[rng.integers(0, 26, rng.integers(2, 10))].tobytes() for _ in range(200)]
    seps = [b" ", b".\n"]
    k = n // 5 + 16
    idx, sep = rng.integers(0, 200, k), (rng.random(k) >= 0.85).astype(int)
    text = b"".join(words[i] + seps[j] for i, j in zip(idx.tolist(), sep.tolist()))
    return np.frombuffer(text[:n], dtype=np.uint8)


def batch(S, reps, rng, name, prec):
    text = pool(rng, 16 << 20)
    offs = rng.integers(0, len(text) - N, S)
    host = np.stack([text[o:o + N] for o in offs]).astype(np.int32)
    syms = torch.from_numpy(host).cuda()
    cap = N + N // 2
    enc = coder.StreamEncoder(S, prec=prec, capacity_bytes=cap)
    counts = coder.Counts(S, 256)
    encode = enc.acs_encode_adaptive if name == "acs" else enc.encode_adaptive
    fin = "safe" if name == "acs" else True

    def prep_enc():
        enc.reset()
        counts.reset()

    enc_ms = timed(lambda: encode(syms, counts, finish=fin), prep_enc, reps)
    streams, nbits = enc.bitstreams()
    del enc
    dec = coder.StreamDecoder(streams, prec=prec)
    dcounts = coder.Counts(S, 256)
    decode = dec.acs_decode_adaptive if name == "acs" else dec.decode_adaptive
    out = {}

    def prep_dec():
        dec.reset(streams)
        dcounts.reset()

    def run_dec():
        out["syms"] = decode(dcounts, N, check_status=False)

    dec_ms = timed(run_dec, prep_dec, reps)
    lossless = bool(torch.equal(out["syms"], syms)) and bool(torch.equal(dcounts.counts, counts.counts))
    nbytes = S * N
    return {"prec": prec, "encode_ms": enc_ms[0], "encode_ms_min": enc_ms[1], "decode_ms": dec_ms[0],
            "decode_ms_min": dec_ms[1], "encode_bytes_per_s": nbytes / (enc_ms[0] / 1e3),
            "decode_bytes_per_s": nbytes / (dec_ms[0] / 1e3), "ratio": float(nbits.sum() / 8 / nbytes),
            "lossless": lossless}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("adaptive_bench.py needs a GPU")
    torch.cuda.set_device(0)
    rng = np.random.default_rng(2026)
    res = {"tool": "adaptive_bench", "card": card(), "config0": config0(args.reps),
           "batch": {"streams": args.streams, "bytes_per_stream": N, "vocab": 256,
                     "ac": batch(args.streams, args.reps, rng, "ac", 32),
                     "acs": batch(args.streams, args.reps, rng, "acs", 48)}}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
