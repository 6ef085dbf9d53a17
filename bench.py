#!/usr/bin/env python
"""bench.py -- coded tokens/s (encode + decode) of the arithmetic-coding hot path.

Workload (BASELINE.json configs[1]): coder-only sweep, precomputed random fp32 logits, vocab
32000, 1024 streams x 2048 tokens, encode + decode on one B200.  One step = the WHOLE job: lac_enc_init once,
128 slices of [1024 streams x 16 tokens] through lac_ac_encode_logits_f32 with the coder state carried, one flush;
then lac_dec_init once and 128 slices through lac_ac_decode_logits_f32; the decoded symbols are compared.  The
268 GB of logits of a whole job do not fit in HBM, so every slice reads the same resident 2.1 GB buffer (far larger
than the 126 MB L2) with its own symbols.  A second timed block repeats the measurement at vocab 128256 (the
north-star's target shape) with its own clock record: roofline.v128256.

  python bench.py --gpus N --steps K --warmup W           # this repo, device-resident `value` + host `e2e`
  python bench.py --impl reference ...                    # the reference's CPU algorithm (oracle port)
  python bench.py --workload llama --model 1b|8b ...      # configs[2] / [3]: model in the loop, sharded, one LACB file
  python bench.py --workload stress                       # configs[4]: 8192 streams x vocab 128256, per-token decode
  python bench.py --dump-outputs DIR ...                  # also the last step's streams and symbols as DIR/*.npy

Under torchrun every rank codes its own 1024 streams (independent chunks shard with no
data-path collective); the only collective is ONE gather of per-stream bit lengths per job.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

VOCAB = 32000
STREAMS = 1024
CHUNK_TOKENS = 2048
SLICE = 16
PREC = 48
METRIC = "coded_tokens_per_s_enc_dec"
UNIT = "tokens/s"


def workload_config(n_gpus):
    return {
        "workload": f"coder-only sweep: precomputed random fp32 logits, vocab {VOCAB}, {STREAMS} streams x "
                    f"{CHUNK_TOKENS} tokens, encode+decode",
        "vocab": VOCAB,
        "streams_per_gpu": STREAMS,
        "tokens_per_stream": CHUNK_TOKENS,
        "step": f"one full job: {STREAMS} streams x {CHUNK_TOKENS} tokens encoded, then decoded, as {CHUNK_TOKENS // SLICE} "
                f"slices of [{STREAMS} x {SLICE}] with the coder state carried (init once, flush once)",
        "prec": PREC,
        "l2": f"inputs larger than L2: {STREAMS * SLICE * VOCAB * 4 / 1e9:.2f} GB of logits per slice vs 126 MB "
              f"(the {STREAMS * CHUNK_TOKENS * VOCAB * 4 / 1e9:.0f} GB of a whole job do not fit in HBM: every slice reads the "
              "same resident buffer with its own symbols)",
        "parallelism": f"chunk-sharded x{n_gpus}, no data-path collective",
    }


def measured_traffic(kernel, vocab, rows):
    """DRAM bytes per launch from the committed ncu capture, if it is for this exact workload; else None."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r2", "traffic.json")))[kernel]
        return t["dram_bytes"] if (t["vocab"], t["rows"]) == (vocab, rows) else None
    except Exception:
        return None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------ clocks sampler
class Clocks:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------ CPU legs (oracle; checker / baseline only)
def cpu_sample(streams, T, seed=1):
    rng = np.random.default_rng(seed)
    logits = (rng.standard_normal((streams, T, VOCAB)) * 3.0).astype(np.float32)
    syms = rng.integers(0, VOCAB, (streams, T)).astype(np.int32)
    return logits, syms


def cpu_baseline_leg(target_seconds=12.0):
    """Reference algorithm (llama_compress.calc_dist + arith_code A_to_bin / A_from_bin with fudged_dist),
    C port in oracle/, all host threads, on a bounded sample of the same workload (the sample is coded
    repeatedly until ~target_seconds of wall time have been spent)."""
    from oracle import oracle as orc
    cores = orc.num_threads()
    T = 16
    streams = max(cores * 4, 64)
    lg, sy = cpu_sample(streams, T, seed=3)
    orc.ref_roundtrip_bulk(lg[:cores], sy[:cores], prec=PREC)  # warm-up (page in, spawn once)
    reps, dt, bits = 0, 0.0, 0
    t0 = time.perf_counter()
    while dt < target_seconds and reps < 1000:
        bad, bits = orc.ref_roundtrip_bulk(lg, sy, prec=PREC)
        assert bad == 0, "reference port failed to round-trip"
        reps += 1
        dt = time.perf_counter() - t0
    return {"value": streams * T * reps / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{streams} streams x {T} tokens, vocab {VOCAB}, encode+decode, coded {reps}x in {dt:.1f} s; "
                      "C port of llama_compress.calc_dist + arith_code (fudged_dist per token), pthreads",
            "bits_per_token": bits / (streams * T)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as orc
    cores = orc.num_threads()
    streams, T = cores * 8, 16
    lg, sy = cpu_sample(streams, T, seed=4)
    for _ in range(args.warmup):
        orc.ref_roundtrip_bulk(lg, sy, prec=PREC)
    t0 = time.perf_counter()
    bits = 0
    for _ in range(args.steps):
        bad, b = orc.ref_roundtrip_bulk(lg, sy, prec=PREC)
        assert bad == 0
        bits += b
    dt = time.perf_counter() - t0
    val = streams * T * args.steps / dt
    sample = f"each step {streams} streams x {T} tokens, vocab {VOCAB}, encode+decode (bounded sample of the workload)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32/f64/bigint", "data": "synthetic", "config": workload_config(args.gpus),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "bits_per_token": bits / (streams * T * args.steps), "gpu_launches": 0,
    }))


# ------------------------------------------------------------------ GPU legs
def pin_to_gpu_numa_node(gpu_index):
    """Run this rank on the CPU cores next to its GPU (NVML's affinity mask), so that the pinned host buffers of the
    e2e leg are first-touched on that GPU's NUMA node: with several ranks per box the host-to-device copies otherwise
    cross the socket interconnect.  Best effort; returns the number of cores or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


class Job:
    """One full coder job on one GPU: S streams x CHUNK tokens coded as CHUNK / SLICE slices with the coder state
    carried from slice to slice (lac_enc_init once, finish once, lac_dec_init once).  The logits of a full job
    (S x CHUNK x V fp32 = 268 GB at configs[1]) do not fit in HBM, so every slice reads the same resident
    [S, SLICE, V] buffer (2.1 GB >> L2) with its own symbols."""

    def __init__(self, L, ffi, torch, dev, S, T, V, chunk_tokens, seed):
        self.L, self.ffi, self.torch = L, ffi, torch
        self.S, self.T, self.V, self.n_slices = S, T, V, chunk_tokens // T
        self.rows = S * T
        self.cap = chunk_tokens * 8 + 64
        gen = torch.Generator(device=dev).manual_seed(seed)
        self.logits = torch.randn((S, T, V), generator=gen, device=dev) * 3.0
        # symbols drawn from the model distribution (what an LLM coder sees on in-distribution text):
        # n_slices independent draws per logits row, slice k uses draw k
        probs = torch.softmax(self.logits.view(self.rows, V), -1)
        draws = torch.multinomial(probs, self.n_slices, replacement=True, generator=gen)  # [rows, n_slices]
        del probs
        self.syms = draws.t().contiguous().view(self.n_slices, S, T).to(torch.int32)       # slice-major
        self.back = torch.zeros_like(self.syms)
        self.enc_state = torch.zeros((S, ffi.ENC_STATE_BYTES), dtype=torch.uint8, device=dev)
        self.dec_state = torch.zeros((S, ffi.DEC_STATE_BYTES), dtype=torch.uint8, device=dev)
        self.out = torch.zeros((S, self.cap), dtype=torch.uint8, device=dev)
        self.offsets = torch.arange(S + 1, device=dev, dtype=torch.int64) * self.cap
        self.ws_bytes = int(L.lac_workspace_bytes(self.rows, V))     # caller-provided scratch: no allocation per call
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=dev)
        self.stream = torch.cuda.current_stream().cuda_stream
        # kernels per job: enc_init + n x (summary, pair, encode_pairs) + dec_init + n x (summary, decode_serial)
        # (slices of <= 4 tokens: summary + one fused encoder kernel)
        self.launches = 2 + (5 if T > 4 else 4) * self.n_slices

    def encode(self, ev=None):
        L, ck, S, T, V, st = self.L, self.ffi.check, self.S, self.T, self.V, self.stream
        ck(L.lac_enc_init(self.enc_state.data_ptr(), S, PREC, st))
        for k in range(self.n_slices):
            if ev is not None: ev[k][0].record()
            # summary pass (fused softmax -> quantise -> clamp -> segment sums, one HBM pass over the logits), then
            # (lo, hi) of the coded symbols (one warp per row) and the range coder (one thread per stream)
            ck(L.lac_ac_encode_logits_f32(self.logits.data_ptr(), S, T, T * V, V, V, self.syms[k].data_ptr(), T, None,
                                          self.enc_state.data_ptr(), self.out.data_ptr(), self.cap,
                                          int(k == self.n_slices - 1), PREC, self.ws.data_ptr(), self.ws_bytes, st))
            if ev is not None: ev[k][1].record()

    def decode(self, ev=None):
        L, ck, S, T, V, st = self.L, self.ffi.check, self.S, self.T, self.V, self.stream
        ck(L.lac_dec_init(self.dec_state.data_ptr(), S, PREC, self.out.data_ptr(), self.offsets.data_ptr(), st))
        for k in range(self.n_slices):
            if ev is not None: ev[k][2].record()
            # row summaries from the same logits (bandwidth-bound pass), then the serial pass per stream
            ck(L.lac_ac_decode_logits_f32(self.logits.data_ptr(), S, T, T * V, V, V, None,
                                          self.dec_state.data_ptr(), self.out.data_ptr(), self.offsets.data_ptr(),
                                          self.back[k].data_ptr(), T, PREC, self.ws.data_ptr(), self.ws_bytes, st))
            if ev is not None: ev[k][3].record()

    def nbits(self):
        return self.enc_state.view(self.torch.int64).view(self.S, 4)[:, 2]

    def check(self):
        assert self.torch.equal(self.back, self.syms), "round trip failed"
        st = self.enc_state.view(self.torch.int32).view(self.S, 8)[:, 6]
        assert int(st.max().item()) == 0, "encoder status set"
        st = self.dec_state.view(self.torch.int32).view(self.S, 10)[:, 8]
        assert int(st.max().item()) == 0, "decoder status set"

    def events(self):
        E = self.torch.cuda.Event
        return [[E(enable_timing=True) for _ in range(4)] for _ in range(self.n_slices)]

    @staticmethod
    def slice_times(evs_list):
        """mean ms per slice of (encode call, decode call) over the recorded jobs"""
        enc = statistics.mean(e[0].elapsed_time(e[1]) for evs in evs_list for e in evs)
        dec = statistics.mean(e[2].elapsed_time(e[3]) for evs in evs_list for e in evs)
        return enc, dec


DUMP_BYTES = 64 * 10**6 - 4096   # everything --dump-outputs writes, npy headers included


def dump_outputs(path, job):
    """What the caller of the timed path received in the last step, as path/<name>.npy, so that two builds can be
    compared output for output: nbits (bits coded per stream), stream_bytes (each stream's ceil(nbits / 8) coded
    bytes, concatenated in stream order), symbols (the decoded tokens, [streams, tokens]) and stream_index (the
    streams written: all of them, or a fixed seeded sample of whole streams where all would exceed 64 MB)."""
    nbits = job.nbits().cpu().numpy()
    nbytes = (nbits + 7) // 8
    tokens = job.n_slices * job.T
    cost = 4 * nbytes + 4 * tokens + 8 + 8
    order = np.random.default_rng(0).permutation(job.S)
    keep = np.sort(order[:int(np.searchsorted(np.cumsum(cost[order]), DUMP_BYTES, side="right"))])
    out = job.out.cpu().numpy()
    symbols = job.back.permute(1, 0, 2).reshape(job.S, tokens).cpu().numpy()
    arrays = {"stream_index": keep.astype(np.float64), "nbits": nbits[keep].astype(np.float64),
              "stream_bytes": np.concatenate([out[s, :nbytes[s]] for s in keep]).astype(np.float32),
              "symbols": symbols[keep].astype(np.float32)}
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


def roofline_numbers(rows, V, encode_ms, decode_ms):
    """algorithmic bytes of one call (the logits once, one symbol per row) and the two achieved GB/s figures"""
    alg = rows * (V * 4 + 4)
    return alg, alg / (encode_ms * 1e-3) / 1e9, alg / (decode_ms * 1e-3) / 1e9


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from lac_b200 import _ffi
    L = _ffi.lib()  # raises if the CUDA library is missing: there is no fallback

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cores = pin_to_gpu_numa_node(local) if world > 1 else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    S, T, V = STREAMS, SLICE, VOCAB
    job = Job(L, _ffi, torch, dev, S, T, V, CHUNK_TOKENS, 1234 + rank)
    rows = job.rows
    gathered = torch.zeros((world, S), dtype=torch.int64, device=dev) if world > 1 else None

    def step(ev=None):
        job.encode(ev)
        if world > 1:  # the one collective of a job: per-stream bit lengths for the container index
            dist.all_gather_into_tensor(gathered.view(-1), job.nbits().contiguous())
        job.decode(ev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step()
    torch.cuda.synchronize()
    job.check()
    tokens_per_job = S * CHUNK_TOKENS
    bits_per_token = float(job.nbits().sum().item()) / tokens_per_job

    clocks = Clocks(local)
    if rank == 0:
        clocks.start()
        time.sleep(0.3)
    n_ev = min(args.steps, 4)  # per-slice CUDA events on the first few jobs (the kernels' own times)
    evs = [job.events() for _ in range(n_ev)]
    t_beg, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_beg.record()
    for k in range(args.steps):
        step(evs[k] if k < n_ev else None)
    t_end.record()
    barrier()
    elapsed_ms = t_beg.elapsed_time(t_end)
    if world > 1:
        t = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    clk = clocks.stop() if rank == 0 else None
    job.check()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, job)
    encode_ms, decode_ms = Job.slice_times(evs)

    # ---------------- the north-star target shape: vocab 128256 (configs[3] / [4]), same 2.1 GB per slice
    v128 = None
    if rank == 0 and not args.no_v128 and V != 128256:
        V2, S2 = 128256, 256
        job2 = Job(L, _ffi, torch, dev, S2, T, V2, args.v128_tokens, 99)
        for _ in range(3):
            job2.encode(); job2.decode()
        torch.cuda.synchronize()
        job2.check()
        clocks2 = Clocks(local)
        clocks2.start()
        time.sleep(0.3)
        evs2 = [job2.events() for _ in range(min(4, args.v128_jobs))]
        b2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        b2.record()
        for j in range(args.v128_jobs):
            ev = evs2[j] if j < len(evs2) else None
            job2.encode(ev); job2.decode(ev)
        e2.record()
        torch.cuda.synchronize()
        ms2 = b2.elapsed_time(e2)
        clk2 = clocks2.stop()
        job2.check()
        l2, d2 = Job.slice_times(evs2)
        peak, _ = peaks()
        alg2, lg2, dg2 = roofline_numbers(job2.rows, V2, l2, d2)
        v128 = {"workload": f"vocab {V2}, {S2} streams x {args.v128_tokens} tokens in slices of {T}, encode+decode, "
                            f"{job2.rows * V2 * 4 / 1e9:.2f} GB of logits per slice",
                "encode": {"ms": l2, "achieved": lg2, "frac": lg2 / peak, "algorithmic_bytes_per_call": alg2},
                "decode": {"ms": d2, "achieved": dg2, "frac": dg2 / peak},
                "tokens_per_s": S2 * args.v128_tokens * args.v128_jobs / (ms2 * 1e-3),
                "jobs": args.v128_jobs, "ms_total": ms2, "clocks": clk2,
                "bits_per_token": float(job2.nbits().sum().item()) / (S2 * args.v128_tokens)}
        del job2
        torch.cuda.empty_cache()

    # ---------------- e2e: HOST buffers through the C ABI, copies inside the timed region
    e2e = None
    if not args.no_e2e:
        cap = T * 8 + 64
        e_steps = max(2, min(args.steps, args.e2e_steps))
        h_logits = torch.empty((S, T, V), dtype=torch.float32).pin_memory()
        h_logits.copy_(job.logits)
        h_syms = job.syms[0].cpu().pin_memory()
        h_out = torch.zeros((S, cap), dtype=torch.uint8).pin_memory()
        h_nbits = torch.zeros(S, dtype=torch.int64).pin_memory()
        h_back = torch.zeros((S, T), dtype=torch.int32).pin_memory()
        h_offs = (torch.arange(S + 1, dtype=torch.int64) * cap)
        ck = _ffi.check

        def host_step():
            ck(L.lac_encode_logits_host(h_logits.data_ptr(), h_syms.data_ptr(), S, T, V, h_out.data_ptr(), cap,
                                        h_nbits.data_ptr(), PREC))
            ck(L.lac_decode_logits_host(h_logits.data_ptr(), S, T, V, h_out.data_ptr(), h_offs.data_ptr(),
                                        h_back.data_ptr(), PREC))
        host_step()
        assert torch.equal(h_back, h_syms), "host-API round trip failed"
        barrier()
        t0 = time.perf_counter()
        for _ in range(e_steps):
            host_step()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        h2d = 2 * rows * V * 4 + rows * 4 + S * cap + (S + 1) * 8
        d2h = S * cap + S * _ffi.ENC_STATE_BYTES + rows * 4
        e2e = {"value": world * rows * e_steps / dt, "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "steps": e_steps, "ms_per_step": dt / e_steps * 1e3,
               "step": f"one [{S} x {T}] slice of the job, host logits in, host bytes / symbols out",
               "bound": "pcie", "h2d_gbps": h2d * e_steps / dt / 1e9, "cores_near_gpu": numa_cores,
               "api": "lac_encode_logits_host + lac_decode_logits_host (pinned host logits in, host bytes/symbols out)"}

    if rank == 0:
        peak, peak_src = peaks()
        alg_bytes, enc_gbs, dec_gbs = roofline_numbers(rows, V, encode_ms, decode_ms)
        line = {
            "metric": METRIC, "value": world * tokens_per_job * args.steps / (elapsed_ms * 1e-3), "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32->u32/u64", "data": "synthetic", "config": workload_config(world),
            "roofline": {"bound": "hbm",
                         "kernel": "summary_kernel (fused softmax -> fixed-total quantisation -> min-frequency clamp -> "
                                   "segment prefix sums; the one HBM pass over the logits), timed through the whole "
                                   "lac_ac_encode_logits_f32 call, i.e. together with pair_kernel (symbol ranges) and "
                                   "encode_pairs_staged_kernel (range coder); the ncu launch list under profiles/ gives the split",
                         "achieved": enc_gbs, "peak": peak, "unit": "GB/s", "frac": enc_gbs / peak,
                         "traffic": measured_traffic("summary_kernel", V, rows), "peak_source": peak_src,
                         "peak_note": "the peak is the copy-measured (read + write) figure; a read-only stream reaches 7.2-7.8 TB/s on this part (profiles/microbench/tma_stream_b200.txt), so frac may exceed 1",
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "ms_per_launch": encode_ms,
                         "decode": {"kernels": "summary_kernel + decode_serial_kernel (lac_ac_decode_logits_f32)",
                                    "achieved": dec_gbs, "frac": dec_gbs / peak, "ms_per_call": decode_ms},
                         "timed_over": f"{n_ev} jobs x {job.n_slices} slices, CUDA events around every call",
                         "v128256": v128},
            "e2e": e2e, "gpu_launches": job.launches * args.steps, "clocks": clk,
            "bits_per_token": bits_per_token,
        }
        if world == 1 and not args.no_cpu:
            cb = cpu_baseline_leg()
            line["cpu_baseline"] = cb
            line["bits_per_token_reference_literal"] = cb["bits_per_token"]
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------ model-in-the-loop workloads (configs[2..4])
def _dist_setup():
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    return rank, world, local, dev


def _timed(fn, dev, world):
    """fn() bracketed by barrier + synchronize on both sides; seconds, max over ranks."""
    import torch
    import torch.distributed as dist
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([dt], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    return out, dt


def _step_split(engine, bucket, reps=20):
    """ms per token step at one attention bucket: model forward alone vs the whole encode / decode step (model +
    LQ32 summary + coder kernels), each replayed from its own CUDA graph and timed with CUDA events."""
    import torch
    from lac_b200 import coder, llama_compress as lc
    m = engine.m
    S, dev = m.S, m.device
    if engine.enc is None:
        engine.enc = coder.StreamEncoder(S, prec=engine.prec, capacity_bytes=engine.cap, device=dev)
    engine.enc.reset()
    enc = engine.enc
    engine.ntok.fill_(engine.T)
    res = {}
    prev = torch.full((S,), lc.BOS, dtype=torch.int64, device=dev)

    def model_only():
        m.step(prev, bucket)

    def enc_step():
        engine._enc_step(bucket)
        m.pos.sub_(1)

    st = torch.cuda.Stream(device=dev)
    st.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(st):
        for name, fn in (("model_ms", model_only), ("encode_step_ms", enc_step)):
            m.reset()
            fn()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=st):
                fn()
            for _ in range(3):
                g.replay()
            b, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b.record(st)
            for _ in range(reps):
                g.replay()
            e.record(st)
            e.synchronize()
            res[name] = b.elapsed_time(e) / reps
            if name == "encode_step_ms":
                enc.reset()
    torch.cuda.current_stream(dev).wait_stream(st)
    torch.cuda.synchronize()
    enc.reset()   # the replays above coded the same token over and over: start from clean streams
    res["coder_share_of_encode_step"] = max(0.0, 1.0 - res["model_ms"] / res["encode_step_ms"])
    res["bucket"] = bucket
    return res


def run_llama(args):
    """configs[2] / configs[3]: the llama_compress.py path.  Synthetic text (uniform random token ids), random-init
    weights of the named geometry, chunks of --chunk-tokens tokens coded in model batches of --batch-streams
    streams, batches sharded over the ranks, ONE gather of the index and one of the payload into a LACB file on
    rank 0, then decompressed the same way and compared."""
    import torch
    import torch.distributed as dist
    from lac_b200 import container, llama_compress as lc
    rank, world, local, dev = _dist_setup()
    cfg = lc.CONFIGS[args.model]
    n_tokens = int(args.text_mb * (1 << 20) / 4)          # ~4 bytes of text per token
    if args.tokens:
        n_tokens = args.tokens
    rng = np.random.default_rng(2024)
    toks = rng.integers(0, cfg.vocab, n_tokens).astype(np.int32)
    model = lc.LlamaModel(cfg, n_streams=args.batch_streams, max_len=args.chunk_tokens, seed=0, device=dev)
    comp = lc.LlamaCompressor(model, chunk_tokens=args.chunk_tokens, use_graphs=not args.no_graphs)
    # warm-up: one short job (captures every attention bucket's graphs in both directions)
    wtoks = toks[: args.batch_streams * args.chunk_tokens * world]
    wb = comp.compress(wtoks[: args.chunk_tokens * world * 2] if args.quick_warmup else wtoks)
    if world > 1:
        box = [wb]
        dist.broadcast_object_list(box, src=0)
        wb = box[0]
    comp.decompress(wb)
    clocks = Clocks(local)
    if rank == 0:
        clocks.start()
    blob, t_enc = _timed(lambda: comp.compress(toks), dev, world)
    if world > 1:
        box = [blob]
        dist.broadcast_object_list(box, src=0)
        blob = box[0]
    back, t_dec = _timed(lambda: comp.decompress(blob), dev, world)
    clk = clocks.stop() if rank == 0 else None
    split = _step_split(comp.engine, lc._bucket_for(args.chunk_tokens // 2, args.chunk_tokens)) if rank == 0 else None
    if rank == 0:
        assert np.array_equal(back, toks), "llama path did not round-trip"
        c = container.unpack(blob)
        n_chunks = c.n_chunks
        line = {
            "workload": "llama", "metric": METRIC, "value": n_tokens / (t_enc + t_dec), "unit": UNIT, "n_gpus": world,
            "higher_is_better": True, "scaling": "strong", "data": "synthetic (uniform random token ids)",
            "dtype": "bf16 model forward, f32 logits -> u32/u64 coder",
            "config": {"workload": f"llama_compress path, {cfg.name} random-init model ({cfg.params / 1e9:.2f} B parameters, "
                                   f"vocab {cfg.vocab}), {n_tokens} tokens (~{n_tokens * 4 / (1 << 20):.0f} MB of text) in "
                                   f"{args.chunk_tokens}-token chunks, model batches of {args.batch_streams} streams sharded over "
                                   f"{world} GPU(s), one LACB file",
                       "model": cfg.describe(), "chunks": n_chunks, "batch_streams": args.batch_streams,
                       "cuda_graphs": not args.no_graphs},
            "encode_tokens_per_s": n_tokens / t_enc, "decode_tokens_per_s": n_tokens / t_dec,
            "encode_s": t_enc, "decode_s": t_dec, "lossless": True,
            "bits_per_token": float(c.nbits.sum()) / max(n_tokens, 1), "container_bytes": len(blob),
            "step_split": split, "clocks": clk,
            # this workload IS end to end: host token ids in, LACB bytes out (and back); the logits never leave the GPU
            "e2e": {"value": n_tokens / (t_enc + t_dec), "unit": UNIT, "h2d_bytes_per_step": 4 * n_tokens + len(blob),
                    "d2h_bytes_per_step": len(blob) + 4 * n_tokens,
                    "api": "LlamaCompressor.compress(tokens) -> bytes, LlamaCompressor.decompress(bytes) -> tokens"},
            "collectives": "one all_gather of (tokens, bits) per chunk + one all_gather of the payload per job; none in the coding loop",
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_stress(args):
    """configs[4]: decode-heavy stress -- --streams concurrent streams (default 8192), vocab 128256, sequential
    per-token decode with the model in the loop, lossless round trip verified."""
    import torch
    from lac_b200 import llama_compress as lc
    rank, world, local, dev = _dist_setup()
    cfg = lc.CONFIGS[args.model]
    S, T = args.stress_streams, args.stress_tokens
    rng = np.random.default_rng(7 + rank)
    toks = rng.integers(0, cfg.vocab, (S, T)).astype(np.int32)
    ntok = np.full(S, T, dtype=np.int32)
    model = lc.LlamaModel(cfg, n_streams=S, max_len=T, seed=0, device=dev)
    eng = lc.StepEngine(model, T, PREC, use_graphs=not args.no_graphs)
    eng.encode_batch(toks[:, :T], ntok)                      # warm-up (graph capture) + the streams to decode
    (streams, nbits), t_enc = _timed(lambda: eng.encode_batch(toks, ntok), dev, world)
    eng.decode_batch(streams, ntok)                          # warm-up (graph capture)
    clocks = Clocks(local)
    if rank == 0:
        clocks.start()
    back, t_dec = _timed(lambda: eng.decode_batch(streams, ntok), dev, world)
    clk = clocks.stop() if rank == 0 else None
    assert np.array_equal(back, toks), "stress decode did not round-trip"
    # per-step latency of the decoder call alone (summary pass + serial pass) on this shape, CUDA events
    from lac_b200 import _ffi, coder
    L = _ffi.lib()
    logits = torch.randn((S, 1, cfg.vocab), device=dev) * 3.0
    dec = coder.StreamDecoder(streams, prec=PREC, device=dev)
    out = torch.zeros((S, 1), dtype=torch.int32, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    reps = 20
    for k in range(reps + 3):
        if k == 3:
            ev[0].record()
        _ffi.check(L.lac_ac_decode_logits_f32(logits.data_ptr(), S, 1, cfg.vocab, cfg.vocab, cfg.vocab, None,
                                              dec.state.data_ptr(), dec.bytes.data_ptr(), dec.offsets.data_ptr(),
                                              out.data_ptr(), 1, PREC, eng.ws.ptr, eng.ws.nbytes, st))
    ev[1].record()
    torch.cuda.synchronize()
    dec_call_ms = ev[0].elapsed_time(ev[1]) / reps
    peak, _ = peaks()
    if rank == 0:
        line = {
            "workload": "stress", "metric": "decoded_tokens_per_s", "value": world * S * T / t_dec, "unit": UNIT,
            "n_gpus": world, "higher_is_better": True, "scaling": "weak", "data": "synthetic (uniform random token ids)",
            "config": {"workload": f"decode-heavy stress: {S} concurrent streams x {T} tokens, vocab {cfg.vocab}, sequential "
                                   f"per-token decode with the {cfg.name} model in the loop, lossless round trip verified",
                       "model": cfg.describe(), "cuda_graphs": not args.no_graphs},
            "decode_s": t_dec, "encode_s": t_enc, "ms_per_token_step": t_dec / T * 1e3, "lossless": True,
            "bits_per_token": float(np.sum(nbits)) / (S * T),
            "decoder_call": {"api": "lac_ac_decode_logits_f32, T = 1", "ms": dec_call_ms,
                             "logits_bytes": S * cfg.vocab * 4,
                             "achieved_gbs": S * cfg.vocab * 4 / (dec_call_ms * 1e-3) / 1e9,
                             "frac_of_measured_hbm_peak": S * cfg.vocab * 4 / (dec_call_ms * 1e-3) / 1e9 / peak},
            "clocks": clk,
        }
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="lac_b200", choices=["lac_b200", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=4)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the coded streams and decoded symbols of the last timed step (rank 0's) to DIR/*.npy")
    # measurement switches (the driver's contract run uses the defaults = BASELINE.json configs[1])
    ap.add_argument("--vocab", type=int, default=VOCAB)
    ap.add_argument("--streams", type=int, default=STREAMS)
    ap.add_argument("--slice", type=int, default=SLICE)
    ap.add_argument("--chunk-tokens", type=int, default=CHUNK_TOKENS)
    ap.add_argument("--no-v128", action="store_true")
    ap.add_argument("--v128-tokens", type=int, default=256)
    ap.add_argument("--v128-jobs", type=int, default=100)
    # model-in-the-loop workloads (extra lines, not the driver's headline): configs[2] / [3] / [4]
    ap.add_argument("--workload", default="coder", choices=["coder", "llama", "stress"])
    ap.add_argument("--model", default="1b", help="lac_b200.llama_compress.CONFIGS key: tiny, 1b, 8b, 1b-128k")
    ap.add_argument("--text-mb", type=float, default=16.0)
    ap.add_argument("--tokens", type=int, default=0, help="override the token count derived from --text-mb")
    ap.add_argument("--batch-streams", type=int, default=256)
    ap.add_argument("--no-graphs", action="store_true")
    ap.add_argument("--quick-warmup", action="store_true")
    ap.add_argument("--stress-streams", type=int, default=8192)
    ap.add_argument("--stress-tokens", type=int, default=64)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl, args.workload) != ("lac_b200", "coder"):
        ap.error("--dump-outputs writes the outputs of the coder workload of lac_b200")
    globals().update(VOCAB=args.vocab, STREAMS=args.streams, SLICE=args.slice, CHUNK_TOKENS=args.chunk_tokens)
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "llama":
        run_llama(args)
    elif args.workload == "stress":
        run_stress(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
