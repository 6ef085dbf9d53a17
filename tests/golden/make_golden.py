"""Generate golden vectors by RUNNING the real reference (pramasoul/lac).

Run in the build container only (the GPU box has no /root/reference):

    python tests/golden/make_golden.py

Writes tests/golden/*.npz.  Everything stored is either an input or an output of the
unmodified reference code imported from /root/reference; nothing comes from oracle/ or
lac_b200/.  tests/test_oracle_golden.py then pins oracle/lac_oracle.c to these files.
"""
import os
import random
import sys
import warnings

import numpy as np

REF = os.environ.get("LAC_REFERENCE", "/root/reference")
sys.path.insert(0, REF)
warnings.simplefilter("ignore")

import arith_code as ac  # noqa: E402
import arithmetic_coding as acs  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


# ---------------------------------------------------------------- helpers
class TablePredictor(ac.CDFPredictor):
    """CDFPredictor whose table changes per accepted symbol (reference classes untouched)."""

    def __init__(self, tables):
        self.tables = tables
        self.k = 0

    @property
    def dist(self):
        return self.tables[min(self.k, len(self.tables) - 1)]

    @property
    def minp(self):
        return min(filter(lambda v: v > 0, self.pdf_iter))

    def accept(self, symbol):
        self.k += 1

    def copy(self):
        return TablePredictor(self.tables)


def run_decoder(coder, bits, stop):
    """list(from_bin.run(bits, stop)) but keeping what came out before an exception."""
    out, err = [], ""
    try:
        for s in coder.from_bin.run(bits, stop):
            out.append(int(s))
    except Exception as e:  # AssertionError / ValueError / ZeroDivisionError in the reference
        err = type(e).__name__
    return out, err


def pack_case(store, name, **kw):
    for k, v in kw.items():
        store[f"{name}/{k}"] = np.asarray(v)


def save_by_field(path, store, names):
    """One array per field instead of one per case and field (an npz pays ~200 bytes per member): a scalar field
    holds one value per case, an array field the cases' arrays concatenated, split at '<field>_off'.
    tests/conftest.py reads it back keyed '<case>/<field>'."""
    out = {"names": np.array(names)}
    for f in sorted({k.split("/", 1)[1] for k in store if "/" in k}):
        vals = [store[f"{nm}/{f}"] for nm in names]
        if vals[0].ndim == 0:
            out[f] = np.array(vals)
        else:
            out[f] = np.concatenate(vals)
            out[f"{f}_off"] = np.cumsum([0] + [len(v) for v in vals]).astype(np.int64)
    np.savez_compressed(path, **out)


# ---------------------------------------------------------------- arith_code: shared small tables
def gen_ac_small(rng):
    store, names = {}, []
    cfgs = []
    for prec in (8, 12, 16, 24, 32, 48):
        for V in (2, 3, 5, 17, 64):
            cfgs.append((prec, V))
    for ci, (prec, V) in enumerate(cfgs):
        if V >= (1 << (prec - 2)):
            continue
        for style in ("flat", "skew", "big"):
            if style == "flat":
                pdf = [1] * V
            elif style == "skew":
                pdf = [int(rng.integers(1, 40)) for _ in range(V)]
                pdf[int(rng.integers(0, V))] += 500
            else:  # totals above the coder width -> fudged_dist branch
                pdf = [int(rng.integers(0, 1 << 30)) for _ in range(V)]
                pdf[0] += 1
            dist = list(np.cumsum(np.array(pdf, dtype=object)))
            pred = ac.CDFPredictor(dist)
            coder = ac.AC(pred, prec)
            for n in (0, 1, 7, 60):
                p = np.array(pdf, dtype=np.float64) + 1e-9
                syms = [int(s) for s in rng.choice(V, size=n, p=p / p.sum())] if rng.random() < 0.5 \
                    else [int(s) for s in rng.integers(0, V, size=n)]
                if style == "big":
                    # zero-width symbols are unencodable in the unfudged branch only; fine when fudged
                    pass
                for stop in (0, 1):
                    try:
                        bits = [int(b) for b in coder.to_bin.bits(syms, stop)]
                        r, length = coder.to_bin.encode(syms, stop)
                    except Exception:
                        continue
                    assert length == len(bits)
                    assert all(b in (0, 1) for b in bits)
                    assert r == int("0" + "".join(map(str, bits)), 2)
                    dec, err = run_decoder(coder, bits, stop)
                    name = f"c{len(names)}"
                    names.append(name)
                    pack_case(store, name, prec=prec, dist=np.array(dist, dtype=np.int64),
                              minp=int(pred.minp), syms=np.array(syms, dtype=np.int32), stop=stop,
                              bits=np.array(bits, dtype=np.uint8), dec=np.array(dec, dtype=np.int32),
                              dec_err=err)
    save_by_field(os.path.join(HERE, "ac_small.npz"), store, names)
    print("ac_small:", len(names), "cases")


# ---------------------------------------------------------------- llama_compress.Llama_AC with a fake llm
class FakeLlm:
    """Stands in for llama_cpp.Llama: _scores[-1] is the logits row for the current position."""

    def __init__(self, logits, n_ctx=1 << 30):
        self.logits = logits
        self._n_ctx = n_ctx
        self.reset()

    def reset(self):
        self.pos = -1
        self._scores = None

    def eval(self, toks):
        self.pos += len(toks)
        k = min(self.pos, len(self.logits) - 1)
        self._scores = self.logits[k:k + 1]

    def n_ctx(self):
        return self._n_ctx


def load_llama_compress():
    # llama_compress.py does `from arith_code import *` and needs numpy only; llama_cpp is
    # imported lazily inside r(), which we never call.
    import importlib
    return importlib.import_module("llama_compress")


def gen_ac_llama(rng):
    lc = load_llama_compress()
    store, names = {}, []
    for V, T, scale in ((50, 40, 3.0), (300, 30, 6.0), (2000, 12, 4.0), (2000, 12, 12.0)):
        logits = (rng.standard_normal((T + 4, V)) * scale).astype(np.float32)
        syms = []
        for t in range(T):
            p = np.exp(logits[t].astype(np.float64) - logits[t].max())
            syms.append(int(rng.choice(V, p=p / p.sum())) if rng.random() < 0.8 else int(rng.integers(0, V)))
        enc_pred = lc.Llama_AC(FakeLlm(logits))
        coder = ac.AC(enc_pred, 48)
        bits = [int(b) for b in coder.to_bin.bits(syms, 1)]
        # tables the reference actually used, position by position
        tab_pred = lc.Llama_AC(FakeLlm(logits))
        tables, minps = [], []
        for t in range(T + 4):
            d = tab_pred.dist
            tables.append(np.array(d, dtype=np.int64))
            minps.append(int(tab_pred.minp))
            tab_pred.accept(syms[t] if t < T else 0)
        dec_pred = lc.Llama_AC(FakeLlm(logits))
        dec, err = [], ""
        try:
            for s in ac.AC(dec_pred, 48).from_bin.run(bits, 0):
                dec.append(int(s))
        except Exception as e:
            err = type(e).__name__
        name = f"l{len(names)}"
        names.append(name)
        pack_case(store, name, prec=48, logits=logits, tables=np.stack(tables), minp=np.array(minps, dtype=np.int64),
                  syms=np.array(syms, dtype=np.int32), bits=np.array(bits, dtype=np.uint8),
                  dec=np.array(dec, dtype=np.int32), dec_err=err)
        print("  llama case", name, "V", V, "T", T, "bits", len(bits), "dec", len(dec), err)
    store["names"] = np.array(names)
    np.savez_compressed(os.path.join(HERE, "ac_llama.npz"), **store)
    print("ac_llama:", len(names), "cases")


# ---------------------------------------------------------------- arith_code: adaptive count model over bytes
class AdaptiveCounts(ac.ProbPredictor):
    """'simple adaptive frequency model': prob(s) = 1 + occurrences of s so far."""

    def __init__(self, n, counts=None):
        super().__init__(n)
        self.counts = [0] * n if counts is None else counts

    def prob(self, symbol):
        return 1 + self.counts[symbol]

    def accept(self, symbol):
        self.counts[symbol] += 1
        return super().accept(symbol)

    def copy(self):
        return AdaptiveCounts(self.n, list(self.counts))


def synth_bytes(n, seed):
    r = random.Random(seed)
    words = [bytes(r.choice(b"abcdefghijklmnopqrstuvwxyz") for _ in range(r.randint(2, 9))) for _ in range(200)]
    out = bytearray()
    while len(out) < n:
        out += r.choice(words) + (b" " if r.random() < 0.85 else b".\n")
    return bytes(out[:n])


def gen_ac_adaptive():
    data = synth_bytes(16384, 7)
    coder = ac.AC(AdaptiveCounts(256), 32)
    comp = ac.measure_compress(coder.to_bin, list(data), print_every_out=10**9, print_every_inp=10**9)
    dec = []
    for s in coder.from_bin.run(ac.ungroup_bits(comp), 0):
        dec.append(s)
        if len(dec) == len(data):
            break
    assert bytes(dec) == data
    np.savez_compressed(os.path.join(HERE, "ac_adaptive.npz"), seed=7, n=len(data), prec=32,
                        data=np.frombuffer(data, dtype=np.uint8), comp=np.frombuffer(comp, dtype=np.uint8))
    print("ac_adaptive:", len(data), "->", len(comp), "bytes")


# ---------------------------------------------------------------- arithmetic_coding.ACSampler
def acs_encode(prec, cdfs, toks):
    s = acs.ACSampler(prec)
    out = []
    s.compress_tokens = toks
    s.compress_output = out.append

    def done():
        s.on_compress_done = None
        s.flush_compress()
        s.compress_output = None
    s.on_compress_done = done
    i = 0
    while not s.compress_done:
        s.sample_scaled_cdf(cdfs[min(i, len(cdfs) - 1)])
        i += 1
    return [int(b) for b in out]


def acs_decode(prec, cdfs, bits, n):
    s = acs.ACSampler(prec)
    s.decompress_bits = bits
    out, err = [], ""
    try:
        for i in range(n):
            out.append(int(s.sample_scaled_cdf(cdfs[i])))
    except Exception as e:
        err = type(e).__name__
    return out, err


def gen_acs(rng):
    store, names = {}, []
    for prec in (16, 32, 48):
        for V in (2, 3, 10, 50, 256):
            for conc in (0.3, 5.0):
                n = int(rng.integers(1, 50))
                pdfs = [rng.dirichlet(np.ones(V) * conc) for _ in range(n)]
                toks = [int(rng.choice(V, p=p)) for p in pdfs]
                cdfs = []
                for p in pdfs:
                    # ACSampler.sample's own expressions (arithmetic_coding.py:58-61), kept exact as ints
                    smp = acs.ACSampler(prec)
                    q = np.array(p, dtype=np.float64)
                    q += smp.get_lop_bias(q)
                    q *= smp.region.one / np.sum(q)
                    c = np.cumsum(q).astype(np.uint64)
                    cdfs.append(np.array([int(x) for x in c], dtype=object))
                try:
                    bits = acs_encode(prec, cdfs, toks)
                except AssertionError:
                    continue  # "cdf has unencodable token"
                dec, err = acs_decode(prec, cdfs, bits, n)
                name = f"s{len(names)}"
                names.append(name)
                pack_case(store, name, prec=prec, cdf=np.array([[int(x) for x in c] for c in cdfs], dtype=np.uint64),
                          toks=np.array(toks, dtype=np.int32), bits=np.array(bits, dtype=np.uint8),
                          dec=np.array(dec, dtype=np.int32), dec_err=err)
    store["names"] = np.array(names)
    np.savez_compressed(os.path.join(HERE, "acs_small.npz"), **store)
    print("acs_small:", len(names), "cases; reference decoder round-trips",
          sum(1 for nm in names if store[f"{nm}/dec_err"] == "" and
              np.array_equal(store[f"{nm}/dec"], store[f"{nm}/toks"])))


def gen_acs_64k():
    """BASELINE config[0]: 64 KB synthetic byte stream, simple adaptive frequency model, ACSampler."""
    data = synth_bytes(65536, 11)
    prec = 48
    counts = np.ones(256, dtype=object)
    s = acs.ACSampler(prec)
    out = bytearray()
    s.compress_tokens = list(data)
    s.compress_output = acs.packbits(out.append)

    def done():
        s.on_compress_done = None
        s.flush_compress()
        s.compress_output.flush()
        s.compress_output = None
    s.on_compress_done = done
    i = 0
    while not s.compress_done:
        cdf = np.cumsum(counts)  # exact Python ints (object dtype): integer-only adaptive model
        tok = s.sample_scaled_cdf(cdf)
        if i < len(data):
            counts[tok] += 1
        i += 1
    np.savez_compressed(os.path.join(HERE, "acs_64k.npz"), seed=11, n=len(data), prec=prec,
                        data=np.frombuffer(data, dtype=np.uint8), comp=np.frombuffer(bytes(out), dtype=np.uint8))
    print("acs_64k:", len(data), "->", len(out), "bytes")
# ---------------------------------------------------------------- arith_code: the uniform base class Predictor(n)
def gen_ac_uniform(rng):
    """AC(Predictor(n), prec) -- the reference's default coder is AC() = AC(ternary = Predictor(3), 16)."""
    store, names = {}, []
    for n in (2, 3, 5, 10, 256, 1000):
        for prec in (16, 24, 32, 48):
            if n >= (1 << (prec - 2)):
                continue
            coder = ac.AC(ac.Predictor(n), prec)
            for length in (0, 1, 7, 60, 300):
                syms = [int(s) for s in rng.integers(0, n, size=length)]
                for stop in (0, 1):
                    bits = [int(b) for b in coder.to_bin.bits(syms, stop)]
                    r, blen = coder.to_bin.encode(syms, stop)
                    assert blen == len(bits) and r == int("0" + "".join(map(str, bits)), 2)
                    dec, err = run_decoder(coder, bits, stop)
                    name = f"u{len(names)}"
                    names.append(name)
                    pack_case(store, name, prec=prec, n=n, syms=np.array(syms, dtype=np.int32), stop=stop,
                              bits=np.array(bits, dtype=np.uint8), dec=np.array(dec, dtype=np.int32), dec_err=err)
    store["names"] = np.array(names)
    np.savez_compressed(os.path.join(HERE, "ac_uniform.npz"), **store)
    print("ac_uniform:", len(names), "cases")


# ---------------------------------------------------------------- call-by-call traces of the incremental APIs
def _ragged(store, name, key, seqs, dtype):
    flat = [x for q in seqs for x in q]
    store[f"{name}/{key}"] = np.array(flat, dtype=dtype)
    store[f"{name}/{key}_off"] = np.cumsum([0] + [len(q) for q in seqs]).astype(np.int64)


def gen_api_traces(rng):
    """What the reference returns call by call: A_to_bin.__call__(symbol) digit tuples (2s included), the state after
    every call (l, h, emitted_bits, certain, info), flush digits; A_from_bin.__call__(bit) symbol tuples and state;
    ACSampler's callback traffic (bits handed to compress_output per sample call, bits_per_token values; in expand
    mode the bits pulled per call)."""
    store, names = {}, []
    cases = []
    for prec, V, style in ((16, 3, "flat"), (16, 5, "skew"), (24, 17, "skew"), (32, 64, "skew"), (48, 64, "flat"),
                           (48, 17, "big"), (32, 5, "big")):
        if style == "flat":
            pdf = [1] * V
        elif style == "skew":
            pdf = [int(rng.integers(1, 40)) for _ in range(V)]
            pdf[int(rng.integers(0, V))] += 500
        else:
            pdf = [int(rng.integers(1, 1 << 30)) for _ in range(V)]
        dist = list(np.cumsum(np.array(pdf, dtype=object)))
        cases.append(("cdf", prec, V, dist))
    for prec, n in ((16, 3), (24, 10), (48, 256)):
        cases.append(("uniform", prec, n, None))
    cases.append(("adaptive", 32, 16, None))
    for kind, prec, V, dist in cases:
        def make():
            if kind == "cdf":
                return ac.CDFPredictor(dist)
            if kind == "uniform":
                return ac.Predictor(V)
            return AdaptiveCounts(V)
        for n in (1, 9, 40):
            syms = [int(x) for x in rng.integers(0, V, size=n)]
            enc = ac.AC(make(), prec).to_bin
            digits, states = [], []
            for sy in syms:
                digits.append([int(d) for d in enc(sy)])
                states.append([enc.l, enc.h, enc.emitted_bits, int(enc.certain)])
            infos = [0.0]  # info after the last symbol, before the flush
            infos[0] = float(enc.info)
            tee = float(enc.total_encoded_entropy)
            digits.append([int(d) for d in enc(None)])
            states.append([enc.l, enc.h, enc.emitted_bits, int(enc.certain)])
            bits = [int(b) for b in ac.AC(make(), prec).to_bin.bits(syms, 1)]
            dec = ac.AC(make(), prec).from_bin
            outs, dstates, err = [], [], ""
            try:
                for b in bits:
                    outs.append([int(x) for x in dec(b)])
                    dstates.append([dec.l, dec.h, dec.lb, dec.hb])
            except Exception as e:
                err = type(e).__name__
            name = f"t{len(names)}"
            names.append(name)
            pack_case(store, name, kind=kind, prec=prec, V=V, dist=np.array(dist if dist else [0], dtype=np.int64),
                      syms=np.array(syms, dtype=np.int32), bits=np.array(bits, dtype=np.uint8),
                      enc_states=np.array(states, dtype=np.int64), info=infos[0], total_encoded_entropy=tee,
                      dec_states=np.array(dstates, dtype=np.int64).reshape(-1, 4), dec_err=err)
            _ragged(store, name, "digits", digits, np.int32)
            _ragged(store, name, "dec_out", outs, np.int32)
    # ACSampler callback protocol
    anames = []
    for prec, V in ((16, 3), (32, 10), (48, 50), (48, 256)):
        n = int(rng.integers(5, 40))
        pdfs = [rng.dirichlet(np.ones(V) * 2.0) for _ in range(n)]
        toks = [int(rng.choice(V, p=p)) for p in pdfs]
        s = acs.ACSampler(prec)
        cdfs = []
        for p in pdfs:
            q = np.array(p, dtype=np.float64)
            q += s.get_lop_bias(q)
            q *= s.region.one / np.sum(q)
            cdfs.append(np.cumsum(q).astype(np.uint64))
        out, per_call, bpt = [], [], []
        s.compress_tokens = toks
        s.compress_output = out.append
        s.bits_per_token = bpt.append

        def done(s=s):
            s.on_compress_done = None
            s.flush_compress()
            s.compress_output = None
            s.bits_per_token = None
        s.on_compress_done = done
        i = 0
        while not s.compress_done:
            before = len(out)
            s.sample_scaled_cdf(cdfs[min(i, n - 1)])
            per_call.append(len(out) - before)
            i += 1
        d = acs.ACSampler(prec)
        pulled = [0]

        def counting(bits):
            for b in bits:
                pulled[0] += 1
                yield b
        d.decompress_bits = counting(out)
        dtoks, dpull, err = [], [], ""
        try:
            for i in range(n):
                before = pulled[0]
                dtoks.append(int(d.sample_scaled_cdf(cdfs[i])))
                dpull.append(pulled[0] - before)
        except Exception as e:
            err = type(e).__name__
        name = f"a{len(anames)}"
        anames.append(name)
        pack_case(store, name, prec=prec, cdf=np.stack(cdfs), toks=np.array(toks, dtype=np.int32),
                  bits=np.array(out, dtype=np.uint8), per_call=np.array(per_call, dtype=np.int32),
                  bits_per_token=np.array(bpt, dtype=np.float64), dec=np.array(dtoks, dtype=np.int32),
                  dec_pulled=np.array(dpull, dtype=np.int32), dec_err=err)
    store["names"] = np.array(names)
    store["acs_names"] = np.array(anames)
    np.savez_compressed(os.path.join(HERE, "api_traces.npz"), **store)
    print("api_traces:", len(names), "coder cases,", len(anames), "sampler cases")


if __name__ == "__main__":
    which = sys.argv[1:]
    if not which or "all" in which:
        rng = np.random.default_rng(20261018)
        gen_ac_small(rng)
        gen_ac_llama(rng)
        gen_ac_adaptive()
        gen_acs(rng)
        gen_acs_64k()
        gen_ac_uniform(np.random.default_rng(20261019))
    if not which or "all" in which or "api_traces" in which:
        gen_api_traces(np.random.default_rng(20261020))
