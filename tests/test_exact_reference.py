"""oracle/pyref.py, an exact Python-int restatement of the reference's coding path, is pinned to every golden file;
the C oracle is then compared with it where no golden reaches: prec 49 .. 60, table totals up to 2^62, vocabularies
above 256, wrap64 products at every width, zero-frequency entries, shared and per-position tables."""
import os

import numpy as np
import pytest

from oracle import oracle as orc
from oracle import pyref, ref_quant


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name), allow_pickle=False)


def _bits(a):
    return [int(b) for b in a]


# ------------------------------------------------------------------------------------------------ pinned to goldens
def test_pyref_reproduces_ac_small(ac_small):
    g = ac_small
    for nm in g["names"]:
        prec, stop = int(g[f"{nm}/prec"]), int(g[f"{nm}/stop"])
        dist, syms = g[f"{nm}/dist"].tolist(), g[f"{nm}/syms"].tolist()
        pred = pyref.CDFPredictor(dist)
        assert pred.minp == int(g[f"{nm}/minp"]), nm
        assert pyref.ac_encode(pred, syms, prec, stop=bool(stop)) == _bits(g[f"{nm}/bits"]), nm
        # the reference's literal decoder returned these symbols first; the value-based decoder returns them as well
        dec = g[f"{nm}/dec"].tolist()
        k = min(len(dec), len(syms))
        if stop:
            assert pyref.ac_decode_n(pred, _bits(g[f"{nm}/bits"]), len(syms), prec) == syms, nm
        assert pyref.ac_decode_n(pred, _bits(g[f"{nm}/bits"]), k, prec) == dec[:k], nm


def test_pyref_reproduces_ac_llama_wrap64(golden_dir):
    g = _load(golden_dir, "ac_llama.npz")
    for nm in g["names"]:
        tabs, minp, syms = g[f"{nm}/tables"], g[f"{nm}/minp"], g[f"{nm}/syms"].tolist()
        preds = [pyref.CDFPredictor(tabs[t].tolist(), int(minp[t]), wrap=True) for t in range(len(tabs))]
        assert [pyref.llama_minp(tabs[t].tolist()) for t in range(len(tabs))] == minp.tolist(), nm
        assert pyref.ac_encode(preds, syms, 48) == _bits(g[f"{nm}/bits"]), nm
        assert pyref.ac_decode_n(preds, _bits(g[f"{nm}/bits"]), len(syms), 48) == syms, nm
        # without the wrap the same tables code differently: the goldens do pin the wrap64 products
        exact = [pyref.CDFPredictor(tabs[t].tolist(), int(minp[t])) for t in range(len(tabs))]
        assert pyref.ac_encode(exact, syms, 48) != _bits(g[f"{nm}/bits"]), nm


def test_pyref_reproduces_ac_uniform(golden_dir):
    g = _load(golden_dir, "ac_uniform.npz")
    for nm in g["names"]:
        prec, stop, n = int(g[f"{nm}/prec"]), int(g[f"{nm}/stop"]), int(g[f"{nm}/n"])
        syms = g[f"{nm}/syms"].tolist()
        assert pyref.ac_encode(pyref.Predictor(n), syms, prec, stop=bool(stop)) == _bits(g[f"{nm}/bits"]), nm
        if stop:
            assert pyref.ac_decode_n(pyref.Predictor(n), _bits(g[f"{nm}/bits"]), len(syms), prec) == syms, nm


def test_pyref_reproduces_acs_small(golden_dir):
    g = _load(golden_dir, "acs_small.npz")
    for nm in g["names"]:
        prec, cdf, toks = int(g[f"{nm}/prec"]), g[f"{nm}/cdf"], g[f"{nm}/toks"].tolist()
        cdfs = [r.tolist() for r in cdf] if cdf.ndim == 2 else cdf.tolist()
        assert pyref.acs_encode(cdfs, toks, prec, finish=1) == _bits(g[f"{nm}/bits"]), nm


def test_pyref_reproduces_api_traces_and_encoder_states(golden_dir):
    g = _load(golden_dir, "api_traces.npz")
    for nm in g["names"]:
        kind, prec, V = str(g[f"{nm}/kind"]), int(g[f"{nm}/prec"]), int(g[f"{nm}/V"])
        syms = g[f"{nm}/syms"].tolist()
        if kind == "cdf":
            preds = pyref.CDFPredictor(g[f"{nm}/dist"].tolist())
        elif kind == "uniform":
            preds = pyref.Predictor(V)
        else:  # the adaptive model: cumsum(1 + counts so far)
            counts, preds = [1] * V, []
            for s in syms:
                preds.append(pyref.CDFPredictor(np.cumsum(counts).tolist()))
                counts[s] += 1
        enc = pyref.A_to_bin(prec)
        states = g[f"{nm}/enc_states"]
        for t, s in enumerate(syms):
            enc.receive_symbol(pyref._pred_at(preds, t), s)
            assert enc.state() == tuple(int(x) for x in states[t][:3]), (nm, t)
        enc.flush()
        assert enc.out.bits() == _bits(g[f"{nm}/bits"]), nm
        assert pyref.ac_decode_n(preds, _bits(g[f"{nm}/bits"]), len(syms), prec) == syms, nm


# ------------------------------------------------------------------------------------------------ oracle == pyref
PRECS = (2, 8, 16, 33, 34, 47, 48, 49, 55, 59, 60)
VOCABS = (1, 2, 3, 31, 32, 33, 63, 64, 65, 257, 1000, 4096)


def random_table(rng, V, total_log2, zero_frac):
    """Inclusive cumulative int table of V entries with a total near 2^total_log2 and about zero_frac of the entries
    at frequency 0 (at least one entry is positive).  Exact ints: totals reach 2^62."""
    w = rng.exponential(1.0, V) ** rng.choice([1.0, 3.0])
    w[rng.random(V) < zero_frac] = 0.0
    if not w.any():
        w[rng.integers(0, V)] = 1.0
    tot = 1 << total_log2
    f = [int(x) for x in np.floor(w / w.sum() * tot)]
    if sum(f) == 0:
        f[int(np.argmax(w))] = 1
    return np.cumsum(np.array(f, dtype=object)).tolist()


def coded_symbols(rng, dist, T):
    """T symbols drawn among the entries of positive frequency (a zero-width symbol is never coded)."""
    pos = [i for i in range(len(dist)) if dist[i] - (dist[i - 1] if i else 0) > 0]
    return [int(pos[k]) for k in rng.integers(0, len(pos), T)]


def draw_tables_case(rng, prec, V):
    """One random case: per-position tables (or one shared table), minp, symbols, wrap64 flag."""
    T = int(rng.integers(1, 4 if V >= 1000 else 13))
    shared = bool(rng.random() < 0.4)
    wrap = bool(rng.random() < 0.5)
    zero_frac = float(rng.choice([0.0, 0.0, 0.2, 0.7]))
    ntab = 1 if shared else T
    tabs, minps = [], []
    for _ in range(ntab):
        # around prec (both branches of fudged_dist) or anywhere in 2^1 .. 2^62
        e = int(np.clip(prec + rng.integers(-8, 9), 1, 62)) if rng.random() < 0.5 else int(rng.integers(1, 63))
        d = random_table(rng, V, e, zero_frac)
        tabs.append(d)
        minps.append(pyref.llama_minp(d) if wrap else pyref.cdf_minp(d))
    syms = []
    for t in range(T):
        syms += coded_symbols(rng, tabs[0 if shared else t], 1)
    return tabs, minps, syms, wrap, shared


def test_oracle_equals_pyref_on_random_tables():
    rng = np.random.default_rng(2024)
    branches = {False: 0, True: 0}
    wraps = {False: 0, True: 0}
    for prec in PRECS:
        for V in VOCABS:
            for _ in range(2):
                tabs, minps, syms, wrap, shared = draw_tables_case(rng, prec, V)
                preds = [pyref.CDFPredictor(d, m, wrap) for d, m in zip(tabs, minps)]
                preds = preds[0] if shared else preds
                stop = bool(rng.random() < 0.8)
                for t, d in enumerate(tabs):
                    thr = (1 << prec) * minps[t]
                    branches[d[-1] > (pyref.wrap64(thr) if wrap else thr)] += 1
                wraps[wrap] += 1
                try:
                    want = pyref.ac_encode(preds, syms, prec, stop)
                except ZeroDivisionError:
                    # a zero-width coded symbol: the reference never terminates, the oracle reports it
                    arr = np.array(tabs[0] if shared else tabs, dtype=np.int64)
                    with pytest.raises(orc.OracleError):
                        orc.ac_encode(arr, syms, prec=prec, stop=int(stop), minp=np.array(minps), wrap64=wrap)
                    continue
                arr = np.array(tabs[0] if shared else tabs, dtype=np.int64)
                mp = np.array(minps, dtype=np.int64)
                bits, st = orc.ac_encode(arr, syms, prec=prec, stop=int(stop), minp=mp, return_state=True, wrap64=wrap)
                assert _bits(bits) == want, (prec, V, wrap, shared)
                if stop:
                    back = orc.ac_decode_n(arr, bits, len(syms), prec=prec, minp=mp, wrap64=wrap)
                    assert back.tolist() == syms == pyref.ac_decode_n(preds, want, len(syms), prec), (prec, V, wrap)
    assert min(branches.values()) >= 20 and min(wraps.values()) >= 20, (branches, wraps)


def test_oracle_equals_pyref_uniform_and_acs_across_precisions():
    rng = np.random.default_rng(77)
    for prec in PRECS:
        for n in (2, 3, 255, 65536, 2 ** 31 - 1):
            if n > 1 << (prec - 1):  # wider alphabets than half the range have zero-width symbols
                continue
            syms = rng.integers(0, n, int(rng.integers(1, 30))).tolist()
            want = pyref.ac_encode(pyref.Predictor(n), syms, prec)
            bits = orc.ac_encode(orc.uniform(n), syms, prec=prec)
            assert _bits(bits) == want, (prec, n)
            assert pyref.ac_decode_n(pyref.Predictor(n), want, len(syms), prec) == syms
        for V in (1, 2, 33, 257, 1000):
            if 4 * V >= 1 << prec:  # acs_cdf needs room for a floor under every entry
                continue
            T = int(rng.integers(1, 12))
            cdf = np.stack([ref_quant.acs_cdf(rng.dirichlet(np.full(V, 0.3)), precision=prec) for _ in range(T)])
            if (np.diff(np.concatenate([np.zeros((T, 1), np.uint64), cdf], axis=1).astype(np.int64), axis=1) <= 0).any():
                continue
            toks = rng.integers(0, V, T).tolist()
            want = pyref.acs_encode([r.tolist() for r in cdf], toks, prec, finish=1)
            assert _bits(orc.acs_encode(cdf, toks, prec=prec)) == want, (prec, V)


def test_wrap64_restatement():
    assert pyref.wrap64((1 << 63) - 1) == (1 << 63) - 1
    assert pyref.wrap64(1 << 63) == -(1 << 63)
    assert pyref.wrap64(-(1 << 63) - 1) == (1 << 63) - 1
    a, b = 0x7FFF_FFFF_FFFF_FFF0, 0x1234_5678
    assert pyref.wrap64(a * b) == int((np.array([a], dtype=np.int64) * np.int64(b))[0])
