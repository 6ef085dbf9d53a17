"""Pin oracle/lac_oracle.c to outputs of the real reference (tests/golden/*.npz)."""
import os

import numpy as np
import pytest

from oracle import oracle as orc


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name), allow_pickle=False)


def _adaptive_tables(data, V=256):
    """Tables of the goldens' AdaptiveCounts predictor: cumsum(1 + counts so far)."""
    counts = np.ones(V, dtype=np.int64)
    tabs = np.empty((len(data) + 1, V), dtype=np.int64)
    for i, b in enumerate(data):
        tabs[i] = np.cumsum(counts)
        counts[b] += 1
    tabs[len(data)] = np.cumsum(counts)
    return tabs


def test_ac_small_encode_and_decode(ac_small):
    g = ac_small
    names = list(g["names"])
    assert len(names) > 500
    n_fudged = 0
    for nm in names:
        prec, stop = int(g[f"{nm}/prec"]), int(g[f"{nm}/stop"])
        dist, syms = g[f"{nm}/dist"], g[f"{nm}/syms"]
        minp = int(g[f"{nm}/minp"])
        assert minp == orc.lib().orc_cdf_minp(orc._ptr(np.ascontiguousarray(dist)), len(dist))
        n_fudged += int(dist[-1] > (1 << prec) * minp)  # fudged at every width
        bits = orc.ac_encode(dist, syms, prec=prec, stop=stop)
        assert np.array_equal(bits, g[f"{nm}/bits"]), nm
        dec, rc = orc.ac_decode(dist, g[f"{nm}/bits"], prec=prec, stop=stop)
        err = str(g[f"{nm}/dec_err"])
        assert np.array_equal(dec, g[f"{nm}/dec"]), (nm, err, rc)
        assert (rc != 0) == (err != ""), (nm, err, rc)
    assert n_fudged >= 16  # the fudged_dist branch is exercised (plus every ac_llama case)


def test_ac_llama_tables_encode_decode(golden_dir):
    g = _load(golden_dir, "ac_llama.npz")
    for nm in g["names"]:
        tabs, minp, syms = g[f"{nm}/tables"], g[f"{nm}/minp"], g[f"{nm}/syms"]
        for t in range(len(tabs)):
            assert minp[t] == orc.lib().orc_llama_minp(orc._ptr(np.ascontiguousarray(tabs[t])), tabs.shape[1])
        # Llama_AC tables are numpy int64: its fudged_dist wraps mod 2^64 (wrap64)
        bits = orc.ac_encode(tabs, syms, prec=48, stop=1, minp=minp, wrap64=True)
        assert np.array_equal(bits, g[f"{nm}/bits"]), nm
        dec, rc = orc.ac_decode(tabs, g[f"{nm}/bits"], prec=48, stop=0, minp=minp, wrap64=True)
        assert rc == 0 and np.array_equal(dec, g[f"{nm}/dec"]), nm
        # value-based decoder == first n symbols of the literal decoder == input
        assert np.array_equal(orc.ac_decode_n(tabs, g[f"{nm}/bits"], len(syms), prec=48, minp=minp, wrap64=True), syms)


def test_ac_llama_numpy_quantisation_reproduces_tables(golden_dir):
    from oracle import ref_quant
    g = _load(golden_dir, "ac_llama.npz")
    for nm in g["names"]:
        logits, tabs = g[f"{nm}/logits"], g[f"{nm}/tables"]
        same = sum(np.array_equal(ref_quant.calc_dist(logits[min(t, len(logits) - 1)]), tabs[t])
                   for t in range(len(tabs)))
        # identical numpy => identical tables; a different numpy build may differ in np.sum / np.exp
        if same != len(tabs):
            pytest.skip(f"numpy here rounds differently from the golden generator ({same}/{len(tabs)} tables equal)")


def test_ac_adaptive_16k(golden_dir):
    g = _load(golden_dir, "ac_adaptive.npz")
    data = g["data"]
    tabs = _adaptive_tables(data)
    bits = orc.ac_encode(tabs, data.astype(np.int32), prec=int(g["prec"]), stop=1)
    assert np.array_equal(orc.pack_bits(bits), g["comp"])
    back = orc.ac_decode_n(tabs, orc.unpack_bits(g["comp"]), len(data), prec=int(g["prec"]))
    assert np.array_equal(back, data)


def test_acs_small(golden_dir):
    g = _load(golden_dir, "acs_small.npz")
    names = list(g["names"])
    assert len(names) >= 20
    for nm in names:
        prec, cdf, toks = int(g[f"{nm}/prec"]), g[f"{nm}/cdf"], g[f"{nm}/toks"]
        bits = orc.acs_encode(cdf, toks, prec=prec)
        assert np.array_equal(bits, g[f"{nm}/bits"]), nm
        dec, rc = orc.acs_decode(cdf, g[f"{nm}/bits"], len(toks), prec=prec)
        err = str(g[f"{nm}/dec_err"])
        if err == "":
            assert rc == 0 and np.array_equal(dec, g[f"{nm}/dec"]), nm
        else:
            assert rc != 0, (nm, err)
            k = len(g[f"{nm}/dec"])
            assert np.array_equal(dec[:k], g[f"{nm}/dec"]), nm


def test_acs_64k_adaptive(golden_dir):
    """BASELINE config[0]: 64 KB byte stream, adaptive frequency model, ACSampler encode."""
    g = _load(golden_dir, "acs_64k.npz")
    data = g["data"]
    tabs = _adaptive_tables(data)[: len(data)].astype(np.uint64)
    bits = orc.acs_encode(tabs, data.astype(np.int32), prec=int(g["prec"]))
    assert np.array_equal(orc.pack_bits(bits), g["comp"])


def test_pack_unpack_roundtrip():
    rng = np.random.default_rng(0)
    for n in (0, 1, 7, 8, 9, 1000):
        bits = rng.integers(0, 2, n).astype(np.uint8)
        by = orc.pack_bits(bits)
        assert len(by) == (n + 7) // 8
        assert np.array_equal(orc.unpack_bits(by)[:n], bits)
        assert not orc.unpack_bits(by)[n:].any()


def test_ac_uniform_predictor(golden_dir):
    """AC(Predictor(n), prec): the reference's uniform, floor-mapped base class (arith_code.py:64-74); its
    default coder AC() is AC(Predictor(3), 16).  Encoder bit-exact, literal decoder identical including the
    junk symbols its flush() appends (negative ones too), value-based decode returns the coded symbols."""
    g = _load(golden_dir, "ac_uniform.npz")
    names = list(g["names"])
    assert len(names) >= 200
    for nm in names:
        prec, stop, n = int(g[f"{nm}/prec"]), int(g[f"{nm}/stop"]), int(g[f"{nm}/n"])
        syms = g[f"{nm}/syms"]
        bits = orc.ac_encode(orc.uniform(n), syms, prec=prec, stop=stop)
        assert np.array_equal(bits, g[f"{nm}/bits"]), nm
        dec, rc = orc.ac_decode(orc.uniform(n), g[f"{nm}/bits"], prec=prec, stop=stop)
        err = str(g[f"{nm}/dec_err"])
        assert np.array_equal(dec, g[f"{nm}/dec"]), (nm, err, rc)
        assert (rc != 0) == (err != ""), (nm, err, rc)
        if stop:
            assert np.array_equal(orc.ac_decode_n(orc.uniform(n), bits, len(syms), prec=prec), syms), nm


def test_api_traces_bits_and_encoder_state(golden_dir):
    """tests/golden/api_traces.npz (call-by-call traces of the reference's incremental API): the oracle produces the
    same carry-resolved bits, the same (l, h, emitted_bits) before the flush, and the value-based decoder the same
    symbols -- for fixed tables (incl. the fudged_dist branch), the uniform base class and the adaptive model."""
    g = _load(golden_dir, "api_traces.npz")
    for nm in g["names"]:
        kind, prec, V = str(g[f"{nm}/kind"]), int(g[f"{nm}/prec"]), int(g[f"{nm}/V"])
        syms, want = g[f"{nm}/syms"], g[f"{nm}/bits"]
        if kind == "cdf":
            tabs = g[f"{nm}/dist"]
        elif kind == "uniform":
            tabs = orc.uniform(V)
        else:
            tabs = _adaptive_tables(syms, V)[: len(syms)]
        bits, st = orc.ac_encode(tabs, syms, prec=prec, stop=1, return_state=True)
        assert np.array_equal(bits, want), nm
        l, h, nb, _ = g[f"{nm}/enc_states"][len(syms) - 1]        # state after the last symbol, before the flush
        assert (int(st[0]), int(st[1]), int(st[2])) == (int(l), int(h), int(nb)), nm
        # the digits the reference yields call by call, summed with carries, are those bits
        flat = g[f"{nm}/digits"]
        r = 0
        for d in flat:
            r = (r << 1) + int(d)
        assert r == int("0" + "".join(map(str, want.tolist())), 2) and len(flat) == len(want), nm
        assert np.array_equal(orc.ac_decode_n(tabs, want, len(syms), prec=prec), syms), nm
