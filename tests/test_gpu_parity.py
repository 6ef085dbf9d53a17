"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C ABI,
against the CPU oracle and the golden vectors generated from the real reference.
Bar: bit-exact everywhere (integer / byte / index work)."""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():  # collected on CPU boxes, deselected by -m "not gpu"
    pytest.skip("no CUDA device", allow_module_level=True)

from lac_b200 import _ffi, coder  # noqa: E402
from oracle import oracle as orc  # noqa: E402


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _special_rows(V, rng):
    rows = [
        rng.standard_normal(V) * 1.0,
        rng.standard_normal(V) * 8.0,
        rng.standard_normal(V) * 30.0,
        np.zeros(V),
        np.full(V, -1e30),
        np.full(V, 3e38),
        rng.standard_normal(V) * 1e-30,
        np.linspace(-200, 50, V),
        -np.abs(rng.standard_normal(V)) * 100,
    ]
    a = rng.standard_normal(V) * 5
    a[rng.integers(0, V, max(1, V // 7))] = -np.inf
    rows.append(a)
    b = rng.standard_normal(V) * 5
    b[rng.integers(0, V)] = np.nan
    rows.append(b)
    c = rng.standard_normal(V)
    c[rng.integers(0, V)] = np.inf
    rows.append(c)
    rows.append(np.full(V, -np.inf))
    rows.append(np.full(V, np.nan))
    d = np.full(V, -np.inf)
    d[rng.integers(0, V)] = 2.5
    rows.append(d)
    return np.stack(rows).astype(np.float32)


@pytest.mark.parametrize("V", [1, 2, 3, 4, 5, 31, 32, 33, 100, 128, 257, 1000, 4096, 8191, 32000, 32768])
def test_cdf_build_bit_exact(V):
    rng = np.random.default_rng(V)
    logits = _special_rows(V, rng)
    want = orc.lq32_cdf(logits)
    got = coder.cdf_build(_dev(logits)).cpu().numpy().view(np.uint32)
    assert np.array_equal(got, want)
    # every frequency >= 1 and the implicit total is 2^32
    full = np.concatenate([want.astype(np.int64), np.full((len(want), 1), 1 << 32)], axis=1)
    assert (np.diff(full, axis=1) >= 1).all()


@pytest.mark.parametrize("V", [32772, 50000, 65536, 65540, 70001, 100000, 128256, 131072, 151936, 200003, 262144])
def test_multi_part_rows_bit_exact(V):
    """Vocabularies wider than one tile (32768): the row is ceil(V / 32768) tiles (2 .. 8 parts, any count);
    odd vocabularies take the scalar-load path with the same segmentation."""
    rng = np.random.default_rng(V)
    logits = _special_rows(V, rng)[:9]
    logits = np.concatenate([logits, (rng.standard_normal((5, V)) * 6).astype(np.float32)])
    got = coder.cdf_build(_dev(logits)).cpu().numpy().view(np.uint32)
    assert np.array_equal(got, orc.lq32_cdf(logits))
    syms = rng.integers(0, V, len(logits)).astype(np.int32)
    syms[:4] = [0, V - 1, V // 2, 32768]
    lo, hi = orc.lq32_lookup(logits, syms)
    pairs = coder.cdf_lookup(_dev(logits), _dev(syms)).cpu().numpy().view(np.uint32)
    assert np.array_equal(pairs[:, 0], lo)
    assert np.array_equal(pairs[:, 1].astype(np.uint64), hi & 0xFFFFFFFF)


@pytest.mark.parametrize("V,S,T", [(128256, 6, 12), (65536, 40, 5), (262144, 3, 7), (151936, 5, 9), (70001, 4, 6)])
def test_multi_part_encode_decode_roundtrip(V, S, T):
    rng = np.random.default_rng(V + S)
    logits = (rng.standard_normal((S, T, V)) * 5).astype(np.float32)
    syms = rng.integers(0, V, (S, T)).astype(np.int32)
    syms[0, :3] = [0, V - 1, 40000]
    dl = _dev(logits)
    enc = coder.StreamEncoder(S, capacity_bytes=T * 8 + 64)
    enc.encode_logits(dl, _dev(syms), finish=True)
    streams, _ = enc.bitstreams()
    for s in range(min(S, 3)):
        assert streams[s] == _oracle_stream(logits[s], syms[s], 48)
    assert np.array_equal(coder.StreamDecoder(streams).decode_logits(dl).cpu().numpy(), syms)
    dec = coder.StreamDecoder(streams)
    step = torch.stack([dec.decode_step(dl[:, t].contiguous()) for t in range(T)], dim=1).cpu().numpy()
    assert np.array_equal(step, syms)


@pytest.mark.parametrize("V,S", [(32000, 60), (65536, 40), (131072, 24)])
def test_streams_ending_inside_the_first_bit_window(V, S):
    """Streams of 15..22 bytes end inside the 16 bytes the decoder loads at stream start: the bytes past the end
    must read as zeros (A_from_bin sees no further bits, arith_code.py:322-326) and the in-range bytes next to them
    must not be disturbed.  (Regression: a predicated byte gather was once miscompiled for exactly this case.)"""
    for T, scale in ((5, 6.0), (5, 8.0), (6, 4.0)):
        rng = np.random.default_rng(V + T)
        logits = (rng.standard_normal((S, T, V)) * scale).astype(np.float32)
        syms = rng.integers(0, V, (S, T)).astype(np.int32)
        dl = _dev(logits)
        enc = coder.StreamEncoder(S, capacity_bytes=T * 8 + 64)
        enc.encode_logits(dl, _dev(syms), finish=True)
        streams, _ = enc.bitstreams()
        assert any(15 <= len(b) <= 22 for b in streams)
        assert np.array_equal(coder.StreamDecoder(streams).decode_logits(dl).cpu().numpy(), syms)


def test_vocab_out_of_range_is_rejected():
    with pytest.raises(_ffi.LacError):
        coder.cdf_build(torch.zeros((1, 262145), dtype=torch.float32, device="cuda"))


def test_caller_workspace_gives_the_same_result_and_small_workspaces_chunk():
    rng = np.random.default_rng(77)
    S, T, V = 9, 7, 4096
    logits = (rng.standard_normal((S, T, V)) * 4).astype(np.float32)
    syms = rng.integers(0, V, (S, T)).astype(np.int32)
    dl, ds = _dev(logits), _dev(syms)
    ref = coder.StreamEncoder(S)
    ref.encode_logits(dl, ds, finish=True)
    want, _ = ref.bitstreams()
    for rows in (S * T, 5, 1):  # full, a few rows, one row of scratch: the calls work through the rows in launches
        ws = coder.Workspace(rows, V)
        enc = coder.StreamEncoder(S)
        enc.encode_logits(dl, ds, finish=True, ws=ws)
        got, _ = enc.bitstreams()
        assert got == want
        assert np.array_equal(coder.StreamDecoder(got).decode_logits(dl, ws=ws).cpu().numpy(), syms)
        pairs = coder.cdf_lookup(dl.view(S * T, V), ds.view(-1), ws=ws).cpu().numpy()
        assert np.array_equal(pairs, coder.cdf_lookup(dl.view(S * T, V), ds.view(-1)).cpu().numpy())
        assert np.array_equal(coder.cdf_build(dl.view(S * T, V), ws=ws).cpu().numpy(),
                              coder.cdf_build(dl.view(S * T, V)).cpu().numpy())


def test_fused_encoder_equals_lookup_plus_pairs_coder():
    """lac_ac_encode_logits_f32 (one fused kernel) against lac_cdf_lookup_f32 + lac_ac_encode_pairs, all slice
    shapes the launcher distinguishes (T = 1 ... 5, 16, 40), ragged streams, state carried across calls."""
    rng = np.random.default_rng(78)
    S, V = 37, 1000
    for T in (1, 2, 3, 4, 5, 16, 40):
        logits = (rng.standard_normal((S, T, V)) * 5).astype(np.float32)
        syms = rng.integers(0, V, (S, T)).astype(np.int32)
        ntok = rng.integers(0, T + 1, S).astype(np.int32)
        dl, ds, dn = _dev(logits), _dev(syms), _dev(ntok)
        a, b = coder.StreamEncoder(S), coder.StreamEncoder(S)
        for rep in range(3):  # three calls on the same streams, the last one finishes
            a.encode_logits(dl, ds, ntok=dn, finish=(rep == 2))
            pairs = coder.cdf_lookup(dl.view(S * T, V), ds.view(-1))
            b.encode_pairs(pairs.view(S, T, 2), ntok=dn, finish=(rep == 2))
        sa, na = a.bitstreams()
        sb, nb = b.bitstreams()
        assert sa == sb and np.array_equal(na, nb)


def test_truncated_stream_is_reported():
    """The reference raises 'predictor range does not correspond to val' (arith_code.py:277-278) on a stream that
    does not belong to the model; here the decoder flags streams from which it consumed more bits than they hold."""
    rng = np.random.default_rng(79)
    S, T, V = 8, 64, 512
    logits = (rng.standard_normal((S, T, V)) * 2).astype(np.float32)
    syms = rng.integers(0, V, (S, T)).astype(np.int32)
    dl = _dev(logits)
    enc = coder.StreamEncoder(S)
    enc.encode_logits(dl, _dev(syms), finish=True)
    streams, _ = enc.bitstreams()
    assert np.array_equal(coder.StreamDecoder(streams).decode_logits(dl).cpu().numpy(), syms)
    cut = [b[: len(b) // 3] if i % 2 else b for i, b in enumerate(streams)]
    dec = coder.StreamDecoder(cut)
    with pytest.raises(_ffi.LacError) as e:
        dec.decode_logits(dl)
    assert e.value.code == _ffi.LAC_E_STREAM
    st = dec.state.cpu().numpy().view(np.uint32).reshape(S, 10)[:, 8]
    assert all(bool(st[i] & _ffi.LAC_ST_TRUNC) == bool(i % 2) for i in range(S))
    data = np.frombuffer(b"".join(cut), dtype=np.uint8)
    offs = np.concatenate([[0], np.cumsum([len(b) for b in cut])]).astype(np.int64)
    with pytest.raises(_ffi.LacError) as e:
        coder.decode_logits_host(logits, data, offs)
    assert e.value.code == _ffi.LAC_E_STREAM
    with pytest.raises(_ffi.LacError) as e:
        coder.decode_logits_host(logits, data, offs[::-1].copy())
    assert e.value.code == _ffi.LAC_E_ARG


def test_cdf_build_unaligned_rows_use_scalar_path():
    rng = np.random.default_rng(5)
    V = 1001  # odd vocab: rows are not 16-byte aligned
    logits = (rng.standard_normal((37, V)) * 4).astype(np.float32)
    got = coder.cdf_build(_dev(logits)).cpu().numpy().view(np.uint32)
    assert np.array_equal(got, orc.lq32_cdf(logits))


@pytest.mark.parametrize("V", [2, 7, 128, 1001, 32000])
def test_cdf_lookup_bit_exact(V):
    rng = np.random.default_rng(100 + V)
    rows = 300 if V < 5000 else 64
    logits = (rng.standard_normal((rows, V)) * rng.choice([0.5, 3.0, 12.0], (rows, 1))).astype(np.float32)
    syms = rng.integers(0, V, rows).astype(np.int32)
    syms[:4] = [0, V - 1, V // 2, max(0, V - 2)]
    lo, hi = orc.lq32_lookup(logits, syms)
    pairs = coder.cdf_lookup(_dev(logits), _dev(syms)).cpu().numpy().view(np.uint32)
    assert np.array_equal(pairs[:, 0], lo)
    assert np.array_equal(pairs[:, 1].astype(np.uint64), hi & 0xFFFFFFFF)  # 2^32 is carried as 0
    assert (hi[syms == V - 1] == (1 << 32)).all()


def test_cdf_lookup_flags_bad_symbols():
    V = 64
    logits = _dev(np.zeros((3, V), dtype=np.float32))
    syms = _dev(np.array([5, -1, V], dtype=np.int32))
    status = torch.zeros(3, dtype=torch.int32, device="cuda")
    coder.cdf_lookup(logits, syms, status)
    assert status.cpu().tolist() == [0, _ffi.LAC_ST_SYMBOL, _ffi.LAC_ST_SYMBOL]


def _oracle_stream(logits_s, syms_s, prec):
    lo, hi = orc.lq32_lookup(logits_s, syms_s)
    return orc.pack_bits(orc.ac_encode_pairs(lo, hi, prec=prec)).tobytes()


@pytest.mark.parametrize("prec", [34, 40, 48, 56, 60])
def test_encode_decode_logits_vs_oracle_and_reference_semantics(prec):
    rng = np.random.default_rng(prec)
    S, T, V = 9, 40, 300
    logits = (rng.standard_normal((S, T, V)) * rng.choice([1.0, 6.0, 20.0], (S, 1, 1))).astype(np.float32)
    syms = np.empty((S, T), dtype=np.int32)
    for s in range(S):
        for t in range(T):
            p = np.exp((logits[s, t] - logits[s, t].max()).astype(np.float64))
            syms[s, t] = rng.choice(V, p=p / p.sum()) if rng.random() < 0.7 else rng.integers(0, V)
    enc = coder.StreamEncoder(S, prec=prec, capacity_bytes=T * 8 + 64)
    enc.encode_logits(_dev(logits), _dev(syms), finish=True)
    streams, nbits = enc.bitstreams()
    for s in range(S):
        assert streams[s] == _oracle_stream(logits[s], syms[s], prec)
        # level-1 parity: the REFERENCE coder (A_to_bin + CDFPredictor restated literally) fed the
        # same integer tables yields the same bits
        dist = orc.lq32_to_dist(orc.lq32_cdf(logits[s]))
        ref_bits = orc.ac_encode(dist, syms[s], prec=prec, stop=1, minp=np.ones(T, dtype=np.int64))
        assert len(ref_bits) == nbits[s]
        assert orc.pack_bits(ref_bits).tobytes() == streams[s]
        # and the literal reference decoder returns our symbols first
        dec, rc = orc.ac_decode(dist, ref_bits, prec=prec, stop=0, minp=np.ones(T, dtype=np.int64), max_syms=T)
        assert rc == 0 and np.array_equal(dec[:T], syms[s])
    back = coder.StreamDecoder(streams, prec=prec).decode_logits(_dev(logits)).cpu().numpy()
    assert np.array_equal(back, syms)


def test_encode_in_slices_and_ragged_matches_one_shot():
    rng = np.random.default_rng(1)
    S, T, V = 33, 64, 128
    logits = (rng.standard_normal((S, T, V)) * 4).astype(np.float32)
    syms = rng.integers(0, V, (S, T)).astype(np.int32)
    ntok = rng.integers(0, T + 1, S).astype(np.int32)
    ntok[:3] = [0, 1, T]
    dl, ds = _dev(logits), _dev(syms)
    one = coder.StreamEncoder(S, capacity_bytes=T * 8 + 64)
    one.encode_logits(dl, ds, ntok=_dev(ntok), finish=True)
    a, abits = one.bitstreams()
    # same thing in 4 slices of 16 tokens with per-slice ragged counts
    sl = coder.StreamEncoder(S, capacity_bytes=T * 8 + 64)
    for k in range(4):
        part = np.clip(ntok - 16 * k, 0, 16).astype(np.int32)
        sl.encode_logits(dl[:, 16 * k:16 * k + 16].contiguous(), ds[:, 16 * k:16 * k + 16].contiguous(), ntok=_dev(part))
    sl.finish()
    b, bbits = sl.bitstreams()
    assert a == b and np.array_equal(abits, bbits)
    for s in range(S):
        assert a[s] == _oracle_stream(logits[s, :ntok[s]], syms[s, :ntok[s]], 48)
    dec = coder.StreamDecoder(a).decode_logits(dl, ntok=_dev(ntok)).cpu().numpy()
    for s in range(S):
        assert np.array_equal(dec[s, :ntok[s]], syms[s, :ntok[s]])


def test_decode_step_by_step_matches_bulk():
    rng = np.random.default_rng(2)
    S, T, V = 20, 24, 1000
    logits = (rng.standard_normal((S, T, V)) * 5).astype(np.float32)
    syms = rng.integers(0, V, (S, T)).astype(np.int32)
    dl = _dev(logits)
    enc = coder.StreamEncoder(S, capacity_bytes=T * 8 + 64)
    enc.encode_logits(dl, _dev(syms), finish=True)
    streams, _ = enc.bitstreams()
    dec = coder.StreamDecoder(streams)
    out = torch.stack([dec.decode_step(dl[:, t].contiguous()) for t in range(T)], dim=1).cpu().numpy()
    assert np.array_equal(out, syms)


def test_peaked_distributions_and_rare_symbols_roundtrip():
    """Very confident rows with the coded symbol deep in the tail: long renormalisations, carries."""
    rng = np.random.default_rng(3)
    S, T, V = 16, 50, 4096
    logits = (rng.standard_normal((S, T, V))).astype(np.float32)
    hot = rng.integers(0, V, (S, T))
    np.put_along_axis(logits, hot[..., None], 60.0, axis=2)
    syms = np.where(rng.random((S, T)) < 0.5, hot, rng.integers(0, V, (S, T))).astype(np.int32)
    dl = _dev(logits)
    enc = coder.StreamEncoder(S, capacity_bytes=T * 8 + 64)
    enc.encode_logits(dl, _dev(syms), finish=True)
    streams, _ = enc.bitstreams()
    for s in range(S):
        assert streams[s] == _oracle_stream(logits[s], syms[s], 48)
    assert np.array_equal(coder.StreamDecoder(streams).decode_logits(dl).cpu().numpy(), syms)


def test_capacity_overflow_is_reported():
    rng = np.random.default_rng(4)
    S, T, V = 2, 64, 256
    logits = _dev((rng.standard_normal((S, T, V))).astype(np.float32))
    syms = _dev(rng.integers(0, V, (S, T)).astype(np.int32))
    enc = coder.StreamEncoder(S, capacity_bytes=8)
    enc.encode_logits(logits, syms, finish=True)
    with pytest.raises(_ffi.LacError) as e:
        enc.bitstreams()
    assert e.value.code == _ffi.LAC_E_CAP


def test_capacity_overflow_never_writes_outside_the_stream_region():
    """Once a stream overflows its out_stride bytes nothing may be written any more: not past the buffer, not into
    the neighbouring stream (carry ripples used to do both)."""
    rng = np.random.default_rng(41)
    S, T, V, cap = 33, 96, 256, 16
    logits = _dev((rng.standard_normal((S, T, V)) * 4).astype(np.float32))
    syms_h = rng.integers(0, V, (S, T)).astype(np.int32)
    ntok_h = np.full(S, T, dtype=np.int32)
    ntok_h[::2] = 2  # every other stream is short enough to fit: its bytes must survive its neighbours' overflow
    syms, ntok = _dev(syms_h), _dev(ntok_h)
    pairs = coder.cdf_lookup(logits.view(S * T, V), syms.view(-1))
    # canaries: [S, cap] stream regions inside a larger buffer filled with 0xA5
    buf = torch.full((S + 4, cap), 0xA5, dtype=torch.uint8, device="cuda")
    state = torch.zeros((S, _ffi.ENC_STATE_BYTES), dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    L = _ffi.lib()
    _ffi.check(L.lac_enc_init(state.data_ptr(), S, 48, st))
    for lo in range(0, T, 32):  # several calls: an overflowed stream is re-opened, too
        n = torch.clamp(ntok - lo, 0, 32).to(torch.int32)
        _ffi.check(L.lac_ac_encode_pairs(pairs.view(S, T, 2)[:, lo:].data_ptr(), S, 32, T, 1, n.data_ptr(),
                                         state.data_ptr(), buf[2:].data_ptr(), cap, int(lo + 32 >= T), 48, st))
    torch.cuda.synchronize()
    host = buf.cpu().numpy()
    assert (host[:2] == 0xA5).all() and (host[S + 2:] == 0xA5).all(), "wrote outside the output buffer"
    status = state.cpu().numpy().view(np.uint32).reshape(S, 8)[:, 6]
    for s in range(S):
        if ntok_h[s] == 2:
            assert status[s] == 0
            lo_, hi_ = orc.lq32_lookup(logits[s, :2].cpu().numpy(), syms_h[s, :2])
            want = orc.pack_bits(orc.ac_encode_pairs(lo_, hi_, prec=48)).tobytes()
            assert host[2 + s, : len(want)].tobytes() == want, f"stream {s} corrupted by a neighbour's overflow"
        else:
            assert status[s] & _ffi.LAC_ST_CAP


def test_bad_symbol_reaches_the_stream_status():
    """A symbol outside [0, V) must not be coded as nothing: the reference raises 'unknown symbol'
    (arith_code.py:100-101)."""
    rng = np.random.default_rng(42)
    S, T, V = 3, 5, 100
    logits = _dev(rng.standard_normal((S, T, V)).astype(np.float32))
    syms_h = rng.integers(0, V, (S, T)).astype(np.int32)
    syms_h[1, 2] = V
    enc = coder.StreamEncoder(S)
    enc.encode_logits(logits, _dev(syms_h), finish=True)
    with pytest.raises(_ffi.LacError) as e:
        enc.bitstreams()
    assert e.value.code == _ffi.LAC_E_SYMBOL
    flat = rng.standard_normal((S, T, V)).astype(np.float32)
    with pytest.raises(_ffi.LacError) as e:
        coder.encode_logits_host(flat, syms_h)
    assert e.value.code == _ffi.LAC_E_SYMBOL


# ------------------------------------------------------------------ golden vectors of the real reference
def _golden(golden_dir, name):
    return np.load(os.path.join(golden_dir, name), allow_pickle=False)


def test_golden_ac_small_tables(ac_small):
    g = ac_small
    n_checked = n_dec = 0
    for nm in g["names"]:
        prec, stop = int(g[f"{nm}/prec"]), int(g[f"{nm}/stop"])
        dist, syms = g[f"{nm}/dist"], g[f"{nm}/syms"].astype(np.int32)
        minp = np.array([int(g[f"{nm}/minp"])], dtype=np.int64)
        T = len(syms)
        enc = coder.StreamEncoder(1, prec=prec, capacity_bytes=T * 8 + 64)
        enc.encode_tables(_dev(dist), _dev(syms[None]), _dev(minp), finish=bool(stop))
        streams, nbits = enc.bitstreams()
        want = g[f"{nm}/bits"]
        assert nbits[0] == len(want), nm
        assert streams[0] == orc.pack_bits(want).tobytes(), nm
        n_checked += 1
        # decode: first T symbols of the reference decoder's own output
        if str(g[f"{nm}/dec_err"]) == "" and len(g[f"{nm}/dec"]) >= T and T > 0:
            assert np.array_equal(g[f"{nm}/dec"][:T], syms)  # the reference round-trips here
            dec = coder.StreamDecoder([orc.pack_bits(want).tobytes()], prec=prec)
            out = dec.decode_tables(_dev(dist), _dev(minp), T).cpu().numpy()[0]
            assert np.array_equal(out, syms), nm
            n_dec += 1
    assert n_checked > 500 and n_dec > 200


def test_golden_ac_llama_wrap64(golden_dir):
    g = _golden(golden_dir, "ac_llama.npz")
    for nm in g["names"]:
        tabs, minp, syms = g[f"{nm}/tables"], g[f"{nm}/minp"], g[f"{nm}/syms"].astype(np.int32)
        T = len(syms)
        enc = coder.StreamEncoder(1, prec=48, capacity_bytes=T * 8 + 64)
        enc.encode_tables(_dev(tabs), _dev(syms[None]), _dev(minp), finish=True, wrap64=True)
        streams, nbits = enc.bitstreams()
        assert nbits[0] == len(g[f"{nm}/bits"])
        assert streams[0] == orc.pack_bits(g[f"{nm}/bits"]).tobytes()
        out = coder.StreamDecoder(streams, prec=48).decode_tables(_dev(tabs), _dev(minp), T, wrap64=True)
        assert np.array_equal(out.cpu().numpy()[0], syms)
        # exact-integer semantics (what CDFPredictor does with Python ints) also round-trips and
        # matches the oracle's exact mode
        enc2 = coder.StreamEncoder(1, prec=48, capacity_bytes=T * 8 + 64)
        enc2.encode_tables(_dev(tabs), _dev(syms[None]), _dev(minp), finish=True)
        s2, _ = enc2.bitstreams()
        assert s2[0] == orc.pack_bits(orc.ac_encode(tabs, syms, prec=48, minp=minp)).tobytes()
        out2 = coder.StreamDecoder(s2, prec=48).decode_tables(_dev(tabs), _dev(minp), T)
        assert np.array_equal(out2.cpu().numpy()[0], syms)


def _adaptive_tables(data, V=256):
    counts = np.ones(V, dtype=np.int64)
    tabs = np.empty((len(data), V), dtype=np.int64)
    for i, b in enumerate(data):
        tabs[i] = np.cumsum(counts)
        counts[b] += 1
    return tabs


def test_golden_ac_adaptive_16k(golden_dir):
    g = _golden(golden_dir, "ac_adaptive.npz")
    data = g["data"]
    T, prec = len(data), int(g["prec"])
    tabs = _dev(_adaptive_tables(data))
    minp = torch.ones(T, dtype=torch.int64, device="cuda")
    enc = coder.StreamEncoder(1, prec=prec, capacity_bytes=T * 2)
    enc.encode_tables(tabs, _dev(data.astype(np.int32)[None]), minp, finish=True)
    streams, _ = enc.bitstreams()
    assert streams[0] == g["comp"].tobytes()
    out = coder.StreamDecoder(streams, prec=prec).decode_tables(tabs, minp, T).cpu().numpy()[0]
    assert np.array_equal(out, data)


def test_golden_acs_small(golden_dir):
    g = _golden(golden_dir, "acs_small.npz")
    for nm in g["names"]:
        prec, cdf, toks = int(g[f"{nm}/prec"]), g[f"{nm}/cdf"], g[f"{nm}/toks"].astype(np.int32)
        T = len(toks)
        enc = coder.StreamEncoder(1, prec=prec, capacity_bytes=T * 8 + 64)
        enc.acs_encode_tables(_dev(cdf.view(np.int64)), _dev(toks[None]), finish=True)
        streams, nbits = enc.bitstreams()
        assert nbits[0] == len(g[f"{nm}/bits"]), nm
        assert streams[0] == orc.pack_bits(g[f"{nm}/bits"]).tobytes(), nm
        # flush_compress does not pin the final interval (the reference's own expand path round-trips
        # only part of these cases); with the safe termination the same Region coder is lossless
        enc2 = coder.StreamEncoder(1, prec=prec, capacity_bytes=T * 8 + 64)
        enc2.acs_encode_tables(_dev(cdf.view(np.int64)), _dev(toks[None]), finish="safe")
        s2, nb2 = enc2.bitstreams()
        assert nb2[0] <= nbits[0] + prec + 2
        out = coder.StreamDecoder(s2, prec=prec).acs_decode_tables(_dev(cdf.view(np.int64)), T)
        assert np.array_equal(out.cpu().numpy()[0], toks), nm


def test_golden_acs_64k_config0(golden_dir):
    """BASELINE config[0]: 64 KB synthetic bytes, adaptive frequency model, ACSampler coder."""
    g = _golden(golden_dir, "acs_64k.npz")
    data = g["data"]
    T, prec = len(data), int(g["prec"])
    tabs = _dev(_adaptive_tables(data))
    enc = coder.StreamEncoder(1, prec=prec, capacity_bytes=T)
    enc.acs_encode_tables(tabs, _dev(data.astype(np.int32)[None]), finish=True)
    streams, _ = enc.bitstreams()
    assert streams[0] == g["comp"].tobytes()
    # round trip with the safe termination (the reference flush leaves the tail undetermined)
    enc2 = coder.StreamEncoder(1, prec=prec, capacity_bytes=T)
    enc2.acs_encode_tables(tabs, _dev(data.astype(np.int32)[None]), finish="safe")
    s2, _ = enc2.bitstreams()
    assert s2[0][:len(streams[0]) - 8] == streams[0][:-8]
    out = coder.StreamDecoder(s2, prec=prec).acs_decode_tables(tabs, T).cpu().numpy()[0]
    assert np.array_equal(out, data)
    # the reference-flushed stream still decodes everything but (at most) its last tokens
    out1 = coder.StreamDecoder(streams, prec=prec).acs_decode_tables(tabs, T).cpu().numpy()[0]
    assert np.array_equal(out1[:-8], data[:-8])


# ------------------------------------------------------------------ full-size properties
def test_full_size_slice_roundtrip_and_size():
    """BASELINE config[1] shape (vocab 32000, 1024 streams), a 4-token slice: lossless round trip and the
    coded size within a few bits per stream of the ideal code length of the LQ32 tables."""
    S, T, V = 1024, 4, 32000
    gen = torch.Generator(device="cuda").manual_seed(7)
    logits = torch.randn((S, T, V), generator=gen, device="cuda") * 3.0
    syms = torch.multinomial(torch.softmax(logits.view(S * T, V), dim=-1), 1, generator=gen).view(S, T).to(torch.int32)
    enc = coder.StreamEncoder(S, capacity_bytes=T * 8 + 64)
    enc.encode_logits(logits, syms, finish=True)
    streams, nbits = enc.bitstreams()
    back = coder.StreamDecoder(streams).decode_logits(logits)
    assert torch.equal(back, syms)
    pairs = coder.u32(coder.cdf_lookup(logits.view(S * T, V), syms.view(-1)))
    hi = torch.where(pairs[:, 1] == 0, torch.full_like(pairs[:, 1], 1 << 32), pairs[:, 1])
    ideal = (32.0 - torch.log2((hi - pairs[:, 0]).double())).view(S, T).sum(1).cpu().numpy()
    assert (nbits.astype(np.float64) <= ideal + 3).all() and (nbits.astype(np.float64) >= ideal - 1).all()
    # spot-check 3 streams bit-exact against the oracle at full vocab
    lg, sy = logits.cpu().numpy(), syms.cpu().numpy()
    for s in (0, 511, 1023):
        assert streams[s] == _oracle_stream(lg[s], sy[s], 48)


def test_host_buffer_api_roundtrip():
    rng = np.random.default_rng(9)
    S, T, V = 12, 10, 32000
    logits = (rng.standard_normal((S, T, V)) * 2).astype(np.float32)
    syms = rng.integers(0, V, (S, T)).astype(np.int32)
    out, nbits = coder.encode_logits_host(logits, syms)
    nbytes = (nbits + 7) // 8
    offs = np.zeros(S + 1, dtype=np.int64)
    offs[1:] = np.cumsum(nbytes)
    data = np.concatenate([out[s, :nbytes[s]] for s in range(S)] + [np.zeros(16, np.uint8)])
    for s in (0, S - 1):
        assert out[s, :nbytes[s]].tobytes() == _oracle_stream(logits[s], syms[s], 48)
    back = coder.decode_logits_host(logits, data, offs)
    assert np.array_equal(back, syms)


_CHUNK_SCRIPT = r"""
import sys, numpy as np, torch
sys.path.insert(0, sys.argv[1])
from lac_b200 import coder
rng = np.random.default_rng(11)
out = {}
for V, S, T in ((1000, 5, 37), (40000, 3, 9)):
    logits = (rng.standard_normal((S, T, V)) * 4).astype(np.float32)
    syms = rng.integers(0, V, (S, T)).astype(np.int32)
    ntok = rng.integers(0, T + 1, S).astype(np.int32)
    ntok[0] = T
    dl, ds, dn = (torch.from_numpy(a).cuda() for a in (logits, syms, ntok))
    enc = coder.StreamEncoder(S, capacity_bytes=T * 8 + 64)
    enc.encode_logits(dl, ds, ntok=dn, finish=True)
    streams, _ = enc.bitstreams()
    dec = coder.StreamDecoder(streams).decode_logits(dl, ntok=dn).cpu().numpy()
    for s in range(S):
        assert np.array_equal(dec[s, :ntok[s]], syms[s, :ntok[s]]), (V, s)
    out[str(V)] = np.frombuffer(b"".join(streams), dtype=np.uint8)
np.savez(sys.argv[2], **out)
"""


@pytest.mark.gpu
def test_row_and_token_chunking_of_the_summary_scratch(tmp_path):
    """lac_cdf_lookup_f32 / lac_ac_decode_logits_f32 process long inputs in chunks of rows / tokens bounded by the
    summary scratch size; with a 4 KB budget every call runs many chunks (ragged streams included) and must
    produce the same bytes and symbols as the unchunked run."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = {}
    for name, budget in (("full", None), ("tiny", "4096")):
        env = dict(os.environ)
        env.pop("LAC_SUMMARY_BYTES", None)
        if budget:
            env["LAC_SUMMARY_BYTES"] = budget
        out = tmp_path / f"{name}.npz"
        r = subprocess.run([sys.executable, "-c", _CHUNK_SCRIPT, root, str(out)], env=env, capture_output=True,
                           text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        res[name] = np.load(out)
    for k in res["full"].files:
        assert np.array_equal(res["full"][k], res["tiny"][k])


_PATH_SCRIPT = r"""
import sys, numpy as np, torch
sys.path.insert(0, sys.argv[1])
from lac_b200 import coder
from oracle import oracle as orc
rng = np.random.default_rng(21)
for V, S, T in ((32000, 6, 5), (4096, 9, 7), (1000, 4, 6), (70004, 3, 20)):
    logits = (rng.standard_normal((S, T, V)) * 5).astype(np.float32)
    syms = rng.integers(0, V, (S, T)).astype(np.int32)
    dl, ds = torch.from_numpy(logits).cuda(), torch.from_numpy(syms).cuda()
    cum = coder.cdf_build(dl.view(S * T, V)).cpu().numpy().view(np.uint32)
    assert np.array_equal(cum, orc.lq32_cdf(logits.reshape(S * T, V))), V
    enc = coder.StreamEncoder(S, capacity_bytes=T * 8 + 64)
    enc.encode_logits(dl, ds, finish=True)
    streams, _ = enc.bitstreams()
    lo, hi = orc.lq32_lookup(logits[0], syms[0])
    assert streams[0] == orc.pack_bits(orc.ac_encode_pairs(lo, hi, prec=48)).tobytes(), V
    assert np.array_equal(coder.StreamDecoder(streams).decode_logits(dl).cpu().numpy(), syms), V
print("ok")
"""


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"LAC_NO_TMA": "1"}, {"LAC_TMA_CHUNKS": "2"}, {"LAC_TMA_CHUNKS": "8"},
                                 {"LAC_TILE_WARPS": "16"}, {"LAC_TILE_WARPS": "8"}, {"LAC_CODER_SPB": "0"},
                                 {"LAC_CODER_SPB": "16"}, {"LAC_CODER_SPB": "0", "LAC_CODER_TPB": "32"}])
def test_alternative_staging_paths_are_bit_exact(env):
    """The measurement switches select other instantiations of pass 1 (128-bit LDG staging, 2 or 8 TMA chunks per
    tile, 2 or 4 CTAs per SM) and of the pairs coder (thread-per-stream with byte stores, other streams-per-warp
    counts); they must stay bit-exact with the oracle like the defaults."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    e = dict(os.environ)
    for k in ("LAC_NO_TMA", "LAC_TMA_CHUNKS", "LAC_TILE_WARPS", "LAC_CODER_SPB", "LAC_CODER_TPB"):
        e.pop(k, None)
    e.update(env)
    r = subprocess.run([sys.executable, "-c", _PATH_SCRIPT, root], env=e, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]


@pytest.mark.gpu
def test_golden_ac_uniform_predictor(golden_dir):
    """AC(Predictor(n), prec), the reference's uniform floor-mapped base class (its default AC() is Predictor(3)
    at 16 bits): GPU bytes identical to the reference's bits, decode returns the coded symbols; all 240 cases
    batched per (n, prec, T, stop) would hide nothing, so they run one stream each plus one batched check."""
    g = _golden(golden_dir, "ac_uniform.npz")
    n_checked = n_dec = 0
    for nm in g["names"]:
        prec, stop, n = int(g[f"{nm}/prec"]), int(g[f"{nm}/stop"]), int(g[f"{nm}/n"])
        syms = g[f"{nm}/syms"].astype(np.int32)
        T = len(syms)
        want = g[f"{nm}/bits"]
        enc = coder.StreamEncoder(1, prec=prec, capacity_bytes=T * 8 + 64)
        if T:
            enc.encode_uniform(_dev(syms[None]), n, finish=bool(stop))
        elif stop:
            enc.finish()
        streams, nbits = enc.bitstreams()
        assert nbits[0] == len(want), nm
        assert streams[0] == orc.pack_bits(want).tobytes(), nm
        n_checked += 1
        if stop and T:
            out = coder.StreamDecoder([streams[0]], prec=prec).decode_uniform(n, T).cpu().numpy()[0]
            assert np.array_equal(out, syms), nm
            n_dec += 1
    assert n_checked == 240 and n_dec >= 90
    # many streams at once, ragged, and a symbol outside the alphabet flags its stream only
    rng = np.random.default_rng(3)
    S, T, n = 70, 50, 3
    syms = rng.integers(0, n, (S, T)).astype(np.int32)
    ntok = rng.integers(0, T + 1, S).astype(np.int32)
    enc = coder.StreamEncoder(S, prec=16, capacity_bytes=T * 8 + 64)
    enc.encode_uniform(_dev(syms), n, ntok=_dev(ntok), finish=True)
    streams, nbits = enc.bitstreams()
    for s in range(S):
        want = orc.ac_encode(orc.uniform(n), syms[s, :ntok[s]], prec=16, stop=1)
        assert nbits[s] == len(want) and streams[s] == orc.pack_bits(want).tobytes()
    out = coder.StreamDecoder(streams, prec=16).decode_uniform(n, T, ntok=_dev(ntok)).cpu().numpy()
    for s in range(S):
        assert np.array_equal(out[s, :ntok[s]], syms[s, :ntok[s]])


@pytest.mark.gpu
@pytest.mark.parametrize("V", [1000, 32000, 65536])
def test_special_rows_through_both_second_passes(V):
    """Degenerate and hostile rows (all -inf, all NaN, a +inf, huge magnitudes, -inf holes) through
    summary + pair + coder and summary + serial decode: pairs equal the oracle's, streams round-trip."""
    rng = np.random.default_rng(V + 7)
    rows = _special_rows(V, rng)                      # 15 rows
    S, T = 3, len(rows)
    logits = np.stack([rows[rng.permutation(T)] for _ in range(S)])
    syms = rng.integers(0, V, (S, T)).astype(np.int32)
    syms[0, :4] = [0, V - 1, V // 2, 1]
    lo, hi = orc.lq32_lookup(logits.reshape(S * T, V), syms.reshape(-1))
    pairs = coder.cdf_lookup(_dev(logits.reshape(S * T, V)), _dev(syms.reshape(-1))).cpu().numpy().view(np.uint32)
    assert np.array_equal(pairs[:, 0], lo) and np.array_equal(pairs[:, 1].astype(np.uint64), hi & 0xFFFFFFFF)
    enc = coder.StreamEncoder(S, capacity_bytes=T * 8 + 64)
    enc.encode_logits(_dev(logits), _dev(syms), finish=True)
    streams, _ = enc.bitstreams()
    for s in range(S):
        assert streams[s] == _oracle_stream(logits[s], syms[s], 48)
    assert np.array_equal(coder.StreamDecoder(streams).decode_logits(_dev(logits)).cpu().numpy(), syms)


@pytest.mark.gpu
@pytest.mark.parametrize("with_ws", [True, False])
def test_encode_and_decode_steps_are_cuda_graph_capturable(with_ws):
    """The device entry points are asynchronous and use only stream-ordered work (with a caller workspace: no
    allocation at all; without: cudaMallocAsync scratch), so a model-in-the-loop step can be captured into a CUDA
    graph and replayed: several replays walk the coder state token by token."""
    rng = np.random.default_rng(9)
    S, V, T = 64, 32000, 5
    logits_all = _dev((rng.standard_normal((S, T, V)) * 4).astype(np.float32))
    syms_all = _dev(rng.integers(0, V, (S, T)).astype(np.int32))
    ref_enc = coder.StreamEncoder(S, capacity_bytes=256)
    ref_enc.encode_logits(logits_all, syms_all, finish=True)           # also warms the scratch pool up
    want, _ = ref_enc.bitstreams()
    ws = coder.Workspace(S, V) if with_ws else None
    wsp = (ws.ptr, ws.nbytes) if ws else (None, 0)
    logits = torch.empty((S, 1, V), dtype=torch.float32, device="cuda")   # static graph inputs
    syms = torch.empty((S, 1), dtype=torch.int32, device="cuda")
    enc = coder.StreamEncoder(S, capacity_bytes=256)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    L = _ffi.lib()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            st = torch.cuda.current_stream().cuda_stream
            _ffi.check(L.lac_ac_encode_logits_f32(logits.data_ptr(), S, 1, V, V, V, syms.data_ptr(), 1, None,
                                                  enc.state.data_ptr(), enc.out.data_ptr(), enc.cap, 0, enc.prec,
                                                  *wsp, st))
    torch.cuda.current_stream().wait_stream(side)
    for t in range(T):
        logits.copy_(logits_all[:, t:t + 1])
        syms.copy_(syms_all[:, t:t + 1])
        graph.replay()
    enc.finish()
    torch.cuda.synchronize()
    got, _ = enc.bitstreams()
    assert got == want
    # decode step captured the same way
    dec = coder.StreamDecoder(want)
    out = torch.zeros((S, 1), dtype=torch.int32, device="cuda")
    g2 = torch.cuda.CUDAGraph()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(g2, stream=side):
            st = torch.cuda.current_stream().cuda_stream
            _ffi.check(L.lac_ac_decode_logits_f32(logits.data_ptr(), S, 1, V, V, V, None, dec.state.data_ptr(),
                                                  dec.bytes.data_ptr(), dec.offsets.data_ptr(), out.data_ptr(), 1,
                                                  dec.prec, *wsp, st))
    torch.cuda.current_stream().wait_stream(side)
    for t in range(T):
        logits.copy_(logits_all[:, t:t + 1])
        g2.replay()
        assert torch.equal(out, syms_all[:, t:t + 1])
    assert dec.status() == 0
