"""The adaptive count models on the GPU (run with -m gpu on a B200): lac_ac_{en,de}code_adaptive (ProbPredictor with
prob(s) = counts[s] under A_to_bin / A_from_bin) and lac_acs_{en,de}code_adaptive (the same counts under ACSampler).

* the goldens ac_adaptive.npz and acs_64k.npz from the counts alone, decoded without tables or plaintext;
* randomised cases against the pinned C oracle on tables materialised on the CPU from the same counts (vocabulary
  1 .. 4096, precision 2 .. 60 with low precisions reaching fudged_dist, 1 .. 40 streams, zero counts, inc 0 .. 5,
  ragged token counts, one to three calls and a flush-only call), with guard bytes around every buffer;
* inc = 0 against the static table coders, tokens a stream cannot code, and the mirror API's CountPredictor."""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():  # collected on CPU boxes, deselected by -m "not gpu"
    pytest.skip("no CUDA device", allow_module_level=True)

from lac_b200 import _ffi, coder  # noqa: E402
from lac_b200 import arith_code as ac  # noqa: E402
from oracle import oracle as orc  # noqa: E402

G = 0xA5                    # guard byte
JUNK = -(1 << 61) + 12345   # guard rows of the counts buffers


def _golden(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _packed(bits):
    return orc.pack_bits(bits).tobytes()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def walk(counts, syms, inc):
    """The reference predictor along syms (table, then accept): tables [max(n, 1), V], minp per table, final counts."""
    c = np.array(counts, dtype=np.int64)
    tabs, minp = [], []
    for a in syms:
        tabs.append(np.cumsum(c))
        pos = c[c > 0]
        minp.append(int(pos.min()) if len(pos) else 1)
        c[int(a)] += inc
    if not tabs:
        tabs, minp = [np.cumsum(c)], [1]
    return np.stack(tabs), np.array(minp, dtype=np.int64), c


class Rig:
    """Device buffers of one batch, each with a guard row before and after."""

    def __init__(self, S, T, V, cap, init, prec):
        self.S, self.T, self.V, self.cap = S, T, V, cap
        self.out = torch.full((S + 2, cap), G, dtype=torch.uint8, device="cuda")
        self.enc = torch.full((S + 2, _ffi.ENC_STATE_BYTES), G, dtype=torch.uint8, device="cuda")
        self.dec = torch.full((S + 2, _ffi.DEC_STATE_BYTES), G, dtype=torch.uint8, device="cuda")
        self.back = torch.full((S + 2, T + 3), -7, dtype=torch.int32, device="cuda")
        c = np.full((S + 2, V), JUNK, dtype=np.int64)
        c[1:S + 1] = init
        self.ecounts, self.dcounts = _dev(c), _dev(c.copy())
        _ffi.check(_ffi.lib().lac_enc_init(self.enc[1:].data_ptr(), S, prec, _stream()))

    def counts(self, which):
        torch.cuda.synchronize()
        c = (self.ecounts if which == "enc" else self.dcounts).cpu().numpy()
        assert (c[0] == JUNK).all() and (c[self.S + 1] == JUNK).all(), "counts buffer overrun"
        return c[1:self.S + 1]

    def streams(self):
        torch.cuda.synchronize()
        st = self.enc[1:self.S + 1].cpu().numpy().view(np.int64).reshape(self.S, 4)
        host = self.out.cpu().numpy()
        assert (host[0] == G).all() and (host[self.S + 1] == G).all(), "bitstream buffer overrun"
        e = self.enc.cpu().numpy()
        assert (e[0] == G).all() and (e[self.S + 1] == G).all(), "encoder state overrun"
        got = []
        for s in range(self.S):
            used = (int(st[s, 2]) + 7) // 8
            assert (host[1 + s, used:] == G).all(), ("bytes written past the stream's end", s)
            got.append(host[1 + s, :used].tobytes())
        return got, st[:, 2].copy(), (st[:, 3] & 0xFFFFFFFF).copy(), st[:, :2].copy()

    def decoded(self, ntok):
        torch.cuda.synchronize()
        got = self.back.cpu().numpy()
        assert (got[0] == -7).all() and (got[self.S + 1] == -7).all(), "symbol buffer overrun"
        d = self.dec.cpu().numpy()
        assert (d[0] == G).all() and (d[self.S + 1] == G).all(), "decoder state overrun"
        for s in range(self.S):
            assert (got[1 + s, int(ntok[s]):] == -7).all(), ("symbols written past the stream's token count", s)
        st = self.dec[1:self.S + 1].cpu().numpy().view(np.int64).reshape(self.S, 5)
        return got[1:self.S + 1], (st[:, 4] & 0xFFFFFFFF).copy()


def _cuts(rng, T):
    """One to three calls: the token range split at up to two random points."""
    k = int(rng.integers(0, 3))
    pts = sorted(int(x) for x in rng.integers(0, T + 1, k))
    b = [0] + pts + [T]
    return [(b[i], b[i + 1]) for i in range(len(b) - 1) if b[i + 1] > b[i]] or [(0, T)]


def _piece(ntok, t0, t1):
    return _dev(np.clip(ntok - t0, 0, t1 - t0).astype(np.int32))


def encode_calls(rng, coder_name, R, d_syms, inc, ntok, prec):
    L = _ffi.lib()
    fn = getattr(L, f"lac_{coder_name}_encode_adaptive")
    for t0, t1 in _cuts(rng, R.T):
        n = _piece(ntok, t0, t1)
        _ffi.check(fn(R.ecounts[1:].data_ptr(), R.V, inc, d_syms.data_ptr() + 4 * t0, R.T + 2, R.S, t1 - t0,
                      n.data_ptr(), R.enc[1:].data_ptr(), R.out[1:].data_ptr(), R.cap, 0, prec, _stream()))


def flush_call(coder_name, R, inc, finish, prec):
    fn = getattr(_ffi.lib(), f"lac_{coder_name}_encode_adaptive")
    _ffi.check(fn(R.ecounts[1:].data_ptr(), R.V, inc, None, 0, R.S, 0, None, R.enc[1:].data_ptr(),
                  R.out[1:].data_ptr(), R.cap, finish, prec, _stream()))


def decode_calls(rng, coder_name, R, streams, inc, dntok, prec):
    L = _ffi.lib()
    fn = getattr(L, f"lac_{coder_name}_decode_adaptive")
    offs = np.zeros(R.S + 1, dtype=np.int64)
    np.cumsum([len(b) for b in streams], out=offs[1:])
    data = _dev(np.frombuffer(b"".join(streams) + b"\0" * 16, dtype=np.uint8).copy())
    d_offs = _dev(offs)
    _ffi.check(L.lac_dec_init(R.dec[1:].data_ptr(), R.S, prec, data.data_ptr(), d_offs.data_ptr(), _stream()))
    for t0, t1 in _cuts(rng, R.T):
        n = _piece(dntok, t0, t1)
        _ffi.check(fn(R.dcounts[1:].data_ptr(), R.V, inc, R.S, t1 - t0, n.data_ptr(), R.dec[1:].data_ptr(),
                      data.data_ptr(), d_offs.data_ptr(), R.back[1:].data_ptr() + 4 * t0, R.T + 3, prec, _stream()))
    return R.decoded(dntok)


# ------------------------------------------------------------------------------------------------ goldens
def test_golden_ac_adaptive_16k_from_counts(golden_dir):
    """ac_adaptive.npz: the byte model from ones with inc 1 at prec 32, encoded to the golden bytes and decoded back
    from the stream alone: no tables, no plaintext."""
    g = _golden(golden_dir, "ac_adaptive.npz")
    data = g["data"]
    T, prec = len(data), int(g["prec"])
    counts = coder.Counts(1, 256)
    enc = coder.StreamEncoder(1, prec=prec, capacity_bytes=T * 2)
    enc.encode_adaptive(_dev(data.astype(np.int32)[None]), counts, finish=True)
    streams, _ = enc.bitstreams()
    assert streams[0] == g["comp"].tobytes()
    want = 1 + np.bincount(data, minlength=256)
    assert np.array_equal(counts.counts.cpu().numpy()[0], want)
    dcounts = coder.Counts(1, 256)
    out = coder.StreamDecoder([g["comp"].tobytes()], prec=prec).decode_adaptive(dcounts, T).cpu().numpy()[0]
    assert np.array_equal(out, data)
    assert np.array_equal(dcounts.counts.cpu().numpy()[0], want)


def test_golden_acs_64k_config0_from_counts(golden_dir):
    """acs_64k.npz (configs[0]): ACSampler with the byte model reproduces the golden bytes; with the safe termination
    all 65536 bytes decode back, and the reference-flushed stream decodes all but at most its last 8."""
    g = _golden(golden_dir, "acs_64k.npz")
    data = g["data"]
    T, prec = len(data), int(g["prec"])
    d_syms = _dev(data.astype(np.int32)[None])
    enc = coder.StreamEncoder(1, prec=prec, capacity_bytes=T)
    enc.acs_encode_adaptive(d_syms, coder.Counts(1, 256), finish=True)
    streams, _ = enc.bitstreams()
    assert streams[0] == g["comp"].tobytes()
    enc2 = coder.StreamEncoder(1, prec=prec, capacity_bytes=T)
    enc2.acs_encode_adaptive(d_syms, coder.Counts(1, 256), finish="safe")
    s2, _ = enc2.bitstreams()
    dcounts = coder.Counts(1, 256)
    out = coder.StreamDecoder(s2, prec=prec).acs_decode_adaptive(dcounts, T).cpu().numpy()[0]
    assert np.array_equal(out, data)
    assert np.array_equal(dcounts.counts.cpu().numpy()[0], 1 + np.bincount(data, minlength=256))
    out1 = coder.StreamDecoder(streams, prec=prec).acs_decode_adaptive(coder.Counts(1, 256), T,
                                                                       check_status=False).cpu().numpy()[0]
    assert np.array_equal(out1[:-8], data[:-8])


# ------------------------------------------------------------------------------------------------ random cases
def draw_case(rng, acs, low=False):
    r = rng.random()
    if r < 0.3:
        V = int(rng.choice([1, 2, 3, 31, 32, 33, 255, 256, 257, 4095, 4096]))
    elif r < 0.8:
        V = int(rng.integers(1, 300))
    else:
        V = int(rng.integers(300, 4097))
    S = int(rng.choice([1, 2, 3, 4, 5, 7, 9, 31, 33, 40]))
    T = int(rng.integers(1, 300 if V <= 300 else 40))
    inc = int(rng.integers(0, 6))
    top = int(rng.choice([1, 3, 100, 10 ** 6]))
    init = rng.integers(0, top + 1, (S, V)).astype(np.int64)
    init[rng.random((S, V)) < float(rng.choice([0.0, 0.3]))] = 0
    for s in range(S):
        if not init[s].any():
            init[s, rng.integers(0, V)] = 1
    ntok = rng.integers(0, T + 1, S).astype(np.int32) if rng.random() < 0.6 else np.full(S, T, dtype=np.int32)
    syms = np.full((S, T + 2), 0x7FFF0000, dtype=np.int32)  # padding columns hold a symbol outside [0, V)
    for s in range(S):
        c = init[s].copy()
        for t in range(T):
            a = int(rng.choice(np.nonzero(c > 0)[0]))
            syms[s, t] = a
            if t < ntok[s]:
                c[a] += inc
    total = int(init.sum(axis=1).max()) + inc * T
    if acs:   # every token keeps a non-empty region: total <= the smallest span, 2^(prec - 2)
        lo = max(2, int(np.ceil(np.log2(total + 1))) + 3)
    else:     # widths >= 2 V, so fudged_dist is defined; low precisions take it once the total passes the width
        lo = max(2, int(np.ceil(np.log2(V))) + 3)
    if low:
        return V, S, T, inc, init, ntok, syms, lo
    prec = int(rng.integers(lo, min(60, lo + 8) + 1)) if rng.random() < 0.5 else int(rng.integers(lo, 61))
    return V, S, T, inc, init, ntok, syms, prec


def run_ac_case(rng, low=False):
    V, S, T, inc, init, ntok, syms, prec = draw_case(rng, acs=False, low=low)
    cap = (T + 3) * (prec + 2) // 8 + 16
    R = Rig(S, T, V, cap, init, prec)
    d_syms = _dev(syms)
    encode_calls(rng, "ac", R, d_syms, inc, ntok, prec)
    _, nb0, _, lh = R.streams()                    # before the flush: compared with the oracle's state
    flush_call("ac", R, inc, 1, prec)
    got, nbits, status, _ = R.streams()
    final = R.counts("enc")
    fudged = 0
    for s in range(S):
        n = int(ntok[s])
        tabs, minp, want_counts = walk(init[s], syms[s, :n], inc)
        fudged += int((tabs[:n, -1] > (1 << prec) * minp[:n]).any())  # past every width: fudged
        bits, st = orc.ac_encode(tabs, syms[s, :n], prec=prec, stop=1, minp=minp, return_state=True)
        case = (V, S, T, inc, prec, s)
        assert status[s] == 0, case + (status[s],)
        assert got[s] == _packed(bits) and int(nbits[s]) == len(bits), case
        assert (int(lh[s, 0]), int(lh[s, 1]), int(nb0[s])) == (int(st[0]), int(st[1]), int(st[2])), case
        assert np.array_equal(final[s], want_counts), case
    back, dstatus = decode_calls(rng, "ac", R, got, inc, ntok, prec)
    for s in range(S):
        n = int(ntok[s])
        assert np.array_equal(back[s, :n], syms[s, :n]) and dstatus[s] == 0, (V, S, T, inc, prec, s)
    assert np.array_equal(R.counts("dec"), final)
    return fudged


def run_acs_case(rng):
    V, S, T, inc, init, ntok, syms, prec = draw_case(rng, acs=True)
    cap = (T + 3) * (prec + 2) // 8 + 16
    R = Rig(S, T, V, cap, init, prec)
    encode_calls(rng, "acs", R, _dev(syms), inc, ntok, prec)
    out0, enc0 = R.out.clone(), R.enc.clone()
    flush_call("acs", R, inc, 1, prec)             # flush_compress: bit-exact with the oracle
    got, nbits, status, _ = R.streams()
    final = R.counts("enc")
    for s in range(S):
        n = int(ntok[s])
        tabs, _, want_counts = walk(init[s], syms[s, :n], inc)
        bits = orc.acs_encode(tabs.view(np.uint64), syms[s, :n], prec=prec, flush=1)
        case = (V, S, T, inc, prec, s)
        assert status[s] == 0 and got[s] == _packed(bits) and int(nbits[s]) == len(bits), case
        assert np.array_equal(final[s], want_counts), case
    R.out.copy_(out0)                              # the same streams, ended with the safe termination instead
    R.enc.copy_(enc0)
    flush_call("acs", R, inc, 2, prec)
    safe, _, status, _ = R.streams()
    assert (status == 0).all()
    assert np.array_equal(R.counts("enc"), final)  # a flush-only call leaves the counts alone
    back, dstatus = decode_calls(rng, "acs", R, safe, inc, ntok, prec)
    for s in range(S):
        n = int(ntok[s])
        assert np.array_equal(back[s, :n], syms[s, :n]) and dstatus[s] == 0, (V, S, T, inc, prec, s)
    assert np.array_equal(R.counts("dec"), final)


@pytest.mark.parametrize("seed", range(12))
def test_ac_adaptive_random(seed):
    rng = np.random.default_rng(7100 + seed)
    for _ in range(6):
        run_ac_case(rng)


def test_ac_adaptive_random_lowest_precision_reaches_fudged_dist():
    """The lowest precision each vocabulary allows: the totals outgrow the width and fudged_dist codes."""
    rng = np.random.default_rng(7200)
    assert sum(run_ac_case(rng, low=True) for _ in range(10)) > 0, "no stream reached fudged_dist"


@pytest.mark.parametrize("seed", range(8))
def test_acs_adaptive_random(seed):
    rng = np.random.default_rng(7300 + seed)
    for _ in range(6):
        run_acs_case(rng)


# ------------------------------------------------------------------------------------------------ inc = 0
@pytest.mark.parametrize("prec", [12, 32, 48])
def test_inc_zero_is_the_static_table(prec):
    """inc = 0 codes every token on the same table: the bytes, states and symbols of encode_tables /
    acs_encode_tables on that shared table."""
    rng = np.random.default_rng(prec)
    S, T, V = 7, 80, 300
    counts = rng.integers(0, 50, V).astype(np.int64)
    counts[rng.random(V) < 0.2] = 0
    counts[3] = 1
    dist = np.cumsum(counts)
    pos = np.nonzero(counts)[0]
    syms = _dev(rng.choice(pos, (S, T)).astype(np.int32))
    minp = int(counts[counts > 0].min())
    a = coder.StreamEncoder(S, prec=prec, capacity_bytes=T * 8 + 64)
    a.encode_adaptive(syms, coder.Counts(S, V, init=counts, inc=0), finish=True)
    b = coder.StreamEncoder(S, prec=prec, capacity_bytes=T * 8 + 64)
    b.encode_tables(_dev(dist), syms, _dev(np.array([minp])), finish=True)
    assert torch.equal(a.out, b.out) and torch.equal(a.state, b.state)
    streams, _ = a.bitstreams()
    da = coder.StreamDecoder(streams, prec=prec).decode_adaptive(coder.Counts(S, V, init=counts, inc=0), T)
    db = coder.StreamDecoder(streams, prec=prec).decode_tables(_dev(dist), _dev(np.array([minp])), T)
    assert torch.equal(da, syms) and torch.equal(db, syms)
    if prec < 20:  # ACSampler needs total <= span
        return
    for finish in (True, "safe"):
        a = coder.StreamEncoder(S, prec=prec, capacity_bytes=T * 8 + 64)
        a.acs_encode_adaptive(syms, coder.Counts(S, V, init=counts, inc=0), finish=finish)
        b = coder.StreamEncoder(S, prec=prec, capacity_bytes=T * 8 + 64)
        b.acs_encode_tables(_dev(dist), syms, finish=finish)
        assert torch.equal(a.out, b.out) and torch.equal(a.state, b.state)
    streams, _ = a.bitstreams()
    da = coder.StreamDecoder(streams, prec=prec).acs_decode_adaptive(coder.Counts(S, V, init=counts, inc=0), T)
    assert torch.equal(da, syms)


# ------------------------------------------------------------------------------------------------ bad tokens
@pytest.mark.parametrize("coder_name", ["ac", "acs"])
def test_bad_tokens_stop_only_their_stream(coder_name):
    """A symbol out of range (LAC_ST_SYMBOL), a zero-count symbol, an all-zero table and a negative count
    (LAC_ST_TABLE) each stop only their own stream.  That stream keeps the bits, state and counts of the tokens before
    the bad one (a negative count: nothing coded, counts untouched); the other streams stay bit-exact and decode."""
    rng = np.random.default_rng(41 if coder_name == "ac" else 42)
    V, S, T, prec, inc = 256, 9, 6, 40, 3
    init = rng.integers(1, 20, (S, V)).astype(np.int64)
    syms = np.full((S, T + 2), 0x7FFF0000, dtype=np.int32)
    syms[:, :T] = rng.integers(0, V, (S, T))
    syms[1, 3] = V                       # out of range at token 3
    init[3, 17] = 0
    syms[3, :T][syms[3, :T] == 17] = 18
    syms[3, 2] = 17                      # zero count at token 2
    init[5] = 0                          # all-zero table at token 0
    init[7, 5] = -1                      # negative count: the table does not load
    bad = {1: (3, _ffi.LAC_ST_SYMBOL), 3: (2, _ffi.LAC_ST_TABLE), 5: (0, _ffi.LAC_ST_TABLE),
           7: (0, _ffi.LAC_ST_TABLE)}
    ntok = np.full(S, T, dtype=np.int32)
    cap = (T + 3) * (prec + 2) // 8 + 16
    R = Rig(S, T, V, cap, init, prec)
    encode_calls(rng, coder_name, R, _dev(syms), inc, ntok, prec)
    out0, enc0 = R.out.clone(), R.enc.clone()
    flush_call(coder_name, R, inc, 1, prec)
    got, nbits, status, lh = R.streams()
    final = R.counts("enc")
    for s in range(S):
        n, want_status = bad.get(s, (T, 0))
        tabs, minp, want_counts = walk(np.maximum(init[s], 0), syms[s, :n], inc)
        stop = 0 if s in bad else 1
        if coder_name == "ac":
            bits, st = orc.ac_encode(tabs, syms[s, :n], prec=prec, stop=stop, minp=minp, return_state=True)
            if s in bad:
                assert (int(lh[s, 0]), int(lh[s, 1])) == (int(st[0]), int(st[1])), s
        else:
            bits = orc.acs_encode(tabs.view(np.uint64), syms[s, :n], prec=prec, flush=stop)
        assert status[s] == want_status, (s, status[s])
        assert got[s] == _packed(bits) and int(nbits[s]) == len(bits), s
        assert np.array_equal(final[s], init[s] if s == 7 else want_counts), s
    if coder_name == "acs":
        # flush_compress does not pin the final region, so decode the same streams ended with the safe termination
        R.out.copy_(out0)
        R.enc.copy_(enc0)
        flush_call(coder_name, R, inc, 2, prec)
        got, _, status2, _ = R.streams()
        assert np.array_equal(status2, status)
    # decode: the two streams whose tables do not serve decode nothing and are flagged; the rest decode back
    dntok = np.array([0 if s in (1, 3) else T for s in range(S)], dtype=np.int32)
    streams = [b"" if s in bad else got[s] for s in range(S)]
    back, dstatus = decode_calls(rng, coder_name, R, streams, inc, dntok, prec)
    dfinal = R.counts("dec")
    for s in range(S):
        if s in (5, 7):
            assert dstatus[s] == _ffi.LAC_ST_TABLE, (s, dstatus[s])
            continue
        assert dstatus[s] == 0, (s, dstatus[s])
        if s not in bad:
            assert np.array_equal(back[s, :T], syms[s, :T]) and np.array_equal(dfinal[s], final[s]), s
    assert np.array_equal(dfinal[7], init[7])


# ------------------------------------------------------------------------------------------------ mirror API
def test_mirror_count_predictor_one_call_each_way(golden_dir, monkeypatch):
    """AC(CountPredictor(256), 32) compresses the 16 KB golden to its bytes and decompresses all of it in one adaptive
    decode call: the per-symbol table path raises if it is reached."""
    g = _golden(golden_dir, "ac_adaptive.npz")
    data = g["data"].astype(int).tolist()
    p = ac.CountPredictor(256)
    assert ac.AC(p, 32).to_bin.compress(data) == g["comp"].tobytes()
    want = (1 + np.bincount(data, minlength=256)).tolist()
    assert p.counts == want

    def no_tables(*a, **k):
        raise AssertionError("per-symbol table path")

    calls = []
    real = coder.StreamDecoder.decode_adaptive

    def counted(self, *a, **k):
        calls.append(1)
        return real(self, *a, **k)

    monkeypatch.setattr(coder.StreamDecoder, "decode_tables", no_tables)
    monkeypatch.setattr(coder.StreamDecoder, "decode_adaptive", counted)
    q = ac.CountPredictor(256)
    assert ac.AC(q, 32).from_bin.decompress(g["comp"].tobytes(), len(data)) == data
    assert len(calls) == 1 and q.counts == want


def test_mirror_count_predictor_outside_the_device_bounds_takes_the_table_path():
    rng = np.random.default_rng(3)
    data = rng.integers(0, 5000, 25).tolist()
    p = ac.CountPredictor(5000, inc=2)
    comp = ac.AC(p, 32).to_bin.compress(data)
    tabs, minp, want = walk(np.ones(5000, dtype=np.int64), data, 2)
    assert comp == _packed(orc.ac_encode(tabs, data, prec=32, stop=1, minp=minp))
    assert p.counts == want.tolist()
    q = ac.CountPredictor(5000, inc=2)
    assert ac.AC(q, 32).from_bin.decompress(comp, len(data)) == data and q.counts == want.tolist()
