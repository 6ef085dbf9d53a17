"""Randomised GPU parity of the integer-table coders (run with -m gpu on a B200), through the raw C ABI:
lac_ac_{en,de}code_tables (CDFPredictor, exact and wrap64), lac_acs_{en,de}code_tables (ACSampler) and
lac_ac_{en,de}code_uniform (Predictor(n)).  Per case the vocabulary (up to 128256), the precision (2 .. 60), the number
of streams (1 .. 40, across the four-warps-per-block and 32-threads-per-block edges), the table layout (padded
[S, T, V], shared [T, V], one table), ragged token counts and a split point are drawn; every stream is compared with
the oracle bit for bit (the oracle is pinned to an exact Python-int restatement by tests/test_exact_reference.py),
decoded back, and the buffers around every output are checked for stray writes."""
import collections

import numpy as np
import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():  # collected on CPU boxes, deselected by -m "not gpu"
    pytest.skip("no CUDA device", allow_module_level=True)

from lac_b200 import _ffi  # noqa: E402
from oracle import oracle as orc  # noqa: E402
from oracle import pyref, ref_quant  # noqa: E402

G = 0xA5          # guard byte
JUNK = -(1 << 61) + 12345  # fills table and minp padding: a coder that reads it codes differently
COUNTS = collections.Counter()  # cases run per coder x vocab class x prec class x layout


def count(coder, V, prec, layout):
    vc = "V<=256" if V <= 256 else ("V<5000" if V < 5000 else "V>=5000")
    pc = "prec<=33" if prec <= 33 else ("prec34-48" if prec <= 48 else "prec49-60")
    COUNTS[(coder, vc, pc, layout)] += 1


@pytest.fixture(scope="module", autouse=True)
def _report_counts():
    yield
    for k in sorted(COUNTS):
        print("cases", " ".join(k), COUNTS[k])


# ------------------------------------------------------------------------------------------------ case drawing
def draw_vocab(rng):
    r = rng.random()
    if r < 0.04:
        return int(rng.choice([32000, 128256]))
    if r < 0.3:
        return int(rng.choice([1, 2, 3, 31, 32, 33, 63, 64, 65, 256, 257]))
    if r < 0.8:
        return int(rng.integers(1, 300))
    return int(rng.integers(300, 5000))


def draw_shape(rng, V):
    big = V >= 20000
    S = int(rng.choice([1, 2, 3, 5])) if big else int(rng.choice([1, 3, 4, 5, 7, 9, 31, 33, 37, 40]))
    T = int(rng.integers(1, 4)) if big else int(rng.integers(1, 12 if V < 2000 else 5))
    return S, T


def draw_layout(rng, S, T, V):
    """(kind, ss, ts, mss, mts, table slots): table of (s, t) at s * ss + t * ts, its minp at s * mss + t * mts."""
    kind = str(rng.choice(["streams", "shared", "single"]))
    if kind == "streams":
        ts = V + int(rng.integers(1, 5))
        ss = T * ts + int(rng.integers(1, 3 * V + 2))
        mts = int(rng.choice([1, 2]))
        mss = T * mts + int(rng.integers(1, 4))
    elif kind == "shared":
        ss, ts, mss, mts = 0, V + int(rng.choice([0, 1, 3])), 0, int(rng.choice([1, 2]))
    else:
        ss = ts = mss = mts = 0
    return kind, ss, ts, mss, mts


def random_freqs(rng, V, total_log2, zero_frac):
    w = rng.exponential(1.0, V) ** float(rng.choice([1.0, 3.0]))
    w[rng.random(V) < zero_frac] = 0.0
    if not w.any():
        w[rng.integers(0, V)] = 1.0
    f = np.floor(w / w.sum() * float(2 ** total_log2)).astype(np.int64)
    if f.sum() == 0:
        f[int(np.argmax(w))] = 1
    return f


def fill_tables(rng, S, T, V, layout, make_row, guard_value):
    """Flat buffer with one table per slot the layout addresses; everything else holds guard_value."""
    kind, ss, ts, mss, mts = layout
    n_tab_len = (S - 1) * ss + (T - 1) * ts + V if kind != "single" else V
    flat = np.full(n_tab_len + 8, guard_value, dtype=np.int64)
    rows = {}
    for s in range(S if ss else 1):
        for t in range(T if ts else 1):
            row = make_row()
            flat[s * ss + t * ts: s * ss + t * ts + V] = row
            rows[(s, t)] = row
    return flat, rows


def table_of(rows, layout, s, t):
    _, ss, ts, _, _ = layout
    return rows[(s if ss else 0, t if ts else 0)]


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _state_words(state, S, words):
    return state[1:S + 1].cpu().numpy().view(np.int64).reshape(S, words)


class Buffers:
    """Encoder / decoder buffers with a guard row before and after, all filled with guard bytes."""

    def __init__(self, S, T, cap):
        self.S, self.T, self.cap = S, T, cap
        self.out = torch.full((S + 2, cap), G, dtype=torch.uint8, device="cuda")
        self.enc = torch.full((S + 2, _ffi.ENC_STATE_BYTES), G, dtype=torch.uint8, device="cuda")
        self.dec = torch.full((S + 2, _ffi.DEC_STATE_BYTES), G, dtype=torch.uint8, device="cuda")
        self.sym_stride = T + 3
        self.back = torch.full((S + 2, self.sym_stride), -7, dtype=torch.int32, device="cuda")

    def out_ptr(self):
        return self.out[1:].data_ptr()

    def enc_ptr(self):
        return self.enc[1:].data_ptr()

    def streams(self):
        """(bytes per stream, nbits, status); asserts nothing was written outside a stream's bytes or the state rows."""
        torch.cuda.synchronize()
        st = _state_words(self.enc, self.S, 4)
        host = self.out.cpu().numpy()
        assert (host[0] == G).all() and (host[self.S + 1] == G).all(), "bitstream buffer overrun"
        e = self.enc.cpu().numpy()
        assert (e[0] == G).all() and (e[self.S + 1] == G).all(), "encoder state overrun"
        got = []
        for s in range(self.S):
            used = (int(st[s, 2]) + 7) // 8
            assert (host[1 + s, used:] == G).all(), ("bytes written past the stream's end", s)
            got.append(host[1 + s, :used].tobytes())
        return got, st[:, 2].copy(), (st[:, 3] & 0xFFFFFFFF).copy()

    def decoder_input(self, streams):
        offs = np.zeros(self.S + 1, dtype=np.int64)
        np.cumsum([len(b) for b in streams], out=offs[1:])
        self.data = _dev(np.frombuffer(b"".join(streams) + b"\0" * 16, dtype=np.uint8).copy())
        self.offs = _dev(offs)
        return self.data.data_ptr(), self.offs.data_ptr()

    def decoded(self, ntok):
        torch.cuda.synchronize()
        got = self.back.cpu().numpy()
        assert (got[0] == -7).all() and (got[self.S + 1] == -7).all(), "symbol buffer overrun"
        d = self.dec.cpu().numpy()
        assert (d[0] == G).all() and (d[self.S + 1] == G).all(), "decoder state overrun"
        for s in range(self.S):
            assert (got[1 + s, int(ntok[s]):] == -7).all(), ("symbols written past the stream's token count", s)
        st = _state_words(self.dec, self.S, 5)
        return got[1:self.S + 1], (st[:, 4] & 0xFFFFFFFF).copy()


def _cuts(rng, T):
    """The tokens go in as one call or two calls split at a random point."""
    cut = int(rng.integers(0, T + 1)) if rng.random() < 0.6 else T
    return [(a, b) for a, b in ((0, cut), (cut, T)) if b > a]


def _ntok_piece(ntok, t0, t1):
    return _dev(np.clip(ntok - t0, 0, t1 - t0).astype(np.int32))


def _packed(bits):
    return orc.pack_bits(bits).tobytes()


# ------------------------------------------------------------------------------------------------ CDFPredictor tables
def draw_ac_case(rng, V=None, prec=None):
    V = V or draw_vocab(rng)
    S, T = draw_shape(rng, V)
    prec = prec or int(rng.choice([int(rng.integers(2, 61)), int(rng.integers(34, 61)), 48]))
    layout = draw_layout(rng, S, T, V)
    wrap = bool(rng.random() < 0.4)
    zero_frac = float(rng.choice([0.0, 0.0, 0.2, 0.6]))
    near = rng.random() < 0.5

    def row():
        e = int(np.clip(prec + rng.integers(-6, 7), 1, 62)) if near else int(rng.integers(1, 63))
        return np.cumsum(random_freqs(rng, V, e, zero_frac))

    ntok = rng.integers(0, T + 1, S).astype(np.int32) if rng.random() < 0.6 else np.full(S, T, dtype=np.int32)
    return dict(V=V, S=S, T=T, prec=prec, layout=layout, wrap=wrap, row=row, ntok=ntok)


def run_ac_case(rng, case, tables=None, minp_of=None, bad=None):
    """Encode (one or two calls, then a flush-only call) and decode one drawn case; returns per-stream outcomes.
    bad: {stream: symbol} codes that symbol at the stream's first token instead of a valid one."""
    V, S, T, prec, layout, wrap = (case[k] for k in ("V", "S", "T", "prec", "layout", "wrap"))
    kind, ss, ts, mss, mts = layout
    ntok = case["ntok"]
    L, st = _ffi.lib(), torch.cuda.current_stream().cuda_stream
    if tables is None:
        flat, rows = fill_tables(rng, S, T, V, layout, case["row"], JUNK)
    else:
        flat, rows = tables
    minp_of = minp_of or (pyref.llama_minp if wrap else pyref.cdf_minp)
    mlen = (S - 1) * mss + (T - 1) * mts + 1
    mflat = np.full(mlen + 4, JUNK, dtype=np.int64)
    for (s, t), r in rows.items():
        mflat[s * mss + t * mts] = minp_of(r.tolist())
    syms = np.full((S, T + 2), 0x7FFF0000, dtype=np.int32)  # padding columns hold a symbol outside [0, V)
    for s in range(S):
        for t in range(T):
            r = table_of(rows, layout, s, t)
            f = np.diff(np.concatenate([[0], r]))
            syms[s, t] = int(rng.choice(np.nonzero(f > 0)[0]))
    for s, v in (bad or {}).items():
        syms[s, 0] = v
    flags = _ffi.LAC_F_WRAP64 if wrap else 0
    count("ac_tables_wrap64" if wrap else "ac_tables", V, prec, kind)
    d_dist, d_minp, d_syms = _dev(flat), _dev(mflat), _dev(syms)
    cap = (T + 3) * (prec + 2) // 8 + 16
    B = Buffers(S, T, cap)
    _ffi.check(L.lac_enc_init(B.enc_ptr(), S, prec, st))
    for t0, t1 in _cuts(rng, T):
        n = _ntok_piece(ntok, t0, t1)
        _ffi.check(L.lac_ac_encode_tables(d_dist.data_ptr() + 8 * t0 * ts, V, ss, ts, d_minp.data_ptr() + 8 * t0 * mts,
                                          mss, mts, d_syms.data_ptr() + 4 * t0, T + 2, S, t1 - t0, n.data_ptr(),
                                          B.enc_ptr(), B.out_ptr(), cap, 0, prec, flags, st))
    _ffi.check(L.lac_ac_encode_tables(d_dist.data_ptr(), V, ss, ts, d_minp.data_ptr(), mss, mts, None, 0, S, 0, None,
                                      B.enc_ptr(), B.out_ptr(), cap, 1, prec, flags, st))       # flush-only call
    got, nbits, status = B.streams()
    want = []
    for s in range(S):
        n = int(ntok[s])
        tabs = np.stack([table_of(rows, layout, s, t) for t in range(max(n, 1))])
        mp = np.array([minp_of(tabs[t].tolist()) for t in range(len(tabs))], dtype=np.int64)
        try:
            bits = orc.ac_encode(tabs, syms[s, :n], prec=prec, stop=1, minp=mp, wrap64=wrap)
            want.append((_packed(bits), len(bits), 0))
        except orc.OracleError as e:
            want.append((None, None, _ffi.LAC_ST_SYMBOL if e.code == -3 else _ffi.LAC_ST_TABLE))
    for s in range(S):
        if want[s][0] is None:
            assert status[s] == want[s][2], (case_id(case), s, status[s])
            continue
        assert status[s] == 0, (case_id(case), s, status[s])
        assert got[s] == want[s][0] and int(nbits[s]) == want[s][1], (case_id(case), s)
    # decode what decodes, through the same layout, in one call or two
    ok = np.array([w[0] is not None for w in want])
    streams = [got[s] if ok[s] else b"" for s in range(S)]
    dntok = np.where(ok, ntok, 0).astype(np.int32)
    data, offs = B.decoder_input(streams)
    _ffi.check(L.lac_dec_init(B.dec[1:].data_ptr(), S, prec, data, offs, st))
    for t0, t1 in _cuts(rng, T):
        n = _ntok_piece(dntok, t0, t1)
        _ffi.check(L.lac_ac_decode_tables(d_dist.data_ptr() + 8 * t0 * ts, V, ss, ts, d_minp.data_ptr() + 8 * t0 * mts,
                                          mss, mts, S, t1 - t0, n.data_ptr(), B.dec[1:].data_ptr(), data, offs,
                                          B.back[1:].data_ptr() + 4 * t0, B.sym_stride, prec, flags, st))
    back, dstatus = B.decoded(dntok)
    for s in range(S):
        n = int(dntok[s])
        assert np.array_equal(back[s, :n], syms[s, :n]), (case_id(case), s)
        assert dstatus[s] == 0, (case_id(case), s, dstatus[s])
    return status


def case_id(case):
    return tuple(case[k] for k in ("V", "S", "T", "prec", "wrap")) + (case["layout"][0],)


@pytest.mark.parametrize("seed", range(16))
def test_ac_tables_random(seed):
    rng = np.random.default_rng(5000 + seed)
    for _ in range(12):
        run_ac_case(rng, draw_ac_case(rng))


def test_ac_tables_wide_vocab_fudged_and_high_precision():
    """Vocabularies past 256 in the fudged branch (every width, every prec), where the lane loops and the lane-block
    max-scan of the decoder's symbol search run many iterations per lane."""
    rng = np.random.default_rng(7)
    for i, (V, prec) in enumerate(((257, 60), (1000, 49), (4096, 55), (4099, 60), (32000, 59), (128256, 60),
                                   (128256, 50))):
        case = draw_ac_case(rng, V=V, prec=prec)
        case["wrap"] = bool(i % 2)

        def row():
            f = random_freqs(rng, V, 62, 0.3)
            f[rng.integers(0, V)] = 1     # minp 1, total ~2^62 > w: fudged at every width
            return np.cumsum(f)

        case["row"] = row
        run_ac_case(rng, case)


@pytest.mark.parametrize("wrap", [True, False])
def test_calc_dist_tables_at_32000(wrap):
    """The reference's own Llama_AC tables (calc_dist, llama_minp) at V = 32000: wrap64 restates it literally,
    wrap64 = 0 is exact CDFPredictor arithmetic on the same tables."""
    rng = np.random.default_rng(32000 + wrap)
    V, S, T = 32000, 5, 3
    layout = ("streams", T * V + 7, V, T, 1)
    flat = np.full((S - 1) * layout[1] + (T - 1) * V + V + 8, JUNK, dtype=np.int64)
    rows = {}
    for s in range(S):
        for t in range(T):
            r = ref_quant.calc_dist((rng.standard_normal(V) * float(rng.choice([1.0, 3.0, 8.0]))).astype(np.float32))
            flat[s * layout[1] + t * V: s * layout[1] + t * V + V] = r
            rows[(s, t)] = r
    case = dict(V=V, S=S, T=T, prec=48, layout=layout, wrap=wrap, ntok=np.array([3, 1, 3, 2, 0], dtype=np.int32))
    run_ac_case(rng, case, tables=(flat, rows), minp_of=lambda r: int(ref_quant.llama_minp(np.array(r))))


def test_ac_tables_bad_symbol_and_zero_width_stay_on_their_stream():
    """A symbol outside [0, V) sets LAC_ST_SYMBOL, a zero-width symbol LAC_ST_TABLE, each on its own stream only;
    the neighbouring streams (same warp-block, same tables) stay bit-exact and decode."""
    rng = np.random.default_rng(11)
    for kind in ("streams", "shared", "single"):
        for S in (5, 9, 33):
            V, T, prec = 300, 6, 40
            layout = {"streams": ("streams", T * (V + 2) + 5, V + 2, T + 1, 1),
                      "shared": ("shared", 0, V + 1, 0, 1), "single": ("single", 0, 0, 0, 0)}[kind]
            f = random_freqs(rng, V, 30, 0.0)
            f[17] = 0                                                  # unfudged (2^30 < 2^39 minp), zero-width 17
            row = np.cumsum(f)
            case = dict(V=V, S=S, T=T, prec=prec, layout=layout, wrap=False, row=lambda: row,
                        ntok=np.full(S, T, dtype=np.int32))
            status = run_ac_case(rng, case, bad={1: V, 3: -1, S - 1: 17})
            assert status[1] == _ffi.LAC_ST_SYMBOL and status[3] == _ffi.LAC_ST_SYMBOL
            assert status[S - 1] == _ffi.LAC_ST_TABLE
            assert (np.delete(status, [1, 3, S - 1]) == 0).all()


# ------------------------------------------------------------------------------------------------ Predictor(n)
def run_uniform_case(rng, n, prec, S, T, ntok, bad=None):
    L, st = _ffi.lib(), torch.cuda.current_stream().cuda_stream
    syms = np.full((S, T + 2), 0x7FFF0000, dtype=np.int32)
    syms[:, :T] = rng.integers(0, n, (S, T))
    for s, v in (bad or {}).items():
        syms[s, 0] = v
    d_syms = _dev(syms)
    count("uniform", n, prec, "none")
    cap = (T + 3) * (prec + 2) // 8 + 16
    B = Buffers(S, T, cap)
    _ffi.check(L.lac_enc_init(B.enc_ptr(), S, prec, st))
    for t0, t1 in _cuts(rng, T):
        nn = _ntok_piece(ntok, t0, t1)
        _ffi.check(L.lac_ac_encode_uniform(d_syms.data_ptr() + 4 * t0, S, t1 - t0, T + 2, nn.data_ptr(), n,
                                           B.enc_ptr(), B.out_ptr(), cap, 0, prec, st))
    _ffi.check(L.lac_ac_encode_uniform(None, S, 0, 0, None, n, B.enc_ptr(), B.out_ptr(), cap, 1, prec, st))
    got, nbits, status = B.streams()
    ok = np.ones(S, dtype=bool)
    for s in range(S):
        k = int(ntok[s])
        if s in (bad or {}) and k > 0:
            ok[s] = False
            assert status[s] == _ffi.LAC_ST_SYMBOL, (n, prec, S, s)
            continue
        bits = orc.ac_encode(orc.uniform(n), syms[s, :k], prec=prec, stop=1)
        assert status[s] == 0 and got[s] == _packed(bits) and int(nbits[s]) == len(bits), (n, prec, S, T, s)
    dntok = np.where(ok, ntok, 0).astype(np.int32)
    data, offs = B.decoder_input([got[s] if ok[s] else b"" for s in range(S)])
    _ffi.check(L.lac_dec_init(B.dec[1:].data_ptr(), S, prec, data, offs, st))
    for t0, t1 in _cuts(rng, T):
        nn = _ntok_piece(dntok, t0, t1)
        _ffi.check(L.lac_ac_decode_uniform(S, t1 - t0, nn.data_ptr(), n, B.dec[1:].data_ptr(), data, offs,
                                           B.back[1:].data_ptr() + 4 * t0, B.sym_stride, prec, st))
    back, dstatus = B.decoded(dntok)
    for s in range(S):
        assert np.array_equal(back[s, :int(dntok[s])], syms[s, :int(dntok[s])]) and dstatus[s] == 0, (n, prec, s)


@pytest.mark.parametrize("n", [2, 3, 255, 65536, 2 ** 31 - 1])
def test_uniform_random(n):
    rng = np.random.default_rng(n % 1000)
    for prec in range(2, 61):
        if n > 1 << (prec - 1):  # wider alphabets than half the range have zero-width symbols
            continue
        S = int(rng.choice([1, 5, 31, 33, 40]))
        T = int(rng.integers(1, 10))
        ntok = rng.integers(0, T + 1, S).astype(np.int32)
        bad = {int(rng.integers(0, S)): int(rng.choice([n, -1]))} if rng.random() < 0.3 else None
        run_uniform_case(rng, n, prec, S, T, ntok, bad)


# ------------------------------------------------------------------------------------------------ ACSampler
def run_acs_case(rng, V, prec, S, T, layout, finish, ntok, bad=None):
    L, st = _ffi.lib(), torch.cuda.current_stream().cuda_stream
    kind, ss, ts, _, _ = layout

    def row():
        return ref_quant.acs_cdf(rng.dirichlet(np.full(V, float(rng.choice([0.05, 0.5, 2.0])))), precision=prec)

    flat, rows = fill_tables(rng, S, T, V, layout, lambda: row().view(np.int64), JUNK)
    syms = np.full((S, T + 2), 0x7FFF0000, dtype=np.int32)
    for s in range(S):
        for t in range(T):  # symbols that keep a non-empty region at every width: frequency >= 3 on a total ~2^prec
            c = table_of(rows, layout, s, t).astype(object)
            f = np.diff(np.concatenate([[0], c]))
            syms[s, t] = int(rng.choice(np.nonzero(f >= 3)[0]))
    for s, v in (bad or {}).items():
        syms[s, 0] = v
    count(f"acs_finish{finish}", V, prec, kind)
    d_cdf, d_syms = _dev(flat), _dev(syms)
    cap = (T + 3) * (prec + 2) // 8 + 16
    B = Buffers(S, T, cap)
    _ffi.check(L.lac_enc_init(B.enc_ptr(), S, prec, st))
    for t0, t1 in _cuts(rng, T):
        nn = _ntok_piece(ntok, t0, t1)
        _ffi.check(L.lac_acs_encode_tables(d_cdf.data_ptr() + 8 * t0 * ts, V, ss, ts, d_syms.data_ptr() + 4 * t0, T + 2,
                                           S, t1 - t0, nn.data_ptr(), B.enc_ptr(), B.out_ptr(), cap, 0, prec, st))
    _ffi.check(L.lac_acs_encode_tables(d_cdf.data_ptr(), V, ss, ts, None, 0, S, 0, None, B.enc_ptr(), B.out_ptr(),
                                       cap, finish, prec, st))
    got, nbits, status = B.streams()
    ok = np.ones(S, dtype=bool)
    for s in range(S):
        k = int(ntok[s])
        if s in (bad or {}) and k > 0:
            ok[s] = False
            assert status[s] == _ffi.LAC_ST_SYMBOL, (V, prec, S, s)
            continue
        tabs = np.stack([table_of(rows, layout, s, t) for t in range(max(k, 1))]).view(np.uint64)
        if finish == 1:
            bits = orc.acs_encode(tabs, syms[s, :k], prec=prec, flush=1)
        else:
            bits = np.array(pyref.acs_encode([r.tolist() for r in tabs], syms[s, :k].tolist(), prec, finish=2),
                            dtype=np.uint8)
        assert status[s] == 0 and got[s] == _packed(bits) and int(nbits[s]) == len(bits), (V, prec, S, T, finish, s)
    if finish != 2:
        return
    dntok = np.where(ok, ntok, 0).astype(np.int32)
    data, offs = B.decoder_input([got[s] if ok[s] else b"" for s in range(S)])
    _ffi.check(L.lac_dec_init(B.dec[1:].data_ptr(), S, prec, data, offs, st))
    for t0, t1 in _cuts(rng, T):
        nn = _ntok_piece(dntok, t0, t1)
        _ffi.check(L.lac_acs_decode_tables(d_cdf.data_ptr() + 8 * t0 * ts, V, ss, ts, S, t1 - t0, nn.data_ptr(),
                                           B.dec[1:].data_ptr(), data, offs, B.back[1:].data_ptr() + 4 * t0,
                                           B.sym_stride, prec, st))
    back, dstatus = B.decoded(dntok)
    for s in range(S):
        assert np.array_equal(back[s, :int(dntok[s])], syms[s, :int(dntok[s])]) and dstatus[s] == 0, (V, prec, s)


@pytest.mark.parametrize("finish", [1, 2])
@pytest.mark.parametrize("seed", range(4))
def test_acs_tables_random(seed, finish):
    """ref_quant.acs_cdf tables up to prec 60: finish 1 (flush_compress) bit-exact with the oracle, finish 2 (safe
    termination) bit-exact with pyref and decoded back."""
    rng = np.random.default_rng(9000 + 10 * seed + finish)
    for _ in range(10):
        V = int(rng.choice([1, 2, 33, 257, 1000, 5000]))
        prec = int(rng.integers(max(8, int(np.log2(4 * V)) + 2), 61))
        S, T = int(rng.choice([1, 4, 7, 31, 33, 40])), int(rng.integers(1, 10))
        layout = draw_layout(rng, S, T, V)
        ntok = rng.integers(0, T + 1, S).astype(np.int32) if rng.random() < 0.6 else np.full(S, T, dtype=np.int32)
        bad = {int(rng.integers(0, S)): int(rng.choice([V, -1]))} if rng.random() < 0.3 else None
        run_acs_case(rng, V, prec, S, T, layout, finish, ntok, bad)
