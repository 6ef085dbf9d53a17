"""The reference-facing Python API (same names as arith_code.py / arithmetic_coding.py /
llama_compress.py).  CPU part: table walking and bit packing.  GPU part: the mirrors produce the
reference's golden bits."""
import os

import numpy as np
import pytest

from lac_b200 import arith_code as ac
from lac_b200 import arithmetic_coding as acs


class AdaptiveCounts(ac.ProbPredictor):
    """Same 'simple adaptive frequency model' the goldens were made with (tests/golden/make_golden.py)."""

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


def test_materialise_tables_walks_like_receive_symbol():
    dist, minp = ac.materialise_tables(AdaptiveCounts(4), [2, 2, 0])
    assert dist.tolist() == [[1, 2, 3, 4], [1, 2, 4, 5], [1, 2, 5, 6]]
    assert minp.tolist() == [1, 1, 1]
    d, m = ac.materialise_tables(ac.CDFPredictor([3, 5, 6, 10]), [0, 3])
    assert d.tolist() == [[3, 5, 6, 10]] * 2 and m.tolist() == [1, 1]


def test_bit_packing_matches_reference_layout():
    from oracle import oracle as orc
    rng = np.random.default_rng(0)
    for n in (0, 1, 7, 8, 9, 77):
        bits = rng.integers(0, 2, n).tolist()
        assert bytes(ac.group_bits(bits)) == orc.pack_bits(np.array(bits, dtype=np.uint8)).tobytes()
        assert list(ac.ungroup_bits(bytes(ac.group_bits(bits))))[:n] == bits
        out = bytearray()
        pk = acs.packbits(out.append)
        for b in bits:
            pk(b)
        pk.flush()
        assert bytes(out) == bytes(ac.group_bits(bits))
        assert list(acs.unpackbits(out))[:n] == bits


def test_scaled_cdf_is_the_reference_expression():
    from oracle import ref_quant
    p = np.random.default_rng(1).dirichlet(np.ones(50))
    assert np.array_equal(acs.ACSampler(48).scaled_cdf(p), ref_quant.acs_cdf(p, 48))


# ------------------------------------------------------------------ GPU
torch = pytest.importorskip("torch")
gpu = pytest.mark.gpu
needs_gpu = pytest.mark.skipif(not torch.cuda.is_available(), reason="no CUDA device")


@gpu
@needs_gpu
def test_mirror_ac_on_goldens(ac_small):
    """Every ac_small golden (696 cases): whole-sequence bits / encode, counted decode."""
    g = ac_small
    for nm in list(g["names"]):
        prec, stop = int(g[f"{nm}/prec"]), int(g[f"{nm}/stop"])
        dist, syms = [int(x) for x in g[f"{nm}/dist"]], [int(x) for x in g[f"{nm}/syms"]]
        coder_ = ac.AC(ac.CDFPredictor(dist), prec)
        want = [int(b) for b in g[f"{nm}/bits"]]
        assert list(coder_.to_bin.bits(syms, stop)) == want, nm
        r, n = coder_.to_bin.encode(syms, stop)
        assert n == len(want) and r == int("0" + "".join(map(str, want)), 2)
        if stop and syms:
            assert list(coder_.from_bin.run(want, stop, count=len(syms))) == syms, nm


@gpu
@needs_gpu
def test_mirror_default_coder_is_the_uniform_ternary_predictor(golden_dir):
    """The reference's AC() is AC(Predictor(3), 16): same defaults, same bits, same round trip here (all 240)."""
    assert ac.AC().predictor.n == 3 and ac.AC().precision == 16
    g = np.load(os.path.join(golden_dir, "ac_uniform.npz"))
    n_default = 0
    for nm in list(g["names"]):
        prec, stop, n = int(g[f"{nm}/prec"]), int(g[f"{nm}/stop"]), int(g[f"{nm}/n"])
        syms = [int(x) for x in g[f"{nm}/syms"]]
        want = [int(b) for b in g[f"{nm}/bits"]]
        coder_ = ac.AC() if (n, prec) == (3, 16) else ac.AC(ac.Predictor(n), prec)
        n_default += (n, prec) == (3, 16)
        assert list(coder_.to_bin.bits(syms, stop)) == want, nm
        if stop and syms:
            assert list(coder_.from_bin.run(want, stop, count=len(syms))) == syms, nm
    assert n_default >= 2


def _trace_predictor(g, nm):
    kind, V = str(g[f"{nm}/kind"]), int(g[f"{nm}/V"])
    if kind == "cdf":
        return ac.CDFPredictor([int(x) for x in g[f"{nm}/dist"]])
    if kind == "uniform":
        return ac.Predictor(V)
    return AdaptiveCounts(V)


def _ragged(g, nm, key):
    flat, off = g[f"{nm}/{key}"], g[f"{nm}/{key}_off"]
    return [tuple(int(x) for x in flat[off[i]:off[i + 1]]) for i in range(len(off) - 1)]


@gpu
@needs_gpu
def test_incremental_encoder_follows_the_reference_call_by_call(golden_dir):
    """tests/golden/api_traces.npz holds what the REFERENCE returns call by call.  A_to_bin.__call__(symbol) must
    return the same digit tuples (the deferred-carry 2s and 3s included) and leave the same (l, h, emitted_bits,
    certain, info, total_encoded_entropy); __call__(None) flushes: same digits after carry resolution, same reset."""
    g = np.load(os.path.join(golden_dir, "api_traces.npz"))
    saw_carry = False
    for nm in list(g["names"]):
        prec = int(g[f"{nm}/prec"])
        syms = [int(x) for x in g[f"{nm}/syms"]]
        digits, states = _ragged(g, nm, "digits"), g[f"{nm}/enc_states"]
        enc = ac.AC(_trace_predictor(g, nm), prec).to_bin
        for i, sy in enumerate(syms):
            got = enc(sy)
            assert got == digits[i], (nm, i, got, digits[i])
            saw_carry |= any(d > 1 for d in got)
            assert [enc.l, enc.h, enc.emitted_bits, int(enc.certain)] == states[i].tolist(), (nm, i)
        assert abs(enc.info - float(g[f"{nm}/info"])) < 1e-9
        assert abs(enc.total_encoded_entropy - float(g[f"{nm}/total_encoded_entropy"])) < 1e-9
        fl, want = enc(None), digits[-1]
        assert len(fl) == len(want), nm
        assert sum(d << (len(fl) - 1 - i) for i, d in enumerate(fl)) == sum(d << (len(want) - 1 - i) for i, d in enumerate(want))
        assert [enc.l, enc.h, enc.emitted_bits, int(enc.certain)] == states[-1].tolist(), nm
        # the carry-resolving generator over an ITERATOR (no length: the incremental path) and encode()
        want_bits = [int(b) for b in g[f"{nm}/bits"]]
        assert list(ac.AC(_trace_predictor(g, nm), prec).to_bin.bits(iter(syms), 1)) == want_bits, nm
        e2 = ac.AC(_trace_predictor(g, nm), prec).to_bin
        e2(syms[0])
        r, n = e2.encode(iter(syms[1:]), 1)          # continues the stream the first call started
        first = len(digits[0])
        assert n == len(want_bits) - first, nm
    assert saw_carry


@gpu
@needs_gpu
def test_incremental_decoder_follows_the_reference_bit_by_bit(golden_dir):
    """A_from_bin.__call__(bit) returns the symbols that bit determines -- the same tuples, after the same bits, as
    the reference -- and (l, h, lb, hb) follow the reference's; run(bits) without a count yields every coded symbol."""
    g = np.load(os.path.join(golden_dir, "api_traces.npz"))
    for nm in list(g["names"]):
        if str(g[f"{nm}/dec_err"]):
            continue
        prec = int(g[f"{nm}/prec"])
        syms = [int(x) for x in g[f"{nm}/syms"]]
        bits = [int(b) for b in g[f"{nm}/bits"]]
        outs, states = _ragged(g, nm, "dec_out"), g[f"{nm}/dec_states"]
        dec = ac.AC(_trace_predictor(g, nm), prec).from_bin
        for j, b in enumerate(bits):
            got = dec(b)
            assert got == outs[j], (nm, j, got, outs[j])
            assert [dec.l, dec.h, dec.lb, dec.hb] == states[j].tolist(), (nm, j)
        got = list(ac.AC(_trace_predictor(g, nm), prec).from_bin.run(bits, 1))
        assert got[: len(syms)] == syms, nm


@gpu
@needs_gpu
def test_mirror_adaptive_model_matches_reference_bytes(golden_dir):
    g = np.load(os.path.join(golden_dir, "ac_adaptive.npz"))
    data = g["data"].tolist()
    coder_ = ac.AC(AdaptiveCounts(256), int(g["prec"]))
    comp = coder_.to_bin.compress(data)
    assert comp == g["comp"].tobytes()
    head = coder_.from_bin.decompress(comp, 300)   # adaptive decode is one GPU call per symbol
    assert head == data[:300]


@gpu
@needs_gpu
def test_measure_compress_is_the_reference_call_sequence(golden_dir):
    """arith_code.py:401-420 run as the reference's own golden generator runs it (tests/golden/make_golden.py:
    measure_compress(coder.to_bin, list(data), ...)): the input is consumed through a generator, one GPU step per
    symbol, progress lines use total_encoded_entropy.  First 1500 bytes of the 16 KB golden."""
    import io
    g = np.load(os.path.join(golden_dir, "ac_adaptive.npz"))
    data = g["data"].tolist()[:1500]
    log = io.StringIO()
    saved = []
    comp = ac.measure_compress(ac.AC(AdaptiveCounts(256), int(g["prec"])).to_bin, data, print_every_out=500,
                               print_every_inp=500, save_bits=saved, out=log)
    assert comp == ac.AC(AdaptiveCounts(256), int(g["prec"])).to_bin.compress(data)
    assert bytes(ac.group_bits(saved)) == comp and "bits/tok" in log.getvalue()
    # the prefix of the full golden stream, up to the bits the flush touches
    full = g["comp"].tobytes()
    assert comp[: len(comp) - 8] == full[: len(comp) - 8]


@gpu
@needs_gpu
def test_mirror_acsampler_on_goldens(golden_dir):
    g = np.load(os.path.join(golden_dir, "acs_small.npz"))
    from oracle import oracle as orc
    for nm in list(g["names"]):
        prec, cdf, toks = int(g[f"{nm}/prec"]), g[f"{nm}/cdf"], g[f"{nm}/toks"].tolist()
        s = acs.ACSampler(prec)
        assert s.compress(cdf, toks) == orc.pack_bits(g[f"{nm}/bits"]).tobytes()
        assert s.last_nbits == len(g[f"{nm}/bits"])
        assert s.expand(cdf, s.compress(cdf, toks, flush="safe"), len(toks)) == toks


@gpu
@needs_gpu
def test_acsampler_callback_protocol(golden_dir):
    """The reference's own driving loops (arithmetic_coding.py:234-266 compress side, :268-300 expand side) against
    the mirror: compress_tokens / compress_output / on_compress_done / bits_per_token / flush_compress, then
    decompress_bits / decompress_output / on_decompress_done."""
    g = np.load(os.path.join(golden_dir, "api_traces.npz"))
    for nm in list(g["acs_names"]):
        prec, cdfs, toks = int(g[f"{nm}/prec"]), g[f"{nm}/cdf"], g[f"{nm}/toks"].tolist()
        n = len(toks)
        s = acs.ACSampler(prec)
        out, bpt = [], []
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
            s.sample_scaled_cdf(cdfs[min(i, n - 1)])
            i += 1
        assert out == g[f"{nm}/bits"].tolist(), nm                       # the reference's bits, in order
        assert np.allclose(bpt, g[f"{nm}/bits_per_token"], atol=1e-6), nm  # and its per-token entropies
        # expand with the callback protocol; the bit source is an iterator that is consumed lazily
        d = acs.ACSampler(prec)
        pulled = [0]

        def counting(bits):
            for b in bits:
                pulled[0] += 1
                yield b
        d.decompress_bits = counting(out)
        got = []
        d.decompress_output = got.append
        fired = []
        d.on_decompress_done = lambda: fired.append(1)
        for i in range(n):
            d.sample_scaled_cdf(cdfs[i])
        # (the reference's own expand path fails or mis-decodes on some of these streams; see DESIGN.md section 6)
        want = toks
        tail_ok = got[: n - 3] == want[: n - 3]
        assert tail_ok, nm
        assert pulled[0] <= len(out)
    # sample(pdf): the reference's table construction in front of the same path
    s = acs.ACSampler(48)
    out = []
    s.compress_tokens = [3, 1, 4, 1, 5]
    s.compress_output = acs.packbits(out.append)

    def done2():
        s.on_compress_done = None
        s.flush_compress()
        s.compress_output.flush()
        s.compress_output = None
    s.on_compress_done = done2
    while not s.compress_done:
        s.sample(np.ones(10))
    ref = acs.ACSampler(48)
    assert bytes(out) == ref.compress(ref.scaled_cdf(np.ones(10)), [3, 1, 4, 1, 5])


class FakeLlm:
    """Stands in for llama_cpp.Llama (the same stand-in tests/golden/make_golden.py drives the real reference with)."""

    def __init__(self, logits, n_ctx=1 << 30):
        self.logits, self._n_ctx = logits, n_ctx
        self.reset()

    def reset(self):
        self.pos, self._scores = -1, None

    def eval(self, toks):
        self.pos += len(toks)
        k = min(self.pos, len(self.logits) - 1)
        self._scores = self.logits[k:k + 1]

    def n_ctx(self):
        return self._n_ctx


@gpu
@needs_gpu
def test_llama_ac_predictor_routes_to_lq32(golden_dir):
    """AC(Llama_AC(llm), 48) as llama_compress.py:4-10 builds it, on the logits of the ac_llama goldens: the
    incremental coder, the whole-sequence coder and the batched StreamEncoder produce the same LQ32 stream, the
    open-ended decoder returns the symbols.  (The stream is NOT the reference's: its re-scaled tables wrap int64 and
    are nearly uniform, DESIGN.md section 1.)"""
    from lac_b200 import coder, llama_compress as lc
    g = np.load(os.path.join(golden_dir, "ac_llama.npz"))
    for nm in list(g["names"]):
        logits, syms = g[f"{nm}/logits"], [int(x) for x in g[f"{nm}/syms"]]
        T = len(syms)
        enc = ac.AC(lc.Llama_AC(FakeLlm(logits)), 48).to_bin
        digits = [enc(s) for s in syms] + [enc(None)]
        inc_bits = list(ac.AC(lc.Llama_AC(FakeLlm(logits)), 48).to_bin.bits(iter(syms), 1))
        assert sum(len(d) for d in digits) == len(inc_bits)
        bulk = ac.AC(lc.Llama_AC(FakeLlm(logits)), 48).to_bin.compress(syms)
        assert bytes(ac.group_bits(inc_bits)) == bulk
        se = coder.StreamEncoder(1)
        se.encode_logits(torch.from_numpy(logits[:T]).cuda().unsqueeze(0), torch.tensor([syms], dtype=torch.int32).cuda(),
                         finish=True)
        assert se.bitstreams()[0][0] == bulk
        got = list(ac.AC(lc.Llama_AC(FakeLlm(logits)), 48).from_bin.run(inc_bits, 1))
        assert got[:T] == syms
        assert ac.AC(lc.Llama_AC(FakeLlm(logits)), 48).from_bin.decompress(bulk, T) == syms
        tab = lc.Llama_AC(FakeLlm(logits)).calc_dist()
        assert int(tab[-1]) == 1 << 32 and (np.diff(np.concatenate([[0], tab])) >= 1).all()


@gpu
@needs_gpu
@pytest.mark.parametrize("use_graphs", [True, False])
def test_llama_compress_roundtrip_and_size(use_graphs):
    """configs[2] in miniature: Llama-style random-init model, vocab 32000, ragged chunks, full-shape batches (the
    last one padded with empty streams), container; per-token step replayed from a CUDA graph."""
    from lac_b200 import container, llama_compress as lc
    chunk, B = 24, 4
    cfg = lc.LlamaConfig("t", 32000, 64, 2, 4, 2, 128, 64)
    model = lc.LlamaModel(cfg, n_streams=B, max_len=chunk, seed=3)
    rng = np.random.default_rng(5)
    toks = rng.integers(0, cfg.vocab, 5 * chunk + 7).astype(np.int32)
    comp = lc.LlamaCompressor(model, chunk_tokens=chunk, use_graphs=use_graphs)
    blob = comp.compress(toks)
    c = container.unpack(blob)
    assert c.n_chunks == 6 and c.ntok.tolist() == [chunk] * 5 + [7] and c.batch_streams == B
    back = comp.decompress(blob)
    assert np.array_equal(back, toks)
    # a second compressor instance (fresh graphs, same seed) reads the file, and writes the same file
    comp2 = lc.LlamaCompressor(lc.LlamaModel(cfg, n_streams=B, max_len=chunk, seed=3), chunk_tokens=chunk,
                               use_graphs=use_graphs)
    assert np.array_equal(comp2.decompress(blob), toks)
    assert comp2.compress(toks) == blob
    # random tokens under a random-init model (logit std ~3) cost about log2(V) + sigma^2 / (2 ln 2) ~ 21 bits each
    bits = float(c.nbits.sum())
    assert 0.9 * np.log2(cfg.vocab) * len(toks) < bits < 2.5 * np.log2(cfg.vocab) * len(toks)
    with pytest.raises(AssertionError):
        comp.compress(np.array([1, 2, cfg.vocab], dtype=np.int32))
    # a file for another predictor is refused, a damaged payload is reported
    other = lc.LlamaCompressor(lc.LlamaModel(lc.LlamaConfig("u", 32000, 64, 1, 4, 2, 128, 64), B, chunk, seed=3),
                               chunk_tokens=chunk, use_graphs=use_graphs)
    with pytest.raises(ValueError):
        other.decompress(blob)


@gpu
@needs_gpu
def test_llama_model_in_distribution_text_compresses():
    """Tokens SAMPLED from the model (in-distribution text) must cost about the model's entropy, far below
    log2(V): the coder is driven by the model, not by a uniform table."""
    import torch
    from lac_b200 import container, llama_compress as lc
    chunk, B = 32, 8
    cfg = lc.LlamaConfig("t", 32000, 64, 2, 4, 2, 128, 64)
    model = lc.LlamaModel(cfg, n_streams=B, max_len=chunk, seed=4)
    g = torch.Generator(device="cuda").manual_seed(0)
    model.reset()
    prev = torch.full((B,), lc.BOS, dtype=torch.int64, device="cuda")
    cols, ent = [], 0.0
    for t in range(chunk):
        logits = model.step(prev, lc._bucket_for(t, chunk))
        p = torch.softmax(logits.double(), -1)
        prev = torch.multinomial(p.float(), 1, generator=g).squeeze(1)
        ent += float(-(p * torch.log2(p.clamp_min(1e-300))).sum(-1).sum())
        cols.append(prev.to(torch.int32))
        model.pos.add_(1)
    toks = torch.stack(cols, 1).cpu().numpy().reshape(-1)
    comp = lc.LlamaCompressor(model, chunk_tokens=chunk, use_graphs=False)
    blob = comp.compress(toks)
    bits = float(container.unpack(blob).nbits.sum())
    assert bits < 1.25 * ent + 64 * B and bits < 0.8 * np.log2(cfg.vocab) * len(toks)
    assert np.array_equal(comp.decompress(blob), toks)
