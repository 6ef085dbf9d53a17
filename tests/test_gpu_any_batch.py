"""Batch-invariant files decoded at any batch size, on the GPU: the small-M GEMM path, the model at n <= S active
streams, and LlamaCompressor reading a batch-invariant file with decoders of other stream counts.

What is pinned: a row's bits do not depend on the launch size (M <= 128 takes a different GEMM tile than M > 128),
a stream's logits do not depend on how many streams run with it or in which slot, and so a packed read of any
range returns the source with each batch run at an active size from the ladder for exactly its needed steps."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():  # collected on CPU boxes, deselected by -m "not gpu"
    pytest.skip("no CUDA device", allow_module_level=True)

from lac_b200 import _ffi, container, sharding, llama_compress as lc  # noqa: E402

BF = torch.bfloat16


def _gemm(x, w, epi, res=None):
    M, (K, N) = x.shape[0], w.shape
    y = torch.empty((M, N), device="cuda", dtype=torch.float32 if epi == _ffi.LAC_MODEL_OUT_F32 else BF)
    _ffi.check(_ffi.lib().lac_model_gemm(x.data_ptr(), w.data_ptr(), M, N, K, epi,
                                         None if res is None else res.data_ptr(), y.data_ptr(),
                                         torch.cuda.current_stream().cuda_stream))
    return y


def _weight_shapes():
    shapes = set()
    for cfg in lc.CONFIGS.values():
        hd = cfg.dim // cfg.heads
        shapes |= {(cfg.dim, (cfg.heads + 2 * cfg.kv_heads) * hd), (cfg.dim, cfg.dim), (cfg.dim, 2 * cfg.ffn),
                   (cfg.ffn, cfg.dim), (cfg.dim, cfg.vocab)}
    return sorted(shapes)


@pytest.mark.parametrize("K,N", _weight_shapes())
def test_small_m_gemm_rows_equal_large_m_rows(K, N):
    g = torch.Generator(device="cuda").manual_seed(K * 3 + N)
    x = torch.randn((256, K), device="cuda", generator=g).to(BF)
    w = (torch.randn((K, N), device="cuda", generator=g) * K ** -0.5).to(BF)
    res = torch.randn((256, N), device="cuda", generator=g).to(BF)
    ref = x.float() @ w.float()
    for epi in (_ffi.LAC_MODEL_OUT_BF16, _ffi.LAC_MODEL_OUT_BF16_ADD, _ffi.LAC_MODEL_OUT_F32):
        r = res if epi == _ffi.LAC_MODEL_OUT_BF16_ADD else None
        full = _gemm(x, w, epi, r)                                   # M = 256: the 128 x 128 tile
        if epi == _ffi.LAC_MODEL_OUT_F32:
            torch.testing.assert_close(full, ref, atol=1e-3, rtol=1e-3)
        elif epi == _ffi.LAC_MODEL_OUT_BF16:
            torch.testing.assert_close(full.float(), ref, atol=2e-2, rtol=1e-2)
        else:
            torch.testing.assert_close(full.float(), res.float() + ref, atol=4e-2, rtol=1e-2)
        m200 = _gemm(x[20:220].contiguous(), w, epi, None if r is None else r[20:220].contiguous())
        assert torch.equal(m200, full[20:220]), epi
        for M, lo in ((1, 0), (1, 255), (5, 3), (64, 100), (127, 129), (128, 0), (128, 128)):
            part = _gemm(x[lo:lo + M].contiguous(), w, epi, None if r is None else r[lo:lo + M].contiguous())
            assert torch.equal(part, full[lo:lo + M]), (epi, M, lo)


def test_active_streams_ladder():
    assert [lc.active_streams(k, 8) for k in range(1, 9)] == [1, 2, 4, 4, 8, 8, 8, 8]
    assert [lc.active_streams(k, 6) for k in (1, 2, 3, 4, 5, 6)] == [1, 2, 4, 4, 6, 6]
    assert lc.active_streams(200, 256) == 256 and lc.active_streams(3, 3) == 3
    for bad in (0, 9):
        with pytest.raises(ValueError):
            lc.active_streams(bad, 8)


def test_stream_logits_do_not_depend_on_n_or_slot():
    cfg, T, S = lc.CONFIGS["tiny"], 80, 8
    m = lc.LlamaModel(cfg, n_streams=S, max_len=T, seed=11, batch_invariant=True)
    rng = np.random.default_rng(1)
    mine = torch.from_numpy(np.concatenate([[lc.BOS], rng.integers(0, cfg.vocab, T - 1)])).cuda()
    runs = {}
    for n, slot in ((1, 0), (3, 2), (8, 7)):
        inp = torch.from_numpy(rng.integers(0, cfg.vocab, (T, n))).cuda()   # the other streams: other text
        inp[:, slot] = mine
        m.reset()
        rows = []
        for t in range(T):
            rows.append(m.step(inp[t], T)[slot].clone())
            m.pos.add_(1)
        runs[(n, slot)] = torch.stack(rows)
        if n == 8:
            pre8 = m.prefill(inp.contiguous(), 0)[:, slot]
    for key, got in runs.items():
        assert torch.equal(got, runs[(1, 0)]), key
    pre1 = m.prefill(mine.view(T, 1).contiguous(), 0)[:, 0]
    assert torch.equal(pre1, pre8) and torch.equal(pre1, runs[(1, 0)])
    with pytest.raises(ValueError):
        m.step(torch.zeros(S + 1, dtype=torch.int64, device="cuda"), T)
    tm = lc.LlamaModel(cfg, n_streams=S, max_len=T, seed=11)
    with pytest.raises(ValueError):                     # torch mode still runs exactly S streams
        tm.step(torch.zeros(3, dtype=torch.int64, device="cuda"), 128)


CHUNK, B = 24, 4
N_TOKENS = 10 * CHUNK + 7          # 11 chunks; the last chunk is ragged
RANGES = [                         # the ranges of tests/test_gpu_token_range.py
    (0, 1),
    (5 * CHUNK + 11, 5 * CHUNK + 12),
    (2 * CHUNK + 2, 2 * CHUNK + 20),
    (CHUNK - 4, CHUNK + 6),
    (4 * CHUNK - 5, 4 * CHUNK + 9),
    (10 * CHUNK, N_TOKENS),
    (10 * CHUNK + 3, N_TOKENS - 1),
    (0, N_TOKENS),
    (3 * CHUNK + 7, 3 * CHUNK + 7),
]


def _compressor(S, use_graphs=True, batch_invariant=True):
    model = lc.LlamaModel(lc.CONFIGS["tiny"], n_streams=S, max_len=CHUNK, seed=3, batch_invariant=batch_invariant)
    return lc.LlamaCompressor(model, chunk_tokens=CHUNK, use_graphs=use_graphs)


def _source():
    return np.random.default_rng(5).integers(0, 32000, N_TOKENS).astype(np.int32)


def _log_calls(comp):
    """Wrap the engine's decode_batch: per call (chunks, active n, model steps run)."""
    eng, orig, log = comp.engine, comp.engine.decode_batch, []

    def decode_batch(streams, ntok):
        out = orig(streams, ntok)
        log.append((len(streams), eng.n, int(eng.m.pos.item()), int(ntok.max())))
        return out
    eng.decode_batch = decode_batch
    return log


@pytest.fixture(scope="module")
def bi_file():
    toks = _source()
    return toks, _compressor(B).compress(toks)


@pytest.mark.parametrize("use_graphs", [True, False])
@pytest.mark.parametrize("S", [1, 3, 4, 16])
def test_any_decoder_size_reads_every_range(bi_file, S, use_graphs):
    toks, blob = bi_file
    comp = _compressor(S, use_graphs)
    log = _log_calls(comp)
    assert np.array_equal(comp.decompress(blob), toks)
    for start, stop in RANGES:
        del log[:]
        got = comp.decompress(blob, start, stop)
        assert got.dtype == np.int32 and np.array_equal(got, toks[start:stop]), (S, start, stop)
        for chunks, n, steps, longest in log:
            assert chunks <= S and n == lc.active_streams(chunks, S) and steps == longest, (start, stop, log)
        c = container.unpack(blob)
        first = np.concatenate([[0], np.cumsum(c.ntok.astype(np.int64))])
        need = sum(1 for i in range(c.n_chunks) if max(first[i], start) < min(first[i + 1], stop))
        assert sum(ch for ch, *_ in log) == need
        if (start, stop) == (0, 1):
            assert [(ch, n) for ch, n, *_ in log] == [(1, 1)] and log[0][2] == 1


def test_files_at_other_batch_sizes_and_refusals(bi_file):
    toks, blob4 = bi_file
    blob3 = _compressor(3).compress(toks)
    a, b = container.unpack(blob3), container.unpack(blob4)
    assert (a.batch_streams, b.batch_streams) == (3, 4)
    assert np.array_equal(a.ntok, b.ntok) and np.array_equal(a.nbits, b.nbits) and a.payload == b.payload
    assert (a.tag, a.vocab, a.chunk_tokens, a.prec) == (b.tag, b.vocab, b.chunk_tokens, b.prec)
    assert blob3[container.HEADER.size:] == blob4[container.HEADER.size:]
    torch4 = _compressor(4, batch_invariant=False).compress(toks)
    with pytest.raises(ValueError):              # torch mode: the batch shape still binds
        _compressor(3, batch_invariant=False).decompress(torch4)
    with pytest.raises(ValueError):              # batch-invariant compressor, torch-mode file
        _compressor(4).decompress(torch4)
    with pytest.raises(ValueError):              # and the other way round
        _compressor(4, batch_invariant=False).decompress(blob4)
    assert np.array_equal(_compressor(4, batch_invariant=False).decompress(torch4), toks)
    # the old path at the file's own shape still reads a batch-invariant file
    comp = _compressor(4)
    assert np.array_equal(sharding.decompress_sharded(blob4, comp.engine.decode_batch, "cuda"), toks)
