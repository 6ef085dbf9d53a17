"""Token-range reads through the model in the loop (LlamaCompressor.decompress(blob, start, stop)), on the GPU.

A range read decodes a chunk in its original batch slot while the batch's other slots are empty streams with no
tokens; when the file was written those rows held other chunks' tokens.  The read is lossless only if every op of
LlamaModel.step keeps rows independent at a fixed batch shape (GEMMs at fixed M, RMSNorm, rope, the KV-cache
index_copy_, SDPA over the cache slice) -- this test is what pins that premise."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():  # collected on CPU boxes, deselected by -m "not gpu"
    pytest.skip("no CUDA device", allow_module_level=True)

from lac_b200 import container, llama_compress as lc  # noqa: E402

CHUNK, B = 24, 4
CFG = lc.LlamaConfig("t", 32000, 64, 2, 4, 2, 128, 64)
N_TOKENS = 10 * CHUNK + 7          # 11 chunks: 3 batches, the last one padded; the last chunk is ragged
RANGES = [
    (0, 1),                        # one token at the file start
    (5 * CHUNK + 11, 5 * CHUNK + 12),   # one token in the middle of a chunk
    (2 * CHUNK + 2, 2 * CHUNK + 20),    # inside one chunk
    (CHUNK - 4, CHUNK + 6),        # across a chunk boundary
    (4 * CHUNK - 5, 4 * CHUNK + 9),     # across a batch boundary (chunk 3 | chunk 4)
    (10 * CHUNK, N_TOKENS),        # the ragged last chunk
    (10 * CHUNK + 3, N_TOKENS - 1),     # inside the ragged last chunk
    (0, N_TOKENS),                 # the whole file
    (3 * CHUNK + 7, 3 * CHUNK + 7),     # empty
]


def _compressor(use_graphs):
    model = lc.LlamaModel(CFG, n_streams=B, max_len=CHUNK, seed=3)
    return lc.LlamaCompressor(model, chunk_tokens=CHUNK, use_graphs=use_graphs)


def _steps_per_batch(blob, start, stop):
    """Model steps each decoded batch needs: the furthest position a needed chunk is read to."""
    c = container.unpack(blob)
    first = np.concatenate([[0], np.cumsum(c.ntok.astype(np.int64))])
    steps = {}
    for i in range(c.n_chunks):
        if max(first[i], start) < min(first[i + 1], stop):
            steps[i // B] = max(steps.get(i // B, 0), min(int(c.ntok[i]), stop - int(first[i])))
    return [steps[k] for k in sorted(steps)]


def _count_steps(comp):
    """Wrap the engine's decode_batch: per call, the steps it ran (the device position after the call)."""
    eng, orig, log = comp.engine, comp.engine.decode_batch, []

    def decode_batch(streams, ntok):
        out = orig(streams, ntok)
        log.append(int(eng.m.pos.item()))
        assert log[-1] == int(ntok.max())
        return out
    eng.decode_batch = decode_batch
    return log


@pytest.mark.parametrize("use_graphs", [True, False])
def test_token_range_reads_match_the_source_and_the_full_decode(use_graphs):
    toks = np.random.default_rng(5).integers(0, CFG.vocab, N_TOKENS).astype(np.int32)
    comp = _compressor(use_graphs)
    blob = comp.compress(toks)
    c = container.unpack(blob)
    assert c.n_chunks == 11 and c.ntok.tolist() == [CHUNK] * 10 + [7] and c.batch_streams == B
    full = comp.decompress(blob)
    assert np.array_equal(full, toks)
    log = _count_steps(comp)
    for start, stop in RANGES:
        del log[:]
        got = comp.decompress(blob, start, stop)
        assert got.dtype == np.int32
        assert np.array_equal(got, toks[start:stop]), (start, stop)
        assert np.array_equal(got, full[start:stop]), (start, stop)
        assert log == _steps_per_batch(blob, start, stop), (start, stop)
    # a fresh compressor (same seed) whose graphs are first captured inside range reads
    fresh = _compressor(use_graphs)
    log = _count_steps(fresh)
    for start, stop in RANGES:
        del log[:]
        assert np.array_equal(fresh.decompress(blob, start=start, stop=stop), toks[start:stop]), (start, stop)
        assert log == _steps_per_batch(blob, start, stop), (start, stop)
    with pytest.raises(ValueError):
        comp.decompress(blob, 5, N_TOKENS + 1)
    with pytest.raises(ValueError):
        comp.decompress(blob, -3)
