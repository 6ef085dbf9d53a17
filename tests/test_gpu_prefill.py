"""The batch-invariant model kernels (lac_model_*) and prefill compression, on the GPU.

What is pinned: each kernel computes the right function (against torch references within a stated tolerance), and
a row's bits do not depend on how many rows or positions its launch covers, or where in a tile it sits -- which is
what lets LlamaCompressor encode with prefill launches while the decoder replays per-token steps."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():  # collected on CPU boxes, deselected by -m "not gpu"
    pytest.skip("no CUDA device", allow_module_level=True)

from lac_b200 import _ffi, container, sharding, llama_compress as lc  # noqa: E402

BF = torch.bfloat16


def _st():
    return torch.cuda.current_stream().cuda_stream


def _gemm(x, w, epi, res=None):
    M, (K, N) = x.shape[0], w.shape
    y = torch.empty((M, N), device="cuda", dtype=torch.float32 if epi == _ffi.LAC_MODEL_OUT_F32 else BF)
    _ffi.check(_ffi.lib().lac_model_gemm(x.data_ptr(), w.data_ptr(), M, N, K, epi,
                                         None if res is None else res.data_ptr(), y.data_ptr(), _st()))
    return y


def _weight_shapes():
    shapes = set()
    for cfg in lc.CONFIGS.values():
        hd = cfg.dim // cfg.heads
        shapes |= {(cfg.dim, (cfg.heads + 2 * cfg.kv_heads) * hd), (cfg.dim, cfg.dim), (cfg.dim, 2 * cfg.ffn),
                   (cfg.ffn, cfg.dim), (cfg.dim, cfg.vocab)}
    return sorted(shapes)


@pytest.mark.parametrize("K,N", _weight_shapes())
def test_gemm_matches_fp32_and_is_row_invariant(K, N):
    g = torch.Generator(device="cuda").manual_seed(K * 7 + N)
    S, Tb = 4, 64
    x = torch.randn((Tb * S, K), device="cuda", generator=g).to(BF)
    w = (torch.randn((K, N), device="cuda", generator=g) * K ** -0.5).to(BF)
    res = torch.randn((Tb * S, N), device="cuda", generator=g).to(BF)
    ref = x.float() @ w.float()
    for epi in (_ffi.LAC_MODEL_OUT_BF16, _ffi.LAC_MODEL_OUT_BF16_ADD, _ffi.LAC_MODEL_OUT_F32):
        r = res if epi == _ffi.LAC_MODEL_OUT_BF16_ADD else None
        full = _gemm(x, w, epi, r)
        if epi == _ffi.LAC_MODEL_OUT_F32:
            torch.testing.assert_close(full, ref, atol=1e-3, rtol=1e-3)
        elif epi == _ffi.LAC_MODEL_OUT_BF16:
            torch.testing.assert_close(full.float(), ref, atol=2e-2, rtol=1e-2)
        else:
            torch.testing.assert_close(full.float(), res.float() + ref, atol=4e-2, rtol=1e-2)
        # the same rows from launches of M = S (at other tile rows), M = T_blk * S and M = 200 (not a multiple of 128)
        for lo, hi in ((0, S), (101, 101 + S), (0, 200)):
            part = _gemm(x[lo:hi].contiguous(), w, epi, None if r is None else r[lo:hi].contiguous())
            assert torch.equal(part, full[lo:hi]), (epi, lo, hi)


def test_gemm_rejects_unsupported_shapes():
    x = torch.zeros((4, 96), device="cuda", dtype=BF)
    w = torch.zeros((96, 128), device="cuda", dtype=BF)
    y = torch.zeros((4, 128), device="cuda", dtype=BF)
    rc = _ffi.lib().lac_model_gemm(x.data_ptr(), w.data_ptr(), 4, 128, 96, 0, None, y.data_ptr(), _st())
    assert rc == _ffi.LAC_E_ARG and b"unsupported shape" in _ffi.lib().lac_last_error()
    rc = _ffi.lib().lac_model_gemm(x.data_ptr(), w.data_ptr(), 4, 100, 64, 0, None, y.data_ptr(), _st())
    assert rc == _ffi.LAC_E_ARG


@pytest.mark.parametrize("dim", [256, 2048, 4096])
def test_rmsnorm_matches_torch_and_is_row_invariant(dim):
    g = torch.Generator(device="cuda").manual_seed(dim)
    x = (torch.randn((300, dim), device="cuda", generator=g) * 2).to(BF)

    def norm(a):
        y = torch.empty_like(a)
        _ffi.check(_ffi.lib().lac_model_rmsnorm(a.data_ptr(), a.shape[0], dim, 1e-6, y.data_ptr(), _st()))
        return y
    y = norm(x)
    ref = torch.nn.functional.rms_norm(x.float(), (dim,), eps=1e-6)
    torch.testing.assert_close(y.float(), ref, atol=2e-2, rtol=1e-2)
    assert torch.equal(norm(x[37:41].contiguous()), y[37:41])


def _attn(qkv, S, n_q, H, KV, hd, kc, vc, max_len, d_pos=None, p0=0):
    out = torch.empty((n_q * S, H * hd), device="cuda", dtype=BF)
    _ffi.check(_ffi.lib().lac_model_attention(qkv.data_ptr(), S, n_q, H, KV, hd,
                                              None if d_pos is None else d_pos.data_ptr(), p0, kc.data_ptr(),
                                              vc.data_ptr(), max_len, out.data_ptr(), _st()))
    return out


@pytest.mark.parametrize("hd,H,KV", [(64, 4, 2), (64, 32, 4), (128, 32, 8)])
def test_attention_matches_torch_and_step_equals_prefill(hd, H, KV):
    S, max_len = 3, 200
    g = torch.Generator(device="cuda").manual_seed(hd + H)
    kc = torch.randn((S, KV, max_len, hd), device="cuda", generator=g).to(BF)
    vc = torch.randn((S, KV, max_len, hd), device="cuda", generator=g).to(BF)
    W = (H + 2 * KV) * hd
    qkv = torch.randn((max_len * S, W), device="cuda", generator=g).to(BF)   # row t * S + s
    full = _attn(qkv, S, max_len, H, KV, hd, kc, vc, max_len)
    # reference: causal softmax over the cache in fp32
    q = qkv.view(max_len, S, W)[:, :, :H * hd].view(max_len, S, H, hd).float()
    k = kc.float().repeat_interleave(H // KV, 1)                 # [S, H, L, hd]
    v = vc.float().repeat_interleave(H // KV, 1)
    sc = torch.einsum("tshd,shld->shtl", q, k) * hd ** -0.5
    sc = sc.masked_fill(torch.ones(max_len, max_len, device="cuda", dtype=torch.bool).triu(1), float("-inf"))
    ref = torch.einsum("shtl,shld->tshd", sc.softmax(-1), v).reshape(max_len * S, H * hd)
    torch.testing.assert_close(full.float(), ref, atol=2e-2, rtol=2e-2)
    # Q = 1 at position p (read from the device) equals row p of the prefill launch, at KV-block edges and the end
    for p in (0, 63, 64, 65, 130, max_len - 1):
        pos = torch.tensor([p], device="cuda", dtype=torch.int64)
        one = _attn(qkv[p * S:(p + 1) * S].contiguous(), S, 1, H, KV, hd, kc, vc, max_len, d_pos=pos)
        assert torch.equal(one, full[p * S:(p + 1) * S]), p
    # a prefill launch that starts at p0 > 0
    p0, n = 60, 11
    part = _attn(qkv[p0 * S:(p0 + n) * S].contiguous(), S, n, H, KV, hd, kc, vc, max_len, p0=p0)
    assert torch.equal(part, full[p0 * S:(p0 + n) * S])


def _inputs(S, T, seed):
    toks = torch.from_numpy(np.random.default_rng(seed).integers(0, 32000, (T, S))).cuda()
    return torch.cat([torch.full((1, S), lc.BOS, device="cuda", dtype=torch.int64), toks[:-1]])


@pytest.mark.parametrize("S", [4, 128])
def test_prefill_logits_equal_step_logits(S):
    cfg, T = lc.CONFIGS["tiny"], 80
    inp = _inputs(S, T, S)
    m = lc.LlamaModel(cfg, n_streams=S, max_len=T, seed=11, batch_invariant=True)
    m.reset()
    step = []
    for t in range(T):
        step.append(m.step(inp[t], T).clone())
        m.pos.add_(1)
    step = torch.stack(step)
    m.reset()
    for p0, n in ((0, 32), (32, 32), (64, 16)):   # the last block is shorter
        blk = m.prefill(inp[p0:p0 + n].contiguous(), p0)
        for t in range(n):
            assert torch.equal(blk[t], step[p0 + t]), (p0, t)
    # the same function as the torch-mode model of the same seed, up to bf16 rounding in different places
    tm = lc.LlamaModel(cfg, n_streams=S, max_len=T, seed=11)
    tm.reset()
    ref = []
    for t in range(T):
        ref.append(tm.step(inp[t], lc._bucket_for(t, T)).clone())
        tm.pos.add_(1)
    d = (torch.stack(ref) - step).abs()
    # measured on a B200: mean 0.016, max 0.13 at S = 4 and 128, against logits of std 3
    assert d.mean().item() < 0.03 and d.max().item() < 0.5


CHUNK, B = 24, 4
N_TOKENS = 10 * CHUNK + 7          # 11 chunks: 3 batches, the last one padded; the last chunk is ragged
RANGES = [(0, 1), (2 * CHUNK + 2, 2 * CHUNK + 20), (4 * CHUNK - 5, 4 * CHUNK + 9), (10 * CHUNK + 3, N_TOKENS - 1)]


def _compressor(use_graphs, batch_invariant=True):
    model = lc.LlamaModel(lc.CONFIGS["tiny"], n_streams=B, max_len=CHUNK, seed=3, batch_invariant=batch_invariant)
    return lc.LlamaCompressor(model, chunk_tokens=CHUNK, use_graphs=use_graphs)


@pytest.mark.parametrize("block", [None, 5])
def test_prefill_compression_is_the_stepwise_file_and_decodes(monkeypatch, block):
    if block is not None:   # blocks of 5 positions: 24 = 5 + 5 + 5 + 5 + 4
        monkeypatch.setattr(lc, "PREFILL_LOGITS_BYTES", block * 4 * B * 32000)
    toks = np.random.default_rng(5).integers(0, 32000, N_TOKENS).astype(np.int32)
    comp = _compressor(True)
    assert block is None or lc.prefill_block(comp.model) == block
    blob = comp.compress(toks)
    stepwise = sharding.compress_sharded(toks, CHUNK, B, comp.engine.encode_batch, comp.prec, comp.vocab,
                                         comp.model.device, comp.tag, None)
    assert blob == stepwise
    c = container.unpack(blob)
    assert c.n_chunks == 11 and c.ntok.tolist() == [CHUNK] * 10 + [7]
    assert np.array_equal(comp.decompress(blob), toks)
    nog = _compressor(False)
    assert np.array_equal(nog.decompress(blob), toks)
    for start, stop in RANGES:
        assert np.array_equal(comp.decompress(blob, start, stop), toks[start:stop]), (start, stop)
    with pytest.raises(ValueError):
        _compressor(False, batch_invariant=False).decompress(blob)
