"""LQ32 (DESIGN.md section 3) against the float64 softmax, element by element.  The CPU test runs the oracle's
restatement of the spec; the gpu test runs lac_cdf_build_f32 on the same rows, checks it bit for bit against the
oracle and the same bounds.  Asserted per row:
  * every element of a live segment meets the per-element lower bound derived in DESIGN.md section 3;
  * KL(p || p_hat) <= V / 2^32 * log2 e + 4e-9 bits when no finite element sits in a dropped (EMPTY) segment;
  * a degenerate row (no finite value, a +inf, or a maximum past the EMPTY / POISON thresholds) is cum_i = i."""
import numpy as np
import pytest

from oracle import oracle as orc

LOG2E_F = float(np.array([0x3FB8AA3B], dtype=np.uint32).view(np.float32)[0])  # log2 e rounded to fp32
EPS_LOG2E = abs(LOG2E_F * np.log(2.0) - 1.0)          # relative error of that rounding, 1.3e-8
DELTA = 1.025e-4      # 2^f polynomial (1.02e-4) plus the roundings of f and of the mantissa
MAGIC = 1.5 * 2.0 ** 23
REF_LO, REF_HI, POISON = 0x4B000040, 0x4B800000, 0xFFFFFF


# ------------------------------------------------------------------------------------------------ rows
def _segments(V):
    parts = (V + 32767) // 32768
    nw, g = 32 * parts, (V + 3) // 4
    b = [4 * ((w * g) // nw) for w in range(nw + 1)]
    return [(b[w], min(V, b[w + 1])) for w in range(nw) if b[w] < min(V, b[w + 1])]


def _code(m):
    """Reference code of a segment maximum, fp32 fma(m, log2e, MAGIC) emulated exactly in float64 (a 24 x 24-bit
    product plus MAGIC fits 53 bits, then one rounding to fp32)."""
    if m == -np.inf:
        return 0
    if m == np.inf:
        return POISON
    n = int(np.array([np.float32(np.float64(m) * LOG2E_F + MAGIC)], dtype=np.float32).view(np.int32)[0])
    return 0 if n < REF_LO else (POISON if n >= REF_HI else n - REF_LO + 1)


def _stepped_row(rng, d_lo, d_hi):
    """65536 elements, 64 segments of 1024: segment w's maximum sits d_w binades below the row maximum, d_w stepping
    through [d_lo, d_hi]; inside a segment the values fall off by up to 4 binades."""
    V = 65536
    x = np.empty(V, dtype=np.float32)
    ds = np.resize(np.arange(d_lo, d_hi + 1), 64)
    ds[0] = 0
    for w, d in enumerate(ds):
        seg = -(d + rng.uniform(0, 4, 1024)) * np.log(2.0)
        seg[rng.integers(0, 1024)] = -(d + 0.1) * np.log(2.0)
        x[w * 1024:(w + 1) * 1024] = seg
    return x


def rows():
    rng = np.random.default_rng(32)
    out = []
    for V in (1, 2, 5, 1000, 32000, 32772, 128256, 262144):
        for scale in (0.3, 3.0, 30.0, 100.0) if V >= 128256 else (0.3, 1.0, 3.0, 10.0, 30.0, 100.0):
            out.append((f"gauss V={V} scale={scale}", (rng.standard_normal(V) * scale + rng.uniform(-50, 50)).astype(np.float32)))
    out.append(("stepped d 36..44", _stepped_row(rng, 36, 44)))
    out.append(("stepped d 12..30", _stepped_row(rng, 12, 30)))
    for V, top in ((32000, 30.0), (128256, 80.0), (1000, 200.0)):
        x = rng.standard_normal(V).astype(np.float32)
        x[rng.integers(0, V)] = top
        out.append((f"spike {top} V={V}", x))
    for V in (1000, 65536):
        x = (rng.standard_normal(V) * 4).astype(np.float32)
        x[rng.random(V) < 0.3] = -np.inf
        x[: 2048 if V > 2048 else 0] = -np.inf                    # whole segments of -inf
        out.append((f"-inf holes V={V}", x))
    # maxima around the EMPTY threshold (m log2e = -(2^22 - 64)) and the POISON threshold (m log2e = 2^22)
    for j in range(-3, 4):
        for edge in (-(2.0 ** 22 - 64), 2.0 ** 22):
            m = np.float32((edge + j) / LOG2E_F)
            x = (m - np.abs(rng.standard_normal(3000)).astype(np.float32) * 2).astype(np.float32)
            x[rng.integers(0, 3000)] = m
            out.append((f"threshold {edge:+.0f}{j:+d}", x))
        # one segment just above the EMPTY threshold, another just below it: the lower one is dropped
        x = np.full(3000, np.float32(-(2.0 ** 22 - 64 + 3) / LOG2E_F), dtype=np.float32)
        x[:1000] = np.float32(-(2.0 ** 22 - 64 - 3 + j) / LOG2E_F)
        out.append((f"straddles EMPTY {j:+d}", x))
    tiny = np.array([1, 7, 0x7FFFFF], dtype=np.uint32).view(np.float32)
    x = np.zeros(1000, dtype=np.float32)
    x[::2] = -0.0
    x[1::3] = tiny[np.arange(len(x[1::3])) % 3]
    x[5::7] = -tiny[np.arange(len(x[5::7])) % 3]
    out.append(("denormals and -0.0", x))
    out.append(("all -0.0", np.full(77, -0.0, dtype=np.float32)))
    for nm, v in (("all -inf", -np.inf), ("+inf", np.inf)):
        x = rng.standard_normal(500).astype(np.float32)
        x[:] = v if nm == "all -inf" else x
        x[123] = v
        out.append((nm, x))
    out.append(("finite max past POISON", np.concatenate([np.zeros(100), [3.0e6]]).astype(np.float32)))
    return out


# ------------------------------------------------------------------------------------------------ checks
def check_row(name, x, cum):
    V = len(x)
    cum = np.asarray(cum, dtype=np.uint64)
    F = np.diff(np.append(cum.astype(np.int64), 1 << 32)).astype(np.float64)
    assert (F >= 1).all(), name
    ph = F / 2.0 ** 32
    segs = _segments(V)
    codes = [_code(float(np.max(x[a:b]))) for a, b in segs]
    r = max(codes)
    if r == 0 or r == POISON:
        assert np.array_equal(cum, np.arange(V, dtype=np.uint64)), f"{name}: degenerate row is not cum_i = i"
        return "degenerate"
    x64 = x.astype(np.float64)
    fin = np.isfinite(x64)
    mx = x64[fin].max()
    p = np.where(fin, np.exp(np.where(fin, x64 - mx, 0.0)), 0.0)
    p /= p.sum()
    rho = np.exp(-EPS_LOG2E * (mx - x64[fin].min()))
    live = np.zeros(V, dtype=bool)
    for (a, b), c in zip(segs, codes):
        live[a:b] = c != 0
    # per-element bound, DESIGN.md section 3
    bound = (1 - V / 2.0 ** 32) * (1 - 2.0 ** -29) * ((1 - DELTA) / (1 + DELTA) * rho * p - 2.0 ** -27.5 * p.max() / rho)
    bad = live & (ph < bound)
    assert not bad.any(), (f"{name}: {int(bad.sum())} elements below the bound, worst at {int(np.argmax(bound - ph))}: "
                           f"p {p[np.argmax(bound - ph)]:.6g} p_hat {ph[np.argmax(bound - ph)]:.6g}")
    if (fin & ~live).any():
        return "dropped segments"
    nz = p > 0
    kl = float(np.sum(p[nz] * np.log2(p[nz] / ph[nz])))
    assert kl <= V / 2.0 ** 32 * np.log2(np.e) + 4e-9, (name, kl)
    rel = np.max(np.where(p >= 2.0 ** -12 * p.max(), 1 - ph / np.maximum(p, 1e-300), 0.0))
    return f"KL {kl:.3g}, max relative deficit {rel:.3g}"


def test_lq32_oracle_against_float64_softmax():
    kinds = {}
    for name, x in rows():
        res = check_row(name, x, orc.lq32_cdf(x[None])[0])
        kinds[res.split(",")[0]] = kinds.get(res.split(",")[0], 0) + 1
    assert kinds.get("degenerate", 0) >= 10 and kinds.get("dropped segments", 0) >= 5


@pytest.mark.gpu
def test_lq32_gpu_against_float64_softmax():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from lac_b200 import _ffi
    L, st = _ffi.lib(), torch.cuda.current_stream().cuda_stream
    for name, x in rows():
        V = len(x)
        d = torch.from_numpy(x[None].copy()).cuda()
        cum = torch.full((3, V), -7, dtype=torch.int32, device="cuda")
        _ffi.check(L.lac_cdf_build_f32(d.data_ptr(), 1, V, V, cum[1].data_ptr(), None, 0, st))
        got = cum.cpu().numpy().view(np.uint32)
        assert (got[0] == 0xFFFFFFF9).all() and (got[2] == 0xFFFFFFF9).all(), name
        assert np.array_equal(got[1], orc.lq32_cdf(x[None])[0]), f"{name}: GPU table differs from the oracle"
        check_row(name, x, got[1])
