"""CPU-side checks of the adaptive count models: the four C entry points reject bad arguments before any CUDA call
(so they return LAC_E_ARG on a machine without a GPU too), and the mirror API's CountPredictor holds the tables of
the reference's adaptive byte model."""
import numpy as np
import pytest

from lac_b200 import _ffi
from lac_b200 import arith_code as ac

FAKE = 0x1000  # a non-NULL pointer that is never dereferenced: every call below fails its argument check first


def _call(name, counts, vocab, inc, prec):
    L = _ffi.lib()
    if "encode" in name:
        return getattr(L, name)(counts, vocab, inc, FAKE, 4, 2, 4, None, FAKE, FAKE, 64, 1, prec, None)
    return getattr(L, name)(counts, vocab, inc, 2, 4, None, FAKE, FAKE, FAKE, FAKE, 4, prec, None)


NAMES = ["lac_ac_encode_adaptive", "lac_ac_decode_adaptive", "lac_acs_encode_adaptive", "lac_acs_decode_adaptive"]


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("counts, vocab, inc, prec", [
    (FAKE, 0, 1, 32), (FAKE, 4097, 1, 32), (FAKE, -1, 1, 32), (FAKE, 256, -1, 32),
    (FAKE, 256, 1, 1), (FAKE, 256, 1, 61), (None, 256, 1, 32),
])
def test_adaptive_entry_points_reject_bad_arguments(name, counts, vocab, inc, prec):
    assert _call(name, counts, vocab, inc, prec) == _ffi.LAC_E_ARG
    assert _ffi.lib().lac_last_error().decode().startswith(name)


def test_adaptive_vocab_limit_matches_header():
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    text = open(os.path.join(root, "include", "lac_b200.h")).read()
    assert int(re.search(r"#define LAC_ADAPTIVE_MAX_VOCAB (\d+)", text).group(1)) == _ffi.LAC_ADAPTIVE_MAX_VOCAB


def test_count_predictor_tables_are_the_adaptive_byte_model():
    """prob(s) = 1 + occurrences of s so far: the table before each symbol, as the goldens were made."""
    rng = np.random.default_rng(1)
    data = rng.integers(0, 256, 500)
    p = ac.CountPredictor(256)
    counts = np.ones(256, dtype=np.int64)
    tabs, minps = ac.materialise_tables(p, data.tolist())
    for t, b in enumerate(data):
        assert np.array_equal(tabs[t], np.cumsum(counts))
        assert minps[t] == counts[counts > 0].min()
        counts[b] += 1
    assert p.counts == counts.tolist()


def test_count_predictor_counts_inc_and_routing():
    p = ac.CountPredictor(4, counts=[0, 3, 0, 2], inc=5)
    assert p.dist == [0, 3, 3, 5] and p.minp == 2
    p.accept(2)
    assert p.counts == [0, 3, 5, 2] and p.dist == [0, 3, 8, 10]
    assert ac._kind(p) == "counts"
    assert ac._kind(ac.ProbPredictor(4)) == "tables"

    class Sub(ac.CountPredictor):
        pass

    assert ac._kind(Sub(4)) == "tables"  # only the exact type: a subclass may change prob()
    with pytest.raises(ValueError):
        ac.CountPredictor(3, counts=[1, 2])


def test_count_predictor_device_bounds():
    fit = ac._counts_fit
    assert fit(ac.CountPredictor(4096), 10, False)
    assert not fit(ac.CountPredictor(4097), 10, False)
    assert not fit(ac.CountPredictor(4), 10, True)                       # numpy-int64 wrap: table path
    assert not fit(ac.CountPredictor(4, counts=[1, -1, 1, 1]), 10, False)
    assert not fit(ac.CountPredictor(4, inc=-1), 10, False)
    big = ac.CountPredictor(2, counts=[(1 << 61), (1 << 61) - 100], inc=10)
    assert fit(big, 9, False) and not fit(big, 10, False)               # the total must stay below 2^62
