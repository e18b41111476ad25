"""Host-side checks of per-utterance seeds and guidance scales (no GPU): what sample_latents(_ragged) accepts as ``seeds`` /
``guidance_scale`` and what it refuses before any device work, and the argument checks of ditto_randn_latents, which need
no engine."""
import ctypes as C

import pytest
import torch

from ditto_tts_b200 import _lib, build
from ditto_tts_b200._lib import DittoError
from ditto_tts_b200.sampler import _check_scale, _check_seeds, _seed_tensor


def test_seeds_accepted_over_the_whole_uint64_range():
    assert _check_seeds(None, 3) is None
    s = [0, 1, 2 ** 63 - 1, 2 ** 63, 2 ** 64 - 1]
    assert _check_seeds(s, 5) == s
    assert _check_seeds(tuple(s), 5) == s
    assert _check_seeds(torch.tensor([3, 4]), 2) == [3, 4]
    # the device reads the int64 bit pattern as uint64
    t = _seed_tensor(s, "cpu")
    assert t.dtype == torch.int64 and [v & (2 ** 64 - 1) for v in t.tolist()] == s


@pytest.mark.parametrize("seeds,B,match", [
    ([1, 2], 3, "3 expected, got 2"),
    ([1, 2, 3, 4], 3, "3 expected, got 4"),
    ([1, -1, 2], 3, "outside"),
    ([1, 2 ** 64, 2], 3, "outside"),
    ([1, 2.0, 3], 3, "integer"),
    ([True, 2, 3], 3, "bool"),
    ("abc", 3, "sequence"),
    (5, 1, "sequence"),
])
def test_bad_seeds_are_refused(seeds, B, match):
    with pytest.raises(DittoError, match=match):
        _check_seeds(seeds, B)


def test_seeds_exclude_noise_and_generator():
    with pytest.raises(DittoError, match="excludes"):
        _check_seeds([1, 2], 2, noise=torch.zeros(1))
    with pytest.raises(DittoError, match="excludes"):
        _check_seeds([1, 2], 2, generator=torch.Generator())


def test_scalar_scales_are_taken_as_before():
    """Whatever float(w) took before per-utterance scales existed stays one scale for every utterance, whatever B is:
    numpy scalars, 0-d arrays and one-element tensors / arrays; a scalar is not checked for finiteness (as before)."""
    np = pytest.importorskip("numpy")
    for w in (np.float32(3.0), np.float64(2.5), np.int64(4), np.array(1.5), np.array([2.0]), torch.tensor(3.0),
              torch.tensor([3.0]), True):
        for B in (1, 3):
            got = _check_scale(w, B)
            assert isinstance(got, float) and got == float(w.item() if hasattr(w, "item") else w), (w, B)
    assert _check_scale(float("inf"), 2) == float("inf")
    assert _check_scale(np.array([1.0, 2.0]), 2) == [1.0, 2.0]


def test_guidance_scales():
    assert _check_scale(None, 2) is None
    assert _check_scale(3.0, 2) == 3.0 and _check_scale(2, 2) == 2
    assert _check_scale([1, 2.5], 2) == [1.0, 2.5]
    assert _check_scale(torch.tensor([1.0, -2.0]), 2) == [1.0, -2.0]
    for bad, match in (([1.0], "2 expected"), ([1.0, float("nan")], "finite"), ([float("inf"), 1.0], "finite"),
                       (object(), "number")):
        with pytest.raises(DittoError, match=match):
            _check_scale(bad, 2)


def test_randn_latents_refuses_null_arrays():
    build.build()
    lib = _lib.load()
    buf = (C.c_int64 * 8)()
    p = C.cast(buf, C.c_void_p)
    assert lib.ditto_randn_latents(None, p, 1, 8, p, None) == -1
    assert lib.ditto_randn_latents(p, None, 1, 8, p, None) == -1
    assert lib.ditto_randn_latents(p, p, 1, 8, None, None) == -1
    assert b"randn_latents" in lib.ditto_last_error()
