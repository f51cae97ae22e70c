"""The stored form of the reference's results (tests/conftest.py: `reference`): an error anywhere along any axis of a
large array -- in its first or last frame, in any band -- must still fail the comparison against the stored sample."""
import numpy as np
import pytest

from conftest import REF_AXIS, REF_WHOLE, RefSample, _ref_load, _ref_store, _sample_index, rel_max


@pytest.mark.parametrize("shape", [(465, 40), (1876, 84), (84, 4096), (3, 7, 513), (REF_WHOLE + 1,)])
def test_sample_covers_every_axis(shape):
    """every index of an axis of up to REF_AXIS entries; of a longer one REF_AXIS evenly spaced, first and last included"""
    idx = np.unravel_index(_sample_index(shape), shape)
    for d, n in enumerate(shape):
        seen = np.unique(idx[d])
        if n <= REF_AXIS:
            assert np.array_equal(seen, np.arange(n)), d
        else:
            assert seen[0] == 0 and seen[-1] == n - 1 and len(seen) >= REF_AXIS and np.diff(seen).max() <= -(-n // (REF_AXIS - 1)), d


@pytest.mark.parametrize("frames", [REF_AXIS, 465, 1876])
def test_stored_sample_catches_an_error_in_a_frame_or_band(frames):
    """an error in the first or last frame, in any frame of a transform of up to REF_AXIS frames, or in any band"""
    a = np.random.default_rng(0).standard_normal((frames, 40)).astype(np.float32)
    out = {}
    _ref_store("k", a, out)
    s = _ref_load("k", out)
    assert isinstance(s, RefSample) and rel_max(a, s) == 0.0
    for t in (range(frames) if frames <= REF_AXIS else (0, frames - 1)):
        b = a.copy()
        b[t] += 1e-3
        assert rel_max(b, s) > 1e-4, t
    for c in range(40):
        b = a.copy()
        b[:, c] -= 1e-3
        assert rel_max(b, s) > 1e-4, c


def test_small_arrays_are_stored_whole():
    a = np.arange(REF_WHOLE, dtype=np.float32).reshape(-1, 8)
    out = {}
    _ref_store("k", a, out)
    assert np.array_equal(_ref_load("k", out), a)
