"""Reassignment (VERDICT r1 missing #3): the numpy oracle `af_oracle.reassign` pinned to the reference build
(oracle/_ref, reassignObj_* of src/reassign_algorithm.c) on the CPU.

Parity bar: the scatter indices are roundf() of float32 divides, so a cell whose reassigned frequency / time sits within
an ulp of a cell boundary may land one cell apart between two implementations.  Numpy oracle vs the reference build:
>= 99.9 % of the cells identical to 1e-5 of the maximum, relative Frobenius error <= 2e-3; the plain half spectrum S_h
returned beside it meets the usual 1e-4."""
import numpy as np
import pytest

from conftest import ref_pair, rel_max
from oracle import af_oracle as O


def _signal(n, sr, seed):
    t = np.arange(n) / sr
    rng = np.random.default_rng(seed)
    return (0.5 * np.sin(2 * np.pi * (300 + 2000 * t) * t) + 0.2 * np.sin(2 * np.pi * 2500 * t) + 0.01 * rng.standard_normal(n)).astype(np.float32)


def agree(a, b):
    scale = np.abs(b).max()
    return 1.0 - (np.abs(a - b) > 1e-5 * scale).mean(), float(np.linalg.norm(a - b) / np.linalg.norm(b))


CASES = [(9, 16000, 1, 128, 0, 0.001, 0, 1, 0), (10, 32000, 1, 256, 0, 0.001, 1, 1, 0), (9, 16000, 2, 100, 1, 0.001, 0, 1, 0),
         (9, 16000, 1, 128, 2, 0.001, 0, 1, 1), (9, 16000, 1, 128, 0, 0.001, 0, 2, 0), (9, 16000, 1, 128, 0, 0.001, 0, 3, 1),
         (10, 32000, 3, 256, 0, 0.01, 1, 2, 0), (8, 8000, 0, 64, 0, 0.0, 0, 1, 0)]


@pytest.mark.parametrize("radix,sr,window,hop,re_type,thresh,pad,order,result_type", CASES)
def test_oracle_reassign_vs_reference_build(reference, radix, sr, window, hop, re_type, thresh, pad, order, result_type):
    import audioflux_b200 as af
    x = _signal(20000, sr, radix)

    def ref(lib):
        r = af.Reassign(radix, sr, af.WindowType(window), hop, af.ReassignType(re_type), thresh, bool(pad), _lib=lib)
        r.set_order(order)
        return r.reassign_planes(x, result_type)
    want = reference("planes", ref)
    got = O.reassign(x, radix, sr, window, hop, re_type, thresh, bool(pad), order, result_type)
    assert rel_max(got[2], want[2]) < 1e-4 and rel_max(got[3], want[3]) < 1e-4
    planes = (0,) if result_type else (0, 1)
    for k in planes:
        same, fro = agree(*ref_pair(got[k], want[k]))
        assert same >= 0.999 and fro <= 2e-3, (k, same, fro)


def test_oracle_reassign_none_is_the_half_spectrum(reference):
    import audioflux_b200 as af
    x = _signal(6000, 16000, 1)
    want = reference("planes", lambda lib: af.Reassign(9, 16000, re_type=af.ReassignType.NONE, _lib=lib).reassign_planes(x))
    got = O.reassign(x, 9, 16000, re_type=O.REASSIGN_NONE)
    assert rel_max(got[0], want[0]) < 1e-5 and rel_max(got[1], want[1]) < 1e-5


def test_reassign_windows_match_the_reference_derivative_rule():
    w = O.fft_window(O.W_HANN, 512)
    h, dh, th = O.reassign_windows(w)
    assert np.array_equal(h, w)
    assert dh[0] == np.float32((w[1] - w[511]) / 2) and dh[511] == np.float32((w[0] - w[510]) / 2)
    assert th[0] == np.float32(-256 * w[0]) and th[256] == 0 and th[511] == np.float32(255 * w[511])
    # energy: the scatter moves cells, it does not create any (|S_h| above the threshold, complex sums can only cancel)
    x = _signal(8000, 16000, 2)
    re, im, sr_, si_ = O.reassign(x, 9, 16000, result_type=1)
    assert abs(re.sum() - np.sqrt(sr_ ** 2 + si_ ** 2).sum()) <= 1e-3 * re.sum()
