"""cqtObj_cqhc / cqtObj_deconv (VERDICT r1 missing #4): the numpy restatement pinned to the reference build on the CPU."""
import numpy as np
import pytest

from conftest import rel_max
from oracle import af_oracle as O


def spectra(T, num, seed):
    rng = np.random.default_rng(seed)
    k = np.arange(num)
    base = np.exp(-((k[None, :] - rng.uniform(5, num - 5, (T, 1))) / 6.0) ** 2) + 0.3 * np.exp(-k[None, :] / 30.0)
    return (base * rng.uniform(0.5, 2.0, (T, 1)) + 0.01 * rng.random((T, num))).astype(np.float32)


@pytest.mark.parametrize("num,bpo,hc", [(84, 12, 20), (96, 24, 30), (36, 12, 8)])
def test_oracle_deconv_cqhc_vs_reference_build(reference, num, bpo, hc):
    import audioflux_b200 as af
    x = (0.1 * np.random.default_rng(0).standard_normal(24000)).astype(np.float32)

    T = af.CQT(num, 32000, bin_per_octave=bpo).cal_time_length(len(x))
    m = spectra(T, num, num + hc)                     # CQT-shaped magnitudes, regenerated identically wherever the test runs

    def ref(lib):
        c = af.CQT(num, 32000, bin_per_octave=bpo, _lib=lib)
        assert c.cqt(x).shape == (num, T)             # sets the object's timeLength
        return tuple(c.deconv_planes(m)) + (c.cqhc_planes(m, hc),)
    tone, pitch, got = reference("tone,pitch,cqhc", ref)
    o_tone, o_pitch = O.cq_deconv(m, bpo)
    assert rel_max(o_tone, tone) < 1e-5 and rel_max(o_pitch, pitch) < 1e-4
    assert rel_max(O.cqhc(m, hc, bpo), got) < 1e-5


@pytest.mark.parametrize("num,scale,r", [(128, "MEL", 11), (40, "BARK", 10), (257, "LINEAR", 9)])
def test_oracle_deconv_vs_reference_spectrogram_deconv(reference, num, scale, r):
    """spectrogramObj_deconv (spectrogram_algorithm.c:1545-1612) is the same per-frame transform as cqtObj_deconv"""
    import audioflux_b200 as af
    x = (0.1 * np.random.default_rng(2).standard_normal(12000)).astype(np.float32)

    T = af.Spectrogram(num, radix2_exp=r, samplate=16000, filter_bank_type=getattr(af.SpectralFilterBankScaleType, scale)).cal_time_length(len(x))
    spec = np.ascontiguousarray(spectra(T, num, num + r).T)   # [num, T], regenerated identically wherever the test runs

    def ref(lib):
        s = af.Spectrogram(num, radix2_exp=r, samplate=16000, filter_bank_type=getattr(af.SpectralFilterBankScaleType, scale), _lib=lib)
        assert s.spectrogram(x).shape == (num, T)     # sets the object's timeLength
        return s.deconv(spec)
    tone, pitch = reference("tone,pitch", ref)
    o_tone, o_pitch = O.cq_deconv(np.ascontiguousarray(spec.T))
    assert tone.shape == spec.shape
    assert rel_max(o_tone.T, tone) < 1e-5 and rel_max(o_pitch.T, pitch) < 1e-4
