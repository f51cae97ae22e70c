"""cqtObj_cqhc / cqtObj_deconv on the GPU (kernels/deconv.cu) against the numpy oracle and the reference build."""
import numpy as np
import pytest

from conftest import rel_max
from oracle import af_oracle as O
from test_deconv_cpu import spectra

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("num,bpo,hc", [(84, 12, 20), (96, 24, 30), (36, 12, 8)])
def test_deconv_cqhc_vs_oracle_and_reference(cuda_device, reference, num, bpo, hc):
    import audioflux_b200 as af
    x = (0.1 * np.random.default_rng(1).standard_normal(24000)).astype(np.float32)
    c = af.CQT(num, 32000, bin_per_octave=bpo)
    z = c.cqt(x)
    zr_abs = reference("cqt_abs", lambda lib: np.abs(af.CQT(num, 32000, bin_per_octave=bpo, _lib=lib).cqt(x)))
    assert rel_max(np.abs(z), zr_abs) < 1e-4
    m = spectra(z.shape[1], num, num + hc)        # CQT-shaped magnitudes, the same input for all three wherever the test runs

    def ref(lib):
        cr = af.CQT(num, 32000, bin_per_octave=bpo, _lib=lib)
        cr.cqt(x)                                                  # sets the object's timeLength
        return tuple(cr.deconv_planes(m)) + (cr.cqhc_planes(m, hc),)
    r_tone, r_pitch, r_cqhc = reference("tone,pitch,cqhc", ref)
    tone, pitch = c.deconv_planes(m)
    o_tone, o_pitch = O.cq_deconv(m, bpo)
    assert rel_max(tone, o_tone) < 1e-4 and rel_max(pitch, o_pitch) < 1e-4
    assert rel_max(tone, r_tone) < 1e-4 and rel_max(pitch, r_pitch) < 1e-4
    got = c.cqhc_planes(m, hc)
    assert rel_max(got, O.cqhc(m, hc, bpo)) < 1e-4 and rel_max(got, r_cqhc) < 1e-4
    # python-layout wrappers: [num, T] in, [.., T] out
    t2, p2 = c.deconv(np.ascontiguousarray(m.T))
    assert t2.shape == (num, m.shape[0]) and np.allclose(t2.T, tone) and np.allclose(p2.T, pitch)
    assert c.cqhc(z, hc).shape == (hc, m.shape[0])


def test_deconv_batch_any_rows_host_and_device(cuda_device):
    import torch
    import audioflux_b200 as af
    c = af.CQT(84, 32000)
    m = spectra(3 * 77, 84, 5).reshape(3, 77, 84)
    tone, pitch = c.deconv_batch(m)
    o_tone, o_pitch = O.cq_deconv(m.reshape(-1, 84))
    assert rel_max(tone.reshape(-1, 84), o_tone) < 1e-4 and rel_max(pitch.reshape(-1, 84), o_pitch) < 1e-4
    td, pd = c.deconv_batch(torch.from_numpy(m).cuda())
    hd = c.cqhc_batch(torch.from_numpy(m).cuda(), 20)
    torch.cuda.synchronize()
    assert np.array_equal(td.cpu().numpy(), tone) and np.array_equal(pd.cpu().numpy(), pitch)
    assert rel_max(hd.cpu().numpy().reshape(-1, 20), O.cqhc(m.reshape(-1, 84), 20)) < 1e-4


@pytest.mark.parametrize("num,scale,r", [(128, "MEL", 11), (40, "BARK", 10), (257, "LINEAR", 9)])
def test_spectrogram_deconv_vs_oracle_and_reference(cuda_device, reference, num, scale, r):
    """spectrogramObj_deconv / spectrogramObj_deconvBatch: same kernel as cqtObj_deconv, band count of the spectrogram"""
    import torch
    import audioflux_b200 as af
    x = (0.1 * np.random.default_rng(3).standard_normal(12000)).astype(np.float32)
    kw = dict(radix2_exp=r, samplate=16000, filter_bank_type=getattr(af.SpectralFilterBankScaleType, scale))
    s = af.Spectrogram(num, **kw)
    spec = s.spectrogram(x)

    def ref(lib):
        q = af.Spectrogram(num, _lib=lib, **kw)
        spec_r = q.spectrogram(x)                      # also sets the object's timeLength
        return (spec_r,) + tuple(q.deconv(np.ascontiguousarray(spectra(spec_r.shape[1], num, num + r).T)))
    spec_r, r_tone, r_pitch = reference("spec,tone,pitch", ref)
    assert rel_max(spec, spec_r) < 1e-4
    spec = np.ascontiguousarray(spectra(spec.shape[1], num, num + r).T)    # [num, T], the same input for all three
    tone, pitch = s.deconv(spec)
    o_tone, o_pitch = O.cq_deconv(np.ascontiguousarray(spec.T))
    assert tone.shape == spec.shape
    assert rel_max(tone.T, o_tone) < 1e-4 and rel_max(pitch.T, o_pitch) < 1e-4
    assert rel_max(tone, r_tone) < 1e-4 and rel_max(pitch, r_pitch) < 1e-4
    m = np.ascontiguousarray(np.stack([spec.T, 2.0 * spec.T]))                # [2, T, num]
    bt, bp = s.deconv_batch(m)
    assert np.array_equal(bt[0], tone.T) and rel_max(bt[1], 2.0 * tone.T) < 1e-5
    dt, dp = s.deconv_batch(torch.from_numpy(m).cuda())
    torch.cuda.synchronize()
    assert np.array_equal(dt.cpu().numpy(), bt) and np.array_equal(dp.cpu().numpy(), bp)
