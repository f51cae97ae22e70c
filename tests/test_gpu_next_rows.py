"""CUDA parity of the SURVEY section 8(f) rows -- xxccObj_xxccStandard, cqtObj_chroma / cqtObj_cqcc and the
SpectrogramObj front door -- through the C ABI: legacy single-clip entry points with host pointers and the
additive batched entry points with device pointers, against the reference-generated fixture
(tests/golden/next_rows.npz), the numpy oracle on seeded inputs, and oracle/_ref when it travelled.
Tolerance |a-b| <= 1e-4 * max|b| per tensor."""
import numpy as np
import pytest

import audioflux_b200 as af
from conftest import noise, ref_absmax, ref_pair, rel_max, tones
from oracle import af_oracle as O
from test_next_rows_cpu import SPEC_CASES, _phase_mask

pytestmark = pytest.mark.gpu

TOL = 1e-4
S, ST, N, D = (af.SpectralFilterBankScaleType, af.SpectralFilterBankStyleType,
               af.SpectralFilterBankNormalType, af.SpectralDataType)
E, CN = af.CepstralEnergyType, af.ChromaDataNormalType


@pytest.fixture(scope="module")
def torch_cuda(cuda_device):
    import torch
    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    return torch


# ------------------------------------------------------------------ xxccStandard
@pytest.mark.parametrize("name,et,order", [("rep", E.REPLACE, 9), ("app", E.APPEND, 5), ("ign", E.IGNORE, 3)])
def test_xxcc_standard_golden_legacy(cuda_device, golden, name, et, order):
    g, c1 = golden("next_rows.npz"), golden("c1_mel_mfcc.npz")
    x = af.XXCC(128)
    got = x.xxcc_standard_planes(c1["mel"][:24], g["energy"], 13, order, et)
    for a, key in zip(got, ("coe", "d1", "d2")):
        want = g[f"std_{name}_{key}"]
        assert a.shape == want.shape and rel_max(a, want) < TOL


@pytest.mark.parametrize("et,order,cc,rect", [(0, 9, 13, 0), (1, 9, 13, 0), (2, 9, 20, 0), (0, 5, 40, 1), (1, 3, 5, 0),
                                               (0, 4, 13, 0), (1, 11, 64, 0)])
def test_xxcc_standard_batch_vs_oracle(torch_cuda, et, order, cc, rect):
    torch = torch_cuda
    rng = np.random.default_rng(7)
    m = (rng.random((3, 37, 64)) ** 4 * 10).astype(np.float32)
    m[0, 3, :5] = 0
    e = (rng.random((3, 37)) * 3).astype(np.float32)
    e[1, 2] = 0
    x = af.XXCC(64)
    got = x.xxcc_standard_batch(torch.from_numpy(m).cuda(), torch.from_numpy(e).cuda(), cc, order, et, rect)
    host = x.xxcc_standard_batch(m, e, cc, order, et, rect)
    for b in range(3):
        want = O.xxcc_standard(m[b], e[b], cc, order, et, rect)
        for a, h, w in zip(got, host, want):
            assert tuple(a.shape) == (3,) + w.shape
            assert rel_max(a[b].cpu().numpy(), w) < TOL
            assert np.array_equal(a[b].cpu().numpy(), h[b])            # host and device entry: same kernel


def test_xxcc_standard_rejects_missing_energy(cuda_device, product_lib):
    x = af.XXCC(16)
    m = np.ones((4, 16), np.float32)
    outs = [np.zeros((4, 5), np.float32) for _ in range(3)]
    rc = product_lib.xxccObj_xxccStandardBatch(x._obj, m.ctypes.data, None, 4, 5, 9, 0, 0, outs[0].ctypes.data,
                                               outs[1].ctypes.data, outs[2].ctypes.data, 0, None)
    assert rc != 0 and b"energy" in product_lib.afb200_lastError()


# ------------------------------------------------------------------ CQT chroma / cqcc
def test_chroma_cqcc_golden_legacy(cuda_device, golden):
    g, c = golden("next_rows.npz"), golden("cqt_84.npz")
    q = af.CQT(84, 48000)
    re, im = q.cqt_planes(c["x"])                       # sets the object's timeLength like the reference
    assert rel_max(re, c["re"]) < TOL and rel_max(im, c["im"]) < TOL
    assert rel_max(q.chroma_planes(re, im, 12, D.POWER, CN.MAX), g["chroma_max"]) < TOL
    assert rel_max(q.chroma_planes(re, im, 12, D.MAG, CN.P2), g["chroma_p2"]) < TOL
    assert rel_max(q.cqcc_planes(re * re + im * im, 20), g["cqcc"]) < 2e-4      # error of the CQT itself rides on it
    # reference-layout front door ([num, T] complex in, [chroma, T] out)
    z = (re + 1j * im).T
    assert rel_max(q.chroma(z), g["chroma_max"].T) < TOL


@pytest.mark.parametrize("cn,dt,norm,bpo,num", [(12, 0, 1, 12, 84), (12, 1, 3, 12, 84), (12, 0, 0, 12, 84), (12, 0, 2, 12, 84),
                                                 (12, 1, 4, 12, 84), (12, 0, 1, 24, 96), (24, 0, 1, 24, 96), (6, 1, 3, 12, 48)])
def test_chroma_cqcc_batch_vs_oracle(torch_cuda, cn, dt, norm, bpo, num):
    torch = torch_cuda
    x = np.stack([tones(11, 9000, 32000), noise(12, 9000)])
    q = af.CQT(num, 32000, bin_per_octave=bpo)
    re, im = q.cqt_batch(torch.from_numpy(x).cuda())
    got = q.chroma_batch(re, im, cn, dt, norm).cpu().numpy()
    p = re * re + im * im
    cc = q.cqcc_batch(p, 13).cpu().numpy()
    ren, imn = re.cpu().numpy(), im.cpu().numpy()
    for b in range(2):
        assert rel_max(got[b], O.cqt_chroma(ren[b], imn[b], cn, dt, norm, bpo)) < TOL
        assert rel_max(cc[b], O.xxcc(p[b].cpu().numpy(), 13)) < TOL
    if norm == 1:
        assert np.abs(np.abs(got).max(axis=-1) - 1).max() < 1e-6             # max-normalised rows peak at 1


def test_chroma_rejects_bad_class_count(cuda_device, product_lib):
    q = af.CQT(84, 32000)
    z = np.zeros((4, 84), np.float32)
    out = np.zeros((4, 5), np.float32)
    assert product_lib.cqtObj_chromaBatch(q._obj, z.ctypes.data, z.ctypes.data, 4, 5, 0, 1, out.ctypes.data, 0, None) != 0
    assert b"binPerOctave" in product_lib.afb200_lastError()


# ------------------------------------------------------------------ SpectrogramObj front door
def test_spectrogram_golden_legacy(cuda_device, golden):
    g = golden("next_rows.npz")
    x = g["xsp"]
    sl = af.Spectrogram(samplate=48000, low_fre=100., high_fre=8000., radix2_exp=10, slide_length=256)
    lin, ph = sl.spectrogram_planes(x, True)
    assert lin.shape == g["lin"].shape and rel_max(lin, g["lin"]) < TOL
    m = _phase_mask(g["lin"])
    assert np.abs(ph - g["lin_phase"])[m].max() < 5e-3
    assert np.array_equal(sl.get_bin_band_arr(), g["lin_bin"]) and np.array_equal(sl.get_fre_band_arr(), g["lin_fre"])
    sm = af.MelSpectrogram(num=64, samplate=48000, radix2_exp=10, slide_length=256, data_type=D.MAG)
    sm.set_data_norm_value(0.5)
    mel = sm.spectrogram_planes(x)
    assert rel_max(mel, g["mel_mag"]) < TOL
    np.testing.assert_allclose(sm.get_fre_band_arr(), g["mel_fre"], rtol=2e-6)
    cc = sm.mfcc(np.ascontiguousarray(mel.T), 13).T            # uses the timeLength of the spectrogram call
    assert rel_max(cc, g["mel_cc"]) < TOL
    assert rel_max(sm.xxcc(np.ascontiguousarray(mel.T), 13).T, g["mel_cc"]) < TOL
    # reference layout front door: [num, T]
    assert rel_max(sm.spectrogram(x), g["mel_mag"].T) < TOL


@pytest.mark.parametrize("kw", SPEC_CASES)
def test_spectrogram_batch_vs_oracle(torch_cuda, kw):
    torch = torch_cuda
    sr = kw["samplate"]
    x = np.stack([tones(12, 20000, sr), noise(13, 20000)])
    scale = af.enum_value(kw.get("filter_bank_type", S.LINEAR))
    for dt, nv in ((D.POWER, 1.0), (D.MAG, 1.0), (D.POWER, 0.7), (D.MAG, 1.5)):
        s = af.Spectrogram(data_type=dt, **kw)
        if nv != 1.0:
            s.set_data_norm_value(nv)
        got = s.spectrogram_batch(torch.from_numpy(x).cuda(), scale == 0)
        host = s.spectrogram_batch(x, scale == 0)
        for b in range(2):
            want = O.spectrogram(x[b], kw["num"], sr, kw.get("low_fre"), kw.get("high_fre"), kw.get("bin_per_octave", 12),
                                 kw["radix2_exp"], hop=kw.get("slide_length"), data_type=af.enum_value(dt), scale=scale,
                                 style=af.enum_value(kw.get("style_type", ST.SLANEY)),
                                 norm=af.enum_value(kw.get("normal_type", N.NONE)), norm_value=nv, want_phase=scale == 0)
            if scale == 0:
                assert rel_max(got[0][b].cpu().numpy(), want[0]) < TOL
                m = _phase_mask(want[0])
                assert np.abs(got[1][b].cpu().numpy() - want[1])[m].max() < 5e-3
                assert np.array_equal(got[0][b].cpu().numpy(), host[0][b])
            else:
                assert rel_max(got[b].cpu().numpy(), want) < TOL
                assert np.array_equal(got[b].cpu().numpy(), host[b])


def test_spectrogram_mfcc_batch_is_the_fused_kernel(torch_cuda, golden):
    """MelSpectrogram -> mfcc through the front door == bftObj_mfccBatch bit for bit, and == the reference fixture."""
    torch = torch_cuda
    g = golden("c1_mel_mfcc.npz")
    x = torch.from_numpy(np.stack([g["x"], noise(3, 48000)])).cuda()
    s = af.MelSpectrogram(num=128, samplate=48000, radix2_exp=11, slide_length=512)
    b = af.BFT(128, 11, 48000, slide_length=512, scale_type=S.MEL, data_type=D.POWER)
    n0 = af.lib.get_lib().afb200_kernelLaunchCount()
    a = s.mfcc_batch(x, 40)
    assert af.lib.get_lib().afb200_kernelLaunchCount() - n0 == 1          # one fused launch
    assert torch.equal(a, b.mfcc_batch(x, 40))
    assert rel_max(a[0].cpu().numpy(), g["mfcc"]) < TOL
    mel = s.spectrogram_batch(x)
    assert rel_max(mel[0].cpu().numpy(), g["mel"]) < TOL


def test_next_rows_against_reference_build(torch_cuda, reference):
    """Same calls into oracle/_ref (the unmodified reference, or its stored results) and into libaudioflux_b200."""
    x = tones(21, 24000, 32000)
    for i, kw in enumerate(SPEC_CASES[:8]):
        xr = tones(22, 24000, kw["samplate"])
        want = reference(f"spec{i}", lambda lib: af.Spectrogram(_lib=lib, **kw).spectrogram_planes(xr))
        assert rel_max(af.Spectrogram(**kw).spectrogram_planes(xr), want) < TOL
    # the cqcc input: the oracle's CQT power, regenerated identically wherever the test runs
    o_re, o_im = O.cqt(x, 84, 32000)
    pr = np.ascontiguousarray(o_re * o_re + o_im * o_im, np.float32)

    def cqt(lib):
        q = af.CQT(84, 32000, _lib=lib)
        rr, ir = q.cqt_planes(x)                       # also sets the object's timeLength
        assert rr.shape == pr.shape
        return q.chroma_planes(rr, ir), q.cqcc_planes(pr, 13)
    (chroma_a, cqcc_a), (chroma_r, cqcc_r) = cqt(None), reference("chroma,cqcc", cqt)
    assert rel_max(chroma_a, chroma_r) < 2e-4
    assert rel_max(cqcc_a, cqcc_r) < TOL
    m = (np.random.default_rng(5).random((30, 40)) * 4).astype(np.float32)
    e = (np.random.default_rng(6).random(30) * 2).astype(np.float32)
    for et in (0, 1, 2):
        want = reference(f"xxcc_standard{et}", lambda lib: af.XXCC(40, _lib=lib).xxcc_standard_planes(m, e, 13, 9, et))
        for a, r in zip(af.XXCC(40).xxcc_standard_planes(m, e, 13, 9, et), want):
            assert rel_max(a, r) < TOL


# ------------------------------------------------------------------ STFT padding modes (reflect / wrap / constant values)
from test_next_rows_cpu import PAD_CASES  # noqa: E402


@pytest.mark.parametrize("pos,mode,v1,v2,L,n,hop", PAD_CASES + [(0, 1, 0, 0, 1, 64, 16), (0, 2, 0, 0, 40, 256, 64)])
def test_stft_padding_modes(torch_cuda, pos, mode, v1, v2, L, n, hop):
    torch = torch_cuda
    x = noise(61, L)
    r = int(np.log2(n))
    s = af.STFT(r, af.WindowType.HANN, hop)
    s.enable_padding(True)
    s.set_padding(pos, mode, v1, v2)
    re, im = s.stft_planes(x)                                    # legacy entry: full mirrored planes
    re2, im2 = O.stft(x, n, hop, O.fft_window(O.W_HANN, n), True, pos, mode, v1, v2)
    assert re.shape == re2.shape
    scale = max(np.abs(re2).max(), np.abs(im2).max(), 1e-30)
    assert np.abs(re - re2).max() <= TOL * scale and np.abs(im - im2).max() <= TOL * scale
    xb = np.stack([x, noise(62, L)])
    bre, bim = s.stft_batch(torch.from_numpy(xb).cuda())        # batched device entry: half spectrum
    assert np.abs(bre[0].cpu().numpy() - re2[:, :n // 2 + 1]).max() <= TOL * scale
    assert np.abs(bim[0].cpu().numpy() - im2[:, :n // 2 + 1]).max() <= TOL * scale


def test_stft_padding_against_reference_build(torch_cuda, reference):
    x = tones(63, 5000, 16000)
    for pos in (0, 1, 2):
        for mode in (0, 1, 2):
            def stft(lib):
                s = af.STFT(9, af.WindowType.HAMM, 128, _lib=lib)
                s.enable_padding(True)
                s.set_padding(pos, mode, 1.25, -0.75)
                return s.stft_planes(x)
            (ar, ai), (rr, ri) = stft(None), reference(f"stft{pos}{mode}", stft)
            scale = max(ref_absmax(rr), ref_absmax(ri))
            (ar, rr), (ai, ri) = ref_pair(ar, rr), ref_pair(ai, ri)
            assert np.abs(ar - rr).max() <= TOL * scale and np.abs(ai - ri).max() <= TOL * scale


# ------------------------------------------------------------------ cwtObj_cwtDet
def test_cwt_det_golden_legacy(cuda_device, golden):
    g = golden("next_rows.npz")
    w = af.CWT(12, 10, 48000, wavelet_type=af.WaveletContinueType.MORLET, is_padding=False)
    re0, im0 = w.cwt_det_planes(g["xdet"])
    assert not re0.any() and not im0.any()                        # silent no-op before enableDet, like the reference
    w.enable_det(True)
    re, im = w.cwt_det_planes(g["xdet"])
    scale = max(np.abs(g["det_re"]).max(), np.abs(g["det_im"]).max())
    assert np.abs(re - g["det_re"]).max() <= TOL * scale and np.abs(im - g["det_im"]).max() <= TOL * scale
    w.cwt_planes(g["xdet"])
    re2, im2 = w.cwt_det_planes(None)                             # dataArr = NULL: spectrum of the preceding call
    assert np.array_equal(re2, re) and np.array_equal(im2, im)


@pytest.mark.parametrize("wav,pad,r", [(1, False, 12), (0, False, 12), (3, True, 11), (2, False, 10), (4, False, 13), (1, False, 14)])
def test_cwt_det_batch_vs_oracle(torch_cuda, wav, pad, r):
    torch = torch_cuda
    x = np.stack([noise(71, 1 << r), tones(72, 1 << r, 48000)])
    w = af.CWT(24, r, 48000, wavelet_type=wav, is_padding=pad)
    w.enable_det(True)
    re, im = w.cwt_det_batch(torch.from_numpy(x).cuda())
    for b in range(2):
        r2, i2 = O.cwt(x[b], 24, r, 48000, wav, O.SCALE_OCTAVE, low=32.703196, is_pad=pad, det=True)
        scale = max(np.abs(r2).max(), np.abs(i2).max())
        assert np.abs(re[b].cpu().numpy() - r2).max() <= TOL * scale
        assert np.abs(im[b].cpu().numpy() - i2).max() <= TOL * scale


def test_cwt_det_2pow19_fast_path(torch_cuda):
    """config-4 length: the warp-level FFT legs with the derivative bank; checked on 3 rows against the oracle."""
    torch = torch_cuda
    x = noise(73, 1 << 19)
    w = af.CWT(84, 19, 48000, wavelet_type=af.WaveletContinueType.MORLET, is_padding=False)
    w.enable_det(True)
    re, im = w.cwt_det_batch(torch.from_numpy(x[None]).cuda())
    r2, i2 = O.cwt(x, 84, 19, 48000, O.WAVE_MORLET, O.SCALE_OCTAVE, low=32.703196, det=True)
    for row in (0, 41, 83):
        scale = max(np.abs(r2[row]).max(), np.abs(i2[row]).max())
        assert np.abs(re[0, row].cpu().numpy() - r2[row]).max() <= TOL * scale
        assert np.abs(im[0, row].cpu().numpy() - i2[row]).max() <= TOL * scale


def test_cwt_det_requires_enable(cuda_device, product_lib):
    w = af.CWT(12, 10, 48000)
    x = noise(1, 1024)
    with pytest.raises(af.lib.AfB200Error):
        w.cwt_det_batch(x[None])


# ------------------------------------------------------------------ stftObj_istft
from test_next_rows_cpu import ISTFT_CASES, istft_conditioned  # noqa: E402


@pytest.mark.parametrize("r,hop,wt,method", ISTFT_CASES + [(13, 2048, 1, 0)])
def test_istft(torch_cuda, r, hop, wt, method):
    torch = torch_cuda
    n = 1 << r
    x = np.stack([noise(81, 20 * hop + n), tones(82, 20 * hop + n, 16000)])
    s = af.STFT(r, wt, hop)
    re, im = s.stft_planes(x[0])                                  # full mirrored planes of the CUDA forward path
    got = s.istft_planes(re, im, method)                          # legacy entry, host pointers
    want = O.istft(re, im, n, hop, O.fft_window(wt, n), method)
    ok = istft_conditioned(n, hop, re.shape[0], O.fft_window(wt, n), method)
    assert got.shape == want.shape and np.abs(got - want)[ok].max() <= TOL * np.abs(want).max()
    assert np.abs(got - want).max() <= 1e-2 * np.abs(want).max()
    # batched device entry on the half-spectrum planes stft_batch produces: round trip on the GPU
    xd = torch.from_numpy(x).cuda()
    bre, bim = s.stft_batch(xd)
    y = s.istft_batch(bre, bim, method)
    assert tuple(y.shape) == (2, want.shape[0])
    assert np.abs(y[0].cpu().numpy() - want)[ok].max() <= TOL * np.abs(want).max()
    if hop <= n // 2 and wt in (1, 2):
        assert (y[:, n:-n] - xd[:, n:y.shape[1] - n]).abs().max().item() < 1e-4
    # the reference adds onto the caller's buffer before normalising
    init = noise(83, want.shape[0])
    buf = init.copy()
    af.lib.get_lib().stftObj_istft(s._obj, re.ctypes.data, im.ctypes.data, re.shape[0], method, buf.ctypes.data)
    want2 = O.istft(re, im, n, hop, O.fft_window(wt, n), method, initial=init)
    assert np.abs(buf - want2)[ok].max() <= TOL * np.abs(want2).max()


def test_istft_against_reference_build(torch_cuda, reference):
    x = tones(84, 6000, 16000)
    for wt, method in ((1, 0), (2, 1), (0, 0)):
        # the same STFT planes (the oracle's, regenerated wherever the test runs) go into both inverses
        re, im = (np.ascontiguousarray(p, np.float32) for p in O.stft(x, 512, 128, O.fft_window(wt, 512)))

        def istft(lib):
            s = af.STFT(9, wt, 128, _lib=lib)
            assert s.stft_planes(x)[0].shape == re.shape
            return s.istft_planes(re, im, method)
        ya, yr = istft(None), reference(f"istft{wt}{method}", istft)
        ok = ref_pair(istft_conditioned(512, 128, re.shape[0], O.fft_window(wt, 512), method), yr)[0]
        scale = ref_absmax(yr)
        ya, yr = ref_pair(ya, yr)
        assert np.abs(ya - yr)[ok].max() <= TOL * scale


# ------------------------------------------------------------------ PWT
from test_next_rows_cpu import PWT_CASES, _pwt_oracle  # noqa: E402


@pytest.mark.parametrize("kw", PWT_CASES)
def test_pwt_vs_oracle(torch_cuda, kw):
    torch = torch_cuda
    r = 12
    x = np.stack([noise(91, 1 << r), tones(92, 1 << r, kw["samplate"])])
    p = af.PWT(radix2_exp=r, **kw)
    re, im = p.pwt_planes(x[0])                                   # legacy entry
    r2, i2, fre, bins = _pwt_oracle(x[0], kw, r)
    scale = max(np.abs(r2).max(), np.abs(i2).max())
    assert np.abs(re - r2).max() <= TOL * scale and np.abs(im - i2).max() <= TOL * scale
    assert np.array_equal(p.get_bin_band_arr(), bins)
    bre, bim = p.pwt_batch(torch.from_numpy(x).cuda())            # batched device entry
    assert np.array_equal(bre[0].cpu().numpy(), re) and np.array_equal(bim[0].cpu().numpy(), im)
    r3, i3, _, _ = _pwt_oracle(x[1], kw, r)
    s3 = max(np.abs(r3).max(), np.abs(i3).max())
    assert np.abs(bre[1].cpu().numpy() - r3).max() <= TOL * s3 and np.abs(bim[1].cpu().numpy() - i3).max() <= TOL * s3
    p.enable_det(True)
    p.pwt_planes(x[0])                                            # single-clip call: its spectrum stays in the workspace
    dr, di = p.pwt_det_planes(None)
    d2, e2, _, _ = _pwt_oracle(x[0], kw, r, det=True)
    sd = max(np.abs(d2).max(), np.abs(e2).max())
    assert np.abs(dr - d2).max() <= TOL * sd and np.abs(di - e2).max() <= TOL * sd


def test_pwt_long_clip_and_reference_build(torch_cuda, reference):
    x = tones(93, 1 << 14, 32000)
    ar, ai = af.PWT(84, 14, 32000, is_padding=False).pwt_planes(x)
    rr, ri = reference("pwt", lambda lib: af.PWT(84, 14, 32000, is_padding=False, _lib=lib).pwt_planes(x))
    scale = max(ref_absmax(rr), ref_absmax(ri))
    (ar, rr), (ai, ri) = ref_pair(ar, rr), ref_pair(ai, ri)
    assert np.abs(ar - rr).max() <= TOL * scale and np.abs(ai - ri).max() <= TOL * scale


# ---- streaming STFT (isContinue, stft_algorithm.c:474-599) ----
@pytest.mark.parametrize("r,hop,chunks", [(9, 128, (1000, 37, 500, 3000, 129, 512)), (10, 1024, (700, 700, 2048, 5000, 1)),
                                          (8, 300, (100, 100, 100, 1000, 40, 2000))])
def test_stft_streaming_matches_oracle_reference_and_one_shot(cuda_device, ref_lib, r, hop, chunks):
    """chunk by chunk through stftObj_stft(isContinue = 1): (i) every call equals the oracle's streaming model and the
    reference build fed the same chunks, (ii) all frames together equal the one-shot transform of the whole signal"""
    import audioflux_b200 as af
    n = 1 << r
    x = noise(77, sum(chunks))
    s = af.STFT(r, af.WindowType.HANN, hop, is_continue=True)
    q = af.STFT(r, af.WindowType.HANN, hop, is_continue=True, _lib=ref_lib)
    model = O.StftStream(n, hop, O.fft_window(O.W_HANN, n))
    got, pos = [], 0
    for c in chunks:
        piece = x[pos:pos + c]
        pos += c
        assert s.cal_time_length(c) == q.cal_time_length(c)
        re, im = s.stft_planes(piece)
        wr, wi = model.push(piece)
        rr, ri = q.stft_planes(piece)
        assert re.shape == wr.shape == rr.shape
        if re.shape[0]:
            assert rel_max(re, wr) < 1e-4 and rel_max(im, wi) < 1e-4
            assert rel_max(re, rr) < 1e-4 and rel_max(im, ri) < 1e-4
            got.append(re + 1j * im)
    whole = af.STFT(r, af.WindowType.HANN, hop).stft_planes(x)
    allf = np.concatenate(got)
    T = allf.shape[0]
    assert T == (len(x) - n) // hop + 1 if hop <= n else T > 0
    assert rel_max(allf.real, whole[0][:T]) < 1e-5 and rel_max(allf.imag, whole[1][:T]) < 1e-5


# ---- streaming CQT (isContinue, cqt_algorithm.c:346-456, 923-928, 1317-1319) ----
@pytest.mark.parametrize("chunks", [(3000, 2500, 5000, 1400), (4000, 4000, 2000), (3000, 100, 37, 3000)])
def test_cqt_streaming_matches_oracle_and_reference(cuda_device, ref_lib, chunks):
    """chunk by chunk through cqtObj_cqt(isContinue = 1) against the oracle's streaming model and -- where the reference
    survives the chunk sequence (it corrupts its heap on chunks shorter than a frame) -- the reference build"""
    import audioflux_b200 as af
    sr = 32000
    x = tones(3, sum(chunks), sr)
    c = af.CQT(84, sr, is_continue=True)
    use_ref = min(chunks) >= 512
    q = af.CQT(84, sr, is_continue=True, _lib=ref_lib) if use_ref else None
    model = O.CqtStream(84, sr, norm=O.NORM_AREA)
    pos, total = 0, 0
    for n in chunks:
        piece = x[pos:pos + n]
        pos += n
        T = c.cal_time_length(n)
        re, im = c.cqt_planes(piece)
        wr, wi = model.push(piece)
        assert re.shape[0] == wr.shape[0] == T
        if T:
            assert rel_max(re, wr) < 1e-4 and rel_max(im, wi) < 1e-4
            if use_ref:
                rr, ri = q.cqt_planes(piece)
                assert rel_max(re, rr) < 1e-4 and rel_max(im, ri) < 1e-4
        total += T
    assert total > 0


@pytest.mark.parametrize("num,sr,beta,norm,bpo", [(84, 32000, 5.0, 0, 12), (48, 44100, 2.0, 1, 12), (72, 22050, 10.0, 2, 12),
                                                   (48, 16000, 3.0, 0, 24)])
def test_vqt_vs_oracle_and_reference(cuda_device, reference, num, sr, beta, norm, bpo):
    """VQT (beta != 0, VERDICT r1 missing #5): per-octave kernel sets through the tcgen05 / mma / FP32 octave kernels"""
    import audioflux_b200 as af
    x = (0.1 * np.random.default_rng(3).standard_normal(30000)).astype(np.float32)
    kw = dict(bin_per_octave=bpo, beta=beta, normal_type=af.SpectralFilterBankNormalType(norm))
    z = af.CQT(num, sr, **kw).cqt(x)
    def vqt(lib):
        zr = af.CQT(num, sr, _lib=lib, **kw).cqt(x)
        return np.ascontiguousarray(zr.real), np.ascontiguousarray(zr.imag)
    zr_re, zr_im = reference("vqt", vqt)
    re, im = O.cqt(x, num, sr, bpo=bpo, beta=beta, norm=norm)
    assert rel_max(z.real, re.T) < 1e-4 and rel_max(z.imag, im.T) < 1e-4
    assert rel_max(z.real, zr_re) < 1e-4 and rel_max(z.imag, zr_im) < 1e-4


def test_istft_16384_round_trip(torch_cuda):
    """fftLength 16384 (ADVICE r1): the forward STFT accepted it, the inverse did not -- now an in-place shared-memory path"""
    n, hop = 16384, 4096
    x = noise(5, n + 9 * hop)
    s = af.STFT(14, af.WindowType.HANN, hop)
    re, im = O.stft(x, n, hop, O.fft_window(O.W_HANN, n))
    y = s.istft_planes(re, im, 0)
    want = O.istft(re, im, n, hop, O.fft_window(O.W_HANN, n), 0)
    ok = istft_conditioned(n, hop, re.shape[0], O.fft_window(O.W_HANN, n), 0)
    assert rel_max(y[ok], want[ok]) < 1e-4
    assert rel_max(y[n:-n], x[n:-n]) < 1e-4                          # round trip where four windows overlap


@pytest.mark.parametrize("r,hop,wt,method", [(15, 8192, 1, 0), (16, 20000, 2, 1), (17, 32768, 1, 0)])
def test_istft_long_frames(torch_cuda, r, hop, wt, method):
    """fftLength 2^15 .. 2^20 (VERDICT r1 missing #6, inverse side): Re(IFFT) of a frame through ONE real-input forward
    four-step transform (Hartley identity); full mirrored planes (legacy entry), half planes and a NON-Hermitian full
    spectrum (the reference takes Re(IFFT(X)) of whatever it is given) against the oracle"""
    n = 1 << r
    w = O.fft_window(wt, n)
    x = noise(r, n + 6 * hop)
    s = af.STFT(r, af.WindowType(wt), hop)
    re, im = O.stft(x, n, hop, w)
    ok = istft_conditioned(n, hop, re.shape[0], w, method)
    want = O.istft(re, im, n, hop, w, method)
    y = s.istft_planes(re, im, method)                                       # legacy entry, full planes, host pointers
    assert rel_max(y[ok], want[ok]) < 1e-4
    half = s.istft_batch(np.ascontiguousarray(re[None, :, :n // 2 + 1]), np.ascontiguousarray(im[None, :, :n // 2 + 1]), method)[0]
    assert rel_max(half[ok], want[ok]) < 1e-4
    rng = np.random.default_rng(r)
    re2 = (re + 0.05 * rng.standard_normal(re.shape)).astype(np.float32)     # no longer Hermitian
    im2 = (im + 0.05 * rng.standard_normal(im.shape)).astype(np.float32)
    want2 = O.istft(re2, im2, n, hop, w, method)
    y2 = s.istft_planes(re2, im2, method)
    assert rel_max(y2[ok], want2[ok]) < 1e-4
    if method == 0 and n // hop >= 4:
        assert rel_max(y[n:-n], x[n:-n]) < 1e-4                              # round trip where the windows overlap fully


# ---- streaming spectrogram front door (spectrogramObj_new(isContinue = 1), spectrogram_algorithm.c:655-664) ----
@pytest.mark.parametrize("r,hop,scale,chunks", [(9, 128, "MEL", (1000, 37, 500, 3000, 129, 512)), (10, 1024, "BARK", (700, 700, 2048, 5000, 1)),
                                                (11, 512, "MEL", (5000, 3000, 100, 2048)), (8, 300, "LINEAR", (100, 100, 100, 1000, 40, 2000))])
def test_spectrogram_streaming_matches_reference_and_one_shot(cuda_device, ref_lib, r, hop, scale, chunks):
    """chunk by chunk through spectrogramObj_spectrogram(isContinue = 1): the same frame counts and values as the reference
    build fed the same chunks, and all frames together equal the one-shot transform (to rounding: a chunk may take the general path where the whole clip takes the fused one)"""
    S = af.SpectralFilterBankScaleType
    kw = dict(radix2_exp=r, samplate=16000, slide_length=hop, filter_bank_type=getattr(S, scale))
    num = 40 if scale != "LINEAR" else (1 << r) // 2 + 1
    x = noise(78, sum(chunks))
    s = af.Spectrogram(num, is_continue=True, **kw)
    q = af.Spectrogram(num, is_continue=True, _lib=ref_lib, **kw)
    got, pos = [], 0
    for c in chunks:
        piece = x[pos:pos + c]
        pos += c
        assert s.cal_time_length(c) == q.cal_time_length(c)
        a, b = s.spectrogram_planes(piece), q.spectrogram_planes(piece)
        assert a.shape == b.shape
        if a.shape[0]:
            assert rel_max(a, b) < 1e-4
            got.append(a)
    whole = af.Spectrogram(num, **kw).spectrogram_planes(x)
    allf = np.concatenate(got)
    assert allf.shape[0] == whole.shape[0] or hop > (1 << r)
    assert rel_max(allf, whole[:allf.shape[0]]) < 1e-5
