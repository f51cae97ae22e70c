"""Parity tests proper: the CUDA path, called through the C ABI (legacy host-pointer entry points
and the additive batched/device entry points), against
  * the numpy oracle on the same seeded inputs (sizes the oracle finishes in seconds),
  * fixtures generated from the reference itself (tests/golden),
  * the reference build itself when oracle/_ref travelled to this box,
  * size-independent properties at BASELINE.json's full sizes (batch == loop of singles,
    bit-identical repeats, linearity of the STFT, energy conservation of the FFT).
Tolerance: |a-b| <= 1e-4 * max|b| per tensor (BASELINE.md section 3.6; north_star "1e-4 relative fp32").
"""
import numpy as np
import pytest

import audioflux_b200 as af
from conftest import noise, rel_max, tones
from oracle import af_oracle as O

pytestmark = pytest.mark.gpu

TOL = 1e-4
S, ST, N, D, W = (af.SpectralFilterBankScaleType, af.SpectralFilterBankStyleType,
                  af.SpectralFilterBankNormalType, af.SpectralDataType, af.WindowType)


@pytest.fixture(scope="module")
def torch_cuda(cuda_device):
    import torch
    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    return torch


def mel_bft(**kw):
    return af.BFT(128, 11, 48000, slide_length=512, scale_type=S.MEL, data_type=D.POWER, **kw)


# ------------------------------------------------------------------ STFT
@pytest.mark.parametrize("r,hop,wt", [(11, 512, 1), (9, 100, 2), (10, 1024, 0), (12, 1000, 4), (6, 16, 3),
                                      (13, 4096, 1), (1, 1, 0), (2, 2, 1), (3, 3, 0)])
def test_stft_legacy_full_planes(cuda_device, r, hop, wt):
    x = noise(1, 20000)
    s = af.STFT(r, W(wt), hop)
    re, im = s.stft_planes(x)
    re2, im2 = O.stft(x, 1 << r, hop, O.fft_window(wt, 1 << r))
    assert re.shape == re2.shape
    assert rel_max(re, re2) < TOL and rel_max(im, im2) < TOL


@pytest.mark.parametrize("r,hop,wt,pad", [(15, 8192, 1, False), (16, 30000, 2, False), (17, 65536, 1, True), (19, 100000, 0, False)])
def test_stft_long_frames(cuda_device, r, hop, wt, pad):
    """fftLength 2^15 .. 2^20 (VERDICT r1 missing #6): frames that do not fit a CTA go through the four-step kernels"""
    n = 1 << r
    x = noise(r, 3 * n + 777)
    s = af.STFT(r, W(wt), hop)
    if pad:
        s.enable_padding(True)
    re, im = s.stft_planes(x)
    re2, im2 = O.stft(x, n, hop, O.fft_window(wt, n), is_pad=pad)
    assert re.shape == re2.shape and re.shape[0] >= 2
    assert rel_max(re, re2) < TOL and rel_max(im, im2) < TOL
    # batched half-spectrum entry point and the BFT general path on top of it
    hr, hi = s.stft_batch(np.stack([x, x[::-1].copy()]))
    assert rel_max(hr[0], re2[:, :n // 2 + 1]) < TOL and rel_max(hi[0], im2[:, :n // 2 + 1]) < TOL
    if r == 15:
        b = af.BFT(64, r, 48000, slide_length=hop, scale_type=S.MEL, data_type=D.POWER)
        got = b.bft_batch(x[None, :], result_type=1)[0]
        want = O.bft(x, 64, r, 48000, hop)
        assert rel_max(got, want) < TOL


def test_stft_golden_and_user_window(cuda_device, golden):
    g = golden("stft_512.npz")
    s = af.STFT(9, W.HANN, 128)
    re, im = s.stft_planes(g["x"])
    assert re.shape[0] == int(g["T"])
    assert rel_max(re[:8], g["re"]) < TOL and rel_max(im[:8], g["im"]) < TOL
    w = np.linspace(0.1, 1.0, 512).astype(np.float32)
    s.use_window_data_arr(w)
    re, im = s.stft_planes(g["x"])
    re2, im2 = O.stft(g["x"], 512, 128, w)
    assert rel_max(re, re2) < TOL and rel_max(im, im2) < TOL


def test_stft_padding_center(cuda_device):
    x = noise(2, 5037)
    s = af.STFT(9, W.RECT, 128)
    s.enable_padding(True)
    T = s.cal_time_length(len(x))
    assert T == len(x) // 128 + 1
    re, im = s.stft_planes(x)
    re2, im2 = O.stft(x, 512, 128, np.ones(512), is_pad=True)
    assert rel_max(re, re2) < TOL and rel_max(im, im2) < TOL


def test_stft_batch_device_matches_legacy_and_properties(torch_cuda):
    torch = torch_cuda
    x = np.stack([noise(10 + i, 30000) for i in range(5)])
    s = af.STFT(11, W.HANN, 512)
    re, im = s.stft_batch(torch.from_numpy(x).cuda())
    torch.cuda.synchronize()
    re, im = re.cpu().numpy(), im.cpu().numpy()
    for i in range(5):
        r1, i1 = s.stft_planes(x[i])
        assert np.array_equal(re[i], r1[:, :1025]) and np.array_equal(im[i], i1[:, :1025])   # bit-identical
    # Parseval per frame: sum_k |X_k|^2 (mirrored) == n * sum_n (x w)^2
    w = O.fft_window(1, 2048).astype(np.float64)
    fr = x[0][:2048] * w
    full = np.concatenate([re[0, 0] + 1j * im[0, 0], np.conj((re[0, 0] + 1j * im[0, 0])[1:-1][::-1])])
    assert abs((np.abs(full) ** 2).sum() / (2048 * (fr ** 2).sum()) - 1) < 1e-5
    # linearity: STFT(a x + b y) == a STFT(x) + b STFT(y)
    z = (0.5 * x[0] - 2.0 * x[1]).astype(np.float32)
    rz, iz = s.stft_planes(z)
    assert rel_max(rz[:, :1025], 0.5 * re[0] - 2.0 * re[1]) < TOL


# ------------------------------------------------------------------ BFT
def test_c1_mel_golden_legacy(cuda_device, golden):
    g = golden("c1_mel_mfcc.npz")
    b = mel_bft()
    assert b.cal_time_length(48000) == 90
    mel, _ = b.bft_planes(g["x"], 1)
    assert rel_max(mel, g["mel"]) < TOL
    re, im = b.bft_planes(g["x"], 0)
    assert rel_max(re, g["cre"]) < TOL and rel_max(im, g["cim"]) < TOL
    # reference-shaped wrapper output: (num, T)
    assert b.bft(g["x"], result_type=1).shape == (128, 90)


@pytest.mark.parametrize("scale,style,norm,dt,rt,nv", [
    (2, 0, 0, 0, 1, 1.0), (2, 0, 1, 1, 1, 1.0), (3, 1, 0, 0, 1, 0.5), (4, 0, 2, 1, 1, 2.0), (2, 0, 0, 0, 0, 1.0),
    (3, 0, 1, 1, 0, 1.0), (0, 0, 0, 0, 1, 1.0), (0, 0, 0, 1, 0, 1.0), (5, 0, 0, 0, 1, 1.0), (6, 1, 1, 1, 1, 1.0),
    (1, 4, 1, 0, 1, 1.0), (2, 5, 2, 0, 1, 1.0), (4, 10, 0, 1, 1, 1.0)])
def test_bft_modes_vs_oracle(cuda_device, scale, style, norm, dt, rt, nv):
    x = noise(2, 20000)
    kw = {}
    if scale == 6:
        kw = dict(low_fre=32.703196, high_fre=16000.)
    if scale == 1:
        kw = dict(low_fre=1000.0, high_fre=20000.0)
    b = af.BFT(64, 10, 44100, slide_length=256, scale_type=S(scale), style_type=ST(style), normal_type=N(norm),
               data_type=D(dt), **kw)
    if nv != 1.0:
        b.set_data_norm_value(nv)
    re, im = b.bft_planes(x, rt)
    low = kw.get("low_fre", 32.703196 if scale in (5, 6) else None)
    o = O.bft(x, 64, 10, 44100, 256, 1, scale, style, norm, dt, low=low, high=kw.get("high_fre"),
              result_type=rt, norm_value=nv)
    if rt == 1:
        assert rel_max(re, o) < TOL
    else:
        assert rel_max(re, o[0]) < TOL and rel_max(im, o[1]) < TOL


def test_bark_etsi_golden(cuda_device, golden):
    g = golden("bark_etsi_mag.npz")
    b = af.BFT(64, 10, 48000, slide_length=256, scale_type=S.BARK, style_type=ST.ETSI, normal_type=N.AREA, data_type=D.MAG)
    m, _ = b.bft_planes(g["x"], 1)
    assert rel_max(m, g["mel"]) < TOL
    xx = af.XXCC(64)
    assert rel_max(xx.xxcc_planes(g["mel"], 20), g["cc"]) < TOL
    assert rel_max(xx.xxcc_planes(g["mel"], 13, af.CepstralRectifyType.CUBIC_ROOT), g["cc_cubic"]) < TOL


def test_gammatone_dense_bank_golden(torch_cuda, golden):
    """Dense (gammatone) bank: tiled FP32 contraction path, real and complex modes, and the composed MFCC."""
    torch = torch_cuda
    g = golden("erb_gammatone.npz")
    b = af.BFT(64, 10, 32000, slide_length=256, scale_type=S.ERB, style_type=ST.GAMMATONE, data_type=D.POWER)
    m, _ = b.bft_planes(g["x"], 1)
    assert rel_max(m, g["mel"]) < TOL
    cc = b.mfcc_batch(torch.from_numpy(g["x"][None]).cuda(), 13)
    torch.cuda.synchronize()
    assert rel_max(cc[0].cpu().numpy(), g["cc"]) < TOL
    re, im = b.bft_planes(g["x"], 0)
    ore, oim = O.bft(g["x"], 64, 10, 32000, 256, O.W_HANN, O.SCALE_ERB, O.STYLE_GAMMATONE, 0, 0, result_type=0, bank=g["bank"])
    assert rel_max(re, ore) < TOL and rel_max(im, oim) < TOL


# ------------------------------------------------------------------ xxcc
def test_xxcc_vs_oracle(cuda_device):
    m = np.abs(noise(3, 50 * 128).reshape(50, 128)) + 1e-9
    m[3, :5] = 0.0                      # exercises the 1e-8 log floor
    m[4] = 0.0                          # an all-empty frame
    x = af.XXCC(128)
    assert rel_max(x.xxcc_planes(m, 40), O.xxcc(m, 40)) < TOL
    assert rel_max(x.xxcc_planes(m, 128), O.xxcc(m, 128)) < TOL
    x2 = af.XXCC(60)
    assert rel_max(x2.xxcc_planes(m[:, :60], 13), O.xxcc(m[:, :60], 13)) < TOL
    # reference-shaped wrapper: (num, T) -> (cc, T)
    assert x.xxcc(m.T, 13).shape == (13, 50)


# ------------------------------------------------------------------ fused MFCC
def test_mfcc_fused_golden_c1(torch_cuda, golden):
    torch = torch_cuda
    g = golden("c1_mel_mfcc.npz")
    b = mel_bft()
    out = b.mfcc_batch(torch.from_numpy(g["x"][None]).cuda(), 40)
    torch.cuda.synchronize()
    out = out.cpu().numpy()[0]
    assert out.shape == (90, 40)
    assert rel_max(out, g["mfcc"]) < TOL
    # host-pointer flavour of the same entry point
    out2 = b.mfcc_batch(g["x"][None], 40)[0]
    assert np.array_equal(out, out2)


@pytest.mark.parametrize("hop,cc,norm,dt,rect,L", [(512, 40, 0, 0, 0, 48000), (512, 13, 1, 0, 0, 30720), (256, 20, 0, 1, 0, 20480),
                                                    (1024, 40, 0, 0, 1, 40960), (512, 64, 2, 0, 0, 22528), (2048, 24, 0, 0, 0, 30720),
                                                    (128, 40, 0, 0, 0, 8192), (512, 40, 0, 0, 0, 2048)])
def test_mfcc_fused_vs_oracle(torch_cuda, hop, cc, norm, dt, rect, L):
    torch = torch_cuda
    B = 3
    x = np.stack([noise(20 + i, L) if i != 1 else tones(21, L, 48000) for i in range(B)])
    b = af.BFT(128, 11, 48000, slide_length=hop, scale_type=S.MEL, normal_type=N(norm), data_type=D(dt))
    out = b.mfcc_batch(torch.from_numpy(x).cuda(), cc, af.CepstralRectifyType(rect))
    torch.cuda.synchronize()
    out = out.cpu().numpy()
    T = (L - 2048) // hop + 1
    assert out.shape == (B, T, cc)
    for i in range(B):
        mel = O.bft(x[i], 128, 11, 48000, hop, O.W_HANN, O.SCALE_MEL, O.STYLE_SLANEY, norm, dt, result_type=1)
        want = O.xxcc(mel, cc, rect)
        assert rel_max(out[i], want) < TOL, (i, rel_max(out[i], want))


@pytest.mark.parametrize("scale,style,norm,num,sr,dt", [(S.MEL, ST.SLANEY, N.NONE, 128, 48000, D.POWER),
                                                         (S.MEL, ST.SLANEY, N.AREA, 128, 48000, D.POWER),
                                                         (S.MEL, ST.SLANEY, N.BAND_WIDTH, 128, 48000, D.MAG),
                                                         (S.BARK, ST.ETSI, N.AREA, 64, 48000, D.POWER),
                                                         (S.ERB, ST.SLANEY, N.NONE, 128, 48000, D.POWER),
                                                         (S.MEL, ST.ETSI, N.NONE, 128, 48000, D.POWER),
                                                         (S.MEL, ST.HANN, N.NONE, 128, 48000, D.POWER),
                                                         (S.MEL, ST.SLANEY, N.NONE, 40, 16000, D.POWER),
                                                         (S.ERB, ST.ETSI, N.BAND_WIDTH, 77, 22050, D.MAG)])
def test_mfcc_fused_bank_loop_modes(torch_cuda, product_lib, monkeypatch, scale, style, norm, num, sr, dt):
    """The fused kernel has two bank loops: the interval ("shared product") form for triangular banks and the
    filter-per-lane loop for any banded bank.  Both against the oracle, and against each other."""
    torch = torch_cuda
    x = np.stack([tones(31, 20480, sr), noise(32, 20480)])
    xd = torch.from_numpy(x).cuda()
    cc = min(20, num)
    outs = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("AFB200_MFCC_BANK_MODE", mode)
        b = af.BFT(num, 11, sr, slide_length=512, scale_type=scale, style_type=style, normal_type=norm, data_type=dt)
        outs[mode] = b.mfcc_batch(xd, cc).cpu().numpy()
        # every bank above has the structure; -1 = this shape is outside the fused kernel (composed path)
        assert product_lib.bftObj_mfccPlanMode(b._obj) in (int(mode), -1)
    lo, hi, _, _ = O.bft_revise_range(num, 2048, sr, None, None, af.enum_value(scale), 12)
    bank, _, _ = O.auditory_filterbank(num, 2048, sr, af.enum_value(scale), af.enum_value(style), af.enum_value(norm),
                                       float(lo), float(hi), 12)
    for i in range(2):
        mel = O.bft(x[i], num, 11, sr, 512, scale=af.enum_value(scale), data_type=af.enum_value(dt), bank=bank)
        want = O.xxcc(mel, cc)
        assert rel_max(outs["1"][i], want) < TOL
        assert rel_max(outs["0"][i], want) < TOL
    assert rel_max(outs["1"], outs["0"]) < 2e-5


def test_mfcc_fused_non_triangular_bank_uses_filter_loop(torch_cuda, product_lib):
    torch = torch_cuda
    x = noise(33, 20480)
    b = af.BFT(128, 11, 48000, slide_length=512, scale_type=S.MEL, style_type=ST.RECT, data_type=D.POWER)
    got = b.mfcc_batch(torch.from_numpy(x[None]).cuda(), 13).cpu().numpy()[0]
    assert product_lib.bftObj_mfccPlanMode(b._obj) == 0
    mel = O.bft(x, 128, 11, 48000, 512, scale=O.SCALE_MEL, style=O.STYLE_RECT)
    assert rel_max(got, O.xxcc(mel, 13)) < TOL


def test_mfcc_host_pointer_pipeline(torch_cuda):
    """Host-pointer entry: the batch flows through the library's chunked copy-in / transform / copy-out pipeline
    (3 chunks here, the last one partial); pageable and page-locked buffers, result bit-identical to the device entry."""
    torch = torch_cuda
    B, L = 150, 240000
    xh = torch.empty((B, L), dtype=torch.float32).pin_memory()
    g = torch.Generator().manual_seed(5)
    xh.copy_(0.1 * torch.randn((B, L), generator=g))
    b = mel_bft()
    want = b.mfcc_batch(xh.cuda(), 40).cpu().numpy()
    got_pageable = b.mfcc_batch(xh.numpy().copy(), 40)
    assert np.array_equal(got_pageable, want)
    oh = torch.empty((B, b.cal_time_length(L), 40), dtype=torch.float32).pin_memory()
    for _ in range(2):                                            # second call reuses the slots
        oh.zero_()
        ret = b.mfcc_batch(xh.numpy(), 40, out=oh.numpy())
        assert ret.ctypes.data == oh.numpy().ctypes.data and np.array_equal(oh.numpy(), want)
    small = b.mfcc_batch(xh.numpy()[:3], 40)                       # fewer clips than one chunk
    assert np.array_equal(small, want[:3])


def test_host_pointer_pipelines_bft_cqt_stft(torch_cuda):
    """Every batched host-pointer entry point runs the same chunked 3-stream pipeline (af_pipe_run): several chunks,
    the last one partial, results bit-identical to the device-pointer entry."""
    torch = torch_cuda
    g = torch.Generator().manual_seed(6)
    x = (0.1 * torch.randn((100, 240000), generator=g)).numpy()
    xd = torch.from_numpy(x).cuda()
    b = mel_bft()
    assert np.array_equal(b.bft_batch(x), b.bft_batch(xd).cpu().numpy())                  # 64 + 36 clips
    hr, hi = b.bft_batch(x[:70], 0)                                                        # complex mode: two planes
    dr, di = b.bft_batch(xd[:70], 0)
    assert np.array_equal(hr, dr.cpu().numpy()) and np.array_equal(hi, di.cpu().numpy())
    c = af.CQT(84, 48000)
    hre, him = c.cqt_batch(x)
    dre, dim = c.cqt_batch(xd)
    assert np.array_equal(hre, dre.cpu().numpy()) and np.array_equal(him, dim.cpu().numpy())   # 48 + 48 + 4 clips
    s = af.STFT(11, W.HANN, 512)
    hre, him = s.stft_batch(x[:40])
    dre, dim = s.stft_batch(xd[:40])
    assert np.array_equal(hre, dre.cpu().numpy()) and np.array_equal(him, dim.cpu().numpy())   # 16 + 16 + 8 clips


@pytest.mark.parametrize("scale,style,norm,dt,num,fused", [(S.MEL, ST.SLANEY, N.NONE, D.POWER, 128, 1), (S.MEL, ST.SLANEY, N.AREA, D.MAG, 128, 1),
                                                            (S.BARK, ST.SLANEY, N.BAND_WIDTH, D.POWER, 128, 0),   # filters too wide
                                                            (S.ERB, ST.ETSI, N.NONE, D.MAG, 96, 1)])
def test_bft_real_mode_fused_bank_output(torch_cuda, product_lib, monkeypatch, scale, style, norm, dt, num, fused):
    """Real-mode BFT at fftLength 2048 = the fused kernel stopped after the filter bank (ONE launch); against the
    oracle and against the general STFT -> bank composition (AFB200_BFT_GENERAL=1)."""
    torch = torch_cuda
    x = np.stack([tones(41, 30720, 48000), noise(42, 30720)])
    xd = torch.from_numpy(x).cuda()
    b = af.BFT(num, 11, 48000, slide_length=512, scale_type=scale, style_type=style, normal_type=norm, data_type=dt)
    n0 = product_lib.afb200_kernelLaunchCount()
    got = b.bft_batch(xd).cpu().numpy()
    assert product_lib.afb200_kernelLaunchCount() - n0 == (1 if fused else 2)
    monkeypatch.setenv("AFB200_BFT_GENERAL", "1")
    n0 = product_lib.afb200_kernelLaunchCount()
    general = b.bft_batch(xd).cpu().numpy()
    assert product_lib.afb200_kernelLaunchCount() - n0 == 2                      # STFT + bank
    monkeypatch.delenv("AFB200_BFT_GENERAL")
    for i in range(2):
        want = O.bft(x[i], num, 11, 48000, 512, scale=af.enum_value(scale), style=af.enum_value(style),
                     norm=af.enum_value(norm), data_type=af.enum_value(dt))
        assert rel_max(got[i], want) < TOL and rel_max(general[i], want) < TOL
    assert rel_max(got, general) < 2e-5
    # a norm value other than 1 keeps the general composition (pow before / after the bank)
    b.set_data_norm_value(0.5)
    n0 = product_lib.afb200_kernelLaunchCount()
    b.bft_batch(xd)
    assert product_lib.afb200_kernelLaunchCount() - n0 == 2


def test_mfcc_fused_equals_composed_path(torch_cuda):
    """fused kernel == bft_batch(result_type=1) -> xxcc_batch (general kernels), and other banks
    that fit the fused plan (bark / erb, ETSI) agree with the oracle too."""
    torch = torch_cuda
    x = np.stack([noise(30 + i, 40960) for i in range(4)])
    xd = torch.from_numpy(x).cuda()
    for scale, style, num in ((2, 0, 128), (3, 0, 64), (4, 1, 40), (2, 1, 80)):
        b = af.BFT(num, 11, 48000, slide_length=512, scale_type=S(scale), style_type=ST(style), data_type=D.POWER)
        fused = b.mfcc_batch(xd, 20)
        mel = b.bft_batch(xd, result_type=1)
        comp = af.XXCC(num).xxcc_batch(mel, 20)
        torch.cuda.synchronize()
        assert rel_max(fused.cpu().numpy(), comp.cpu().numpy()) < TOL
        want = O.xxcc(O.bft(x[0], num, 11, 48000, 512, O.W_HANN, scale, style, 0, 0, result_type=1), 20)
        assert rel_max(fused[0].cpu().numpy(), want) < TOL


def test_mfcc_general_path_other_fft_lengths(torch_cuda):
    torch = torch_cuda
    x = np.stack([noise(40 + i, 16000) for i in range(2)])
    for r, hop, num in ((10, 256, 64), (9, 160, 40), (12, 1024, 128)):
        b = af.BFT(num, r, 16000, slide_length=hop, scale_type=S.MEL, data_type=D.POWER)
        out = b.mfcc_batch(torch.from_numpy(x).cuda(), 13)
        torch.cuda.synchronize()
        want = O.xxcc(O.bft(x[1], num, r, 16000, hop, O.W_HANN, O.SCALE_MEL, 0, 0, 0, result_type=1), 13)
        assert rel_max(out[1].cpu().numpy(), want) < TOL


def test_mfcc_full_size_properties(torch_cuda):
    """BASELINE config 2 shape (reduced batch keeps this test short; the bench runs the full 1024):
    bit-identical repeats, batch == loop of singles, any clip == oracle."""
    torch = torch_cuda
    B, L = 96, 240000
    g = torch.Generator(device="cuda").manual_seed(1234)
    xd = 0.1 * torch.randn((B, L), generator=g, device="cuda", dtype=torch.float32)
    b = mel_bft()
    o1 = b.mfcc_batch(xd, 40)
    o2 = b.mfcc_batch(xd, 40)
    torch.cuda.synchronize()
    assert o1.shape == (B, 465, 40)
    assert torch.equal(o1, o2)                                   # bit-pattern stable across runs
    single = b.mfcc_batch(xd[17:18].contiguous(), 40)
    sub = b.mfcc_batch(xd[5:29].contiguous(), 40)
    torch.cuda.synchronize()
    assert torch.equal(single[0], o1[17]) and torch.equal(sub, o1[5:29])   # independent of batch size / position
    x = xd[17].cpu().numpy()
    want = O.mfcc(x, 48000, 11, 512, 128, 40)
    assert rel_max(o1[17].cpu().numpy(), want) < TOL
    assert torch.isfinite(o1).all()


def test_mfcc_against_reference_build(torch_cuda, reference):
    torch = torch_cuda
    x = np.stack([noise(50 + i, 240000) for i in range(2)])
    b = mel_bft()
    out = b.mfcc_batch(torch.from_numpy(x).cuda(), 40)
    torch.cuda.synchronize()

    def ref(lib):
        r, xx = mel_bft(_lib=lib), af.XXCC(128, _lib=lib)
        return tuple(xx.xxcc_planes(r.bft_planes(x[i], 1)[0], 40) for i in range(2))
    for i, want in enumerate(reference("mfcc", ref)):
        assert rel_max(out[i].cpu().numpy(), want) < TOL


# ------------------------------------------------------------------ CQT
def test_cqt_golden(cuda_device, golden):
    g = golden("cqt_84.npz")
    c = af.CQT(84, 48000)
    assert c.fft_length == int(g["fft_length"])
    re, im = c.cqt_planes(g["x"])
    assert re.shape == g["re"].shape
    assert rel_max(re, g["re"]) < TOL and rel_max(im, g["im"]) < TOL
    assert c.cqt(g["x"]).shape == (84, re.shape[0])


@pytest.mark.parametrize("L,sr,norm,hop,scale,num,bpo", [(48037, 48000, 1, None, True, 84, 12), (30000, 32000, 0, None, True, 84, 12),
                                                          (22050, 22050, 2, 64, False, 84, 12), (16000, 44100, 1, None, True, 48, 24),
                                                          (5000, 48000, 1, 256, True, 36, 12)])
def test_cqt_vs_oracle(torch_cuda, L, sr, norm, hop, scale, num, bpo):
    torch = torch_cuda
    x = np.stack([noise(60 + i, L) for i in range(2)])
    fmin = 32.703196 if num // bpo >= 4 else 261.6256
    c = af.CQT(num, sr, low_fre=fmin, bin_per_octave=bpo, normal_type=N(norm), slide_length=hop, is_scale=scale)
    re, im = c.cqt_batch(torch.from_numpy(x).cuda())
    torch.cuda.synchronize()
    re2, im2 = O.cqt(x[1], num, sr, fmin, bpo, norm=norm, hop=hop, is_scale=scale)
    assert tuple(re.shape[1:]) == re2.shape
    assert rel_max(re[1].cpu().numpy(), re2) < TOL and rel_max(im[1].cpu().numpy(), im2) < TOL
    r1, i1 = c.cqt_planes(x[1])
    assert np.array_equal(r1, re[1].cpu().numpy())             # legacy entry point == batched entry point


def test_cqt_5s_clip_against_reference_build(torch_cuda, reference):
    torch = torch_cuda
    x = noise(70, 240000)
    c = af.CQT(84, 48000)
    assert c.cal_time_length(240000) == 1876
    re, im = c.cqt_batch(torch.from_numpy(x[None]).cuda())
    torch.cuda.synchronize()
    re2, im2 = reference("cqt", lambda lib: af.CQT(84, 48000, _lib=lib).cqt_planes(x))
    assert rel_max(re[0].cpu().numpy(), re2) < TOL and rel_max(im[0].cpu().numpy(), im2) < TOL


# ------------------------------------------------------------------ CWT
def test_cwt_golden(cuda_device, golden):
    g = golden("cwt_morlet.npz")
    w = af.CWT(36, 11, 48000, wavelet_type=af.WaveletContinueType.MORLET, is_padding=False)
    re, im = w.cwt_planes(g["x"])
    assert rel_max(re, g["re"]) < TOL and rel_max(im, g["im"]) < TOL
    np.testing.assert_allclose(w.get_fre_band_arr(), g["fre"], rtol=1e-6)


@pytest.mark.parametrize("r,wav,scale,pad", [(12, 1, 5, False), (12, 0, 5, False), (12, 2, 5, False), (11, 3, 5, False),
                                             (11, 4, 5, False), (11, 5, 5, False), (11, 6, 5, False), (11, 7, 5, False),
                                             (12, 1, 2, False), (12, 0, 3, False), (12, 1, 5, True), (10, 1, 0, False),
                                             (14, 1, 5, False), (16, 1, 5, False), (15, 0, 5, True)])
def test_cwt_vs_oracle(torch_cuda, r, wav, scale, pad):
    torch = torch_cuda
    x = np.stack([noise(80 + i, 1 << r) for i in range(2)])
    kw = dict(low_fre=1000.) if scale == 0 else {}
    w = af.CWT(40 if scale == 0 else 84, r, 48000, wavelet_type=af.WaveletContinueType(wav), scale_type=S(scale),
               is_padding=pad, **kw)
    re, im = w.cwt_batch(torch.from_numpy(x).cuda())
    torch.cuda.synchronize()
    re2, im2 = O.cwt(x[1], w.num, r, 48000, wav, scale, low=kw.get("low_fre", 32.703196 if scale in (5, 6) else None), is_pad=pad)
    assert rel_max(re[1].cpu().numpy(), re2) < TOL and rel_max(im[1].cpu().numpy(), im2) < TOL


def test_cwt_2pow19_properties(torch_cuda):
    """BASELINE config 4 length (N = 2^19, 84 morlet scales, isPad=0), one clip: the oracle's numpy FFT
    finishes in seconds at this size, so it is compared directly; plus analytic-signal property
    (no negative-frequency content) via linearity on a pure tone."""
    torch = torch_cuda
    N = 1 << 19
    x = np.zeros(N, np.float32)
    x[:480000] = noise(90, 480000)
    w = af.CWT(84, 19, 48000, wavelet_type=af.WaveletContinueType.MORLET, is_padding=False)
    re, im = w.cwt_batch(torch.from_numpy(x[None]).cuda())
    torch.cuda.synchronize()
    re2, im2 = O.cwt(x, 84, 19, 48000, O.WAVE_MORLET, O.SCALE_OCTAVE, low=32.703196, is_pad=False)
    assert rel_max(re[0].cpu().numpy(), re2) < TOL and rel_max(im[0].cpu().numpy(), im2) < TOL
    r2, i2 = w.cwt_batch(torch.from_numpy(x[None]).cuda())
    torch.cuda.synchronize()
    assert torch.equal(re, r2) and torch.equal(im, i2)
