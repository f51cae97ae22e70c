"""Pins the numpy restatement (oracle/af_oracle.py) to the reference compiled in oracle/_ref.  The tests that take the
`reference` fixture read the reference's stored results (tests/golden/ref) where that library is absent; the others skip."""
import ctypes as C

import numpy as np
import pytest

import audioflux_b200 as af
from conftest import noise, ref_pair, ref_window, rel_max
from oracle import af_oracle as O

S, ST, N, D, W = (af.SpectralFilterBankScaleType, af.SpectralFilterBankStyleType,
                  af.SpectralFilterBankNormalType, af.SpectralDataType, af.WindowType)


@pytest.mark.parametrize("wt", range(14))
def test_windows(reference, wt):
    for n in (16, 512, 2048):
        w = reference(f"window{n}", lambda lib: ref_window(lib, wt, n))
        o, w = ref_pair(O.fft_window(wt, n), w)
        assert np.abs(w - o).max() < 2e-6


def _ref_bank(ref, num, n, sr, scale, style, norm, low, high, bpo):
    bank = np.zeros((num + 4, n // 2 + 1), np.float32)
    fb = np.zeros(num + 2, np.float32)
    bb = np.zeros(num + 2, np.int32)
    ref.auditory_filterBank(num, n, sr, 0, scale, style, norm, low, high, bpo, bank.ctypes.data, fb.ctypes.data, bb.ctypes.data)
    return bank[:num], fb[:num], bb[:num]


def bank_cases():
    for scale in range(1, 7):
        for style in (0, 1, 3, 4, 5, 6, 7, 8, 9, 10):
            for norm in (0, 1, 2):
                yield scale, style, norm


@pytest.mark.parametrize("scale,style,norm", list(bank_cases()))
def test_filter_banks(ref_lib, scale, style, norm):
    for num, n, sr in ((128, 2048, 48000), (40, 1024, 16000)):
        low = 32.703196 if scale in (5, 6) else None
        high = None
        if scale == 1:                       # the reference writes out of bounds when revised edges leave [0, sr/2]
            low, high = 1000.0, sr / 2 - 1000.0
        if scale == 6:
            low, high = 32.703196, sr / 2 * 0.8
        lo, hi, _, _ = O.bft_revise_range(num, n, sr, low, high, scale, 12)
        if scale == 5 and float(hi) > sr / 2:
            continue
        b1, f1, i1 = _ref_bank(ref_lib, num, n, sr, scale, style, norm, float(lo), float(hi), 12)
        b2, f2, i2 = O.auditory_filterbank(num, n, sr, scale, style, norm, float(lo), float(hi), 12)
        assert np.array_equal(i1, i2)
        assert np.abs(b1 - b2).max() <= 5e-5 * max(1.0, np.abs(b1).max())
        np.testing.assert_allclose(f1, f2, rtol=2e-6, atol=1e-3)


@pytest.mark.parametrize("r,hop,wt", [(11, 512, 1), (9, 100, 2), (10, 1024, 0), (12, 1000, 4)])
def test_stft(reference, r, hop, wt):
    x = noise(1, 20000)
    re, im = reference("stft", lambda lib: af.STFT(r, W(wt), hop, _lib=lib).stft_planes(x))
    re2, im2 = O.stft(x, 1 << r, hop, O.fft_window(wt, 1 << r))
    assert rel_max(re2, re) < 2e-6 and rel_max(im2, im) < 2e-6


@pytest.mark.parametrize("scale,style,norm,dt,rt,nv", [
    (2, 0, 0, 0, 1, 1.0), (2, 0, 1, 1, 1, 1.0), (3, 1, 0, 0, 1, 0.5), (4, 0, 2, 1, 1, 2.0), (2, 0, 0, 0, 0, 1.0),
    (3, 0, 1, 1, 0, 1.0), (0, 0, 0, 0, 1, 1.0), (0, 0, 0, 1, 0, 1.0), (5, 0, 0, 0, 1, 1.0), (6, 1, 1, 1, 1, 1.0)])
def test_bft_modes(reference, scale, style, norm, dt, rt, nv):
    x = noise(2, 20000)
    kw = dict(low_fre=32.703196, high_fre=16000.) if scale == 6 else {}

    def ref(lib):
        b = af.BFT(64, 10, 44100, slide_length=256, scale_type=S(scale), style_type=ST(style), normal_type=N(norm),
                   data_type=D(dt), _lib=lib, **kw)
        if nv != 1.0:
            b.set_data_norm_value(nv)
        re, im = b.bft_planes(x, rt)
        return (re,) if rt == 1 else (re, im)
    re, im = (reference("bft", ref) + (None,))[:2]
    o = O.bft(x, 64, 10, 44100, 256, 1, scale, style, norm, dt, low=32.703196 if scale in (5, 6) else None,
              high=kw.get("high_fre"), result_type=rt, norm_value=nv)
    if rt == 1:
        assert rel_max(o, re) < 2e-5
    else:
        assert rel_max(o[0], re) < 2e-5 and rel_max(o[1], im) < 2e-5


def test_xxcc(reference):
    m = np.abs(noise(3, 50 * 128).reshape(50, 128)) + 1e-9
    m[3, :5] = 0.0

    def ref(lib):
        x, x2 = af.XXCC(128, _lib=lib), af.XXCC(60, _lib=lib)    # 60: not a power of two -> dense DCT in the reference
        return x.xxcc_planes(m, 40), x2.xxcc_planes(m[:, :60], 13), x.xxcc_planes(m, 20, af.CepstralRectifyType.CUBIC_ROOT)
    for want, got in zip(reference("xxcc", ref), (O.xxcc(m, 40), O.xxcc(m[:, :60], 13), O.xxcc(m, 20, O.RECT_CUBIC))):
        g, w = ref_pair(got, want)
        assert np.abs(g - w).max() < 2e-5


def test_decimator(reference):
    x = noise(4, 20001)

    def ref(lib):
        ro = C.c_void_p()
        lib.resampleObj_new.argtypes = [C.POINTER(C.c_void_p), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
        lib.resampleObj_new(C.byref(ro), C.byref(C.c_int(2)), C.byref(C.c_int(1)), None)
        lib.resampleObj_setSamplate.argtypes = [C.c_void_p, C.c_int, C.c_int]
        lib.resampleObj_setSamplate(ro, 2, 1)
        lib.resampleObj_resample.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        lib.resampleObj_resample.restype = C.c_int
        out = np.zeros(len(x), np.float32)
        n = lib.resampleObj_resample(ro, x.ctypes.data, len(x), out.ctypes.data)
        return np.array(n), out[:n]
    n, out = reference("resample", ref)
    y = O.resample_down2(x)
    assert n == len(y) == len(x) // 2
    assert rel_max(y, out) < 2e-6


@pytest.mark.parametrize("L,sr,norm,hop,scale", [(48037, 48000, 1, None, True), (30000, 32000, 0, None, True),
                                                  (22050, 22050, 2, 64, False)])
def test_cqt(reference, L, sr, norm, hop, scale):
    x = noise(5, L)
    re, im = reference("cqt", lambda lib: af.CQT(84, sr, normal_type=N(norm), slide_length=hop, is_scale=scale, _lib=lib).cqt_planes(x))
    re2, im2 = O.cqt(x, 84, sr, norm=norm, hop=hop, is_scale=scale)
    assert rel_max(re2, re) < 1e-5 and rel_max(im2, im) < 1e-5


@pytest.mark.parametrize("r,wav,scale,pad", [(12, 1, 5, False), (12, 0, 5, False), (12, 2, 5, False), (11, 3, 5, False),
                                             (11, 4, 5, False), (11, 5, 5, False), (11, 6, 5, False), (11, 7, 5, False),
                                             (12, 1, 2, False), (12, 0, 3, False), (12, 1, 5, True), (10, 1, 0, False)])
def test_cwt(reference, r, wav, scale, pad):
    x = noise(6, 1 << r)
    kw = dict(low_fre=1000.) if scale == 0 else {}
    num = 40 if scale == 0 else 84
    re, im = reference("cwt", lambda lib: af.CWT(num, r, 48000, wavelet_type=af.WaveletContinueType(wav), scale_type=S(scale),
                                                  is_padding=pad, _lib=lib, **kw).cwt_planes(x))
    re2, im2 = O.cwt(x, num, r, 48000, wav, scale, low=kw.get("low_fre", 32.703196 if scale in (5, 6) else None), is_pad=pad)
    assert rel_max(re2, re) < 1e-5 and rel_max(im2, im) < 1e-5


@pytest.mark.parametrize("num,n,sr,scale,norm", [(64, 1024, 32000, 4, 0), (64, 1024, 32000, 4, 1), (40, 2048, 16000, 2, 2),
                                                  (128, 2048, 48000, 4, 0), (32, 512, 22050, 3, 1), (24, 1024, 44100, 1, 0)])
def test_gammatone_bank(ref_lib, num, n, sr, scale, norm):
    lo, hi = (100.0, sr / 2 - 100.0) if scale == 1 else (0.0, sr / 2)
    b = np.zeros((num + 4, n // 2 + 1), np.float32)
    f = np.zeros(num + 2, np.float32)
    bi = np.zeros(num + 2, np.int32)
    ref_lib.auditory_filterBank(num, n, sr, 0, scale, 2, norm, C.c_float(lo), C.c_float(hi), 12, b.ctypes.data, f.ctypes.data,
                                bi.ctypes.data)
    ob, of, obi = O.auditory_filterbank(num, n, sr, scale, O.STYLE_GAMMATONE, norm, lo, hi)
    assert np.array_equal(obi, bi[:num])
    np.testing.assert_allclose(of, f[:num], rtol=2e-6, atol=1e-3)
    assert (np.abs(ob - b[:num]).max(axis=1) <= 2e-5 * np.maximum(b[:num].max(axis=1), 1e-30)).all()
    # given the reference's own centre frequencies the restatement is bit-exact (area norm: up to its summation order)
    exact = O.gammatone_bank(num, n, sr, norm, f[:num])
    assert (np.abs(exact - b[:num]).max(axis=1) <= (1e-5 if norm == 1 else 0.0) * np.maximum(b[:num].max(axis=1), 1e-30)).all()
