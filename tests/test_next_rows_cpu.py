"""SURVEY section 8(f) rows -- xxccStandard, CQT chroma / cqcc, SpectrogramObj front door -- on the CPU:
the numpy oracle against the committed golden fixture and against oracle/_ref (or its stored results, tests/golden/ref),
and the host-side tables /
parameter rules of libaudioflux_b200 against both.  (The CUDA parity tests are in test_gpu_parity.py.)"""
import ctypes as C

import numpy as np
import pytest

import audioflux_b200 as af
from conftest import RefSample, noise, ref_absmax, ref_pair, rel_max, tones
from oracle import af_oracle as O

S, ST, N, D = (af.SpectralFilterBankScaleType, af.SpectralFilterBankStyleType,
               af.SpectralFilterBankNormalType, af.SpectralDataType)
E, CN = af.CepstralEnergyType, af.ChromaDataNormalType
TOL = 1e-4


# ---------------- oracle vs golden (always runs) ----------------
@pytest.mark.parametrize("name,et,order", [("rep", 0, 9), ("app", 1, 5), ("ign", 2, 3)])
def test_oracle_xxcc_standard_golden(golden, name, et, order):
    g, c1 = golden("next_rows.npz"), golden("c1_mel_mfcc.npz")
    coe, d1, d2 = O.xxcc_standard(c1["mel"][:24], g["energy"], 13, order, et)
    for got, key in ((coe, "coe"), (d1, "d1"), (d2, "d2")):
        want = g[f"std_{name}_{key}"]
        assert got.shape == want.shape
        assert rel_max(got, want) < TOL


def test_oracle_chroma_cqcc_golden(golden):
    g, c = golden("next_rows.npz"), golden("cqt_84.npz")
    assert rel_max(O.cqt_chroma(c["re"], c["im"], 12, O.DATA_POWER, O.CHROMA_NORM_MAX), g["chroma_max"]) < TOL
    assert rel_max(O.cqt_chroma(c["re"], c["im"], 12, O.DATA_MAG, O.CHROMA_NORM_P2), g["chroma_p2"]) < TOL
    p = (c["re"].astype(np.float64) ** 2 + c["im"].astype(np.float64) ** 2).astype(np.float32)
    assert rel_max(O.xxcc(p, 20), g["cqcc"]) < TOL


def _phase_mask(re_like_spec):
    """Bins whose phase is well conditioned: the reference's phase is atan2f(im, max(re, 1e-16)), so wherever
    re < 0 it degenerates to sign(im)*pi/2 and a bin with |im| at rounding-noise level flips sign freely."""
    return re_like_spec > 1e-7 * re_like_spec.max()


def test_oracle_spectrogram_golden(golden):
    g = golden("next_rows.npz")
    x = g["xsp"]
    lin, ph = O.spectrogram(x, sr=48000, low=100., high=8000., radix2_exp=10, hop=256, want_phase=True)
    assert lin.shape == g["lin"].shape == (20, 170)
    assert rel_max(lin, g["lin"]) < TOL
    m = _phase_mask(g["lin"])
    assert m.mean() > 0.8
    assert np.abs(ph - g["lin_phase"])[m].max() < 5e-3
    p = O.spectrogram_params(0, 48000, 100., 8000., 12, 10, O.SCALE_LINEAR)
    fre, bins = O.spectrogram_linear_bands(48000, 10, p["low_idx"], p["num"])
    assert np.array_equal(bins, g["lin_bin"]) and np.array_equal(fre, g["lin_fre"])
    mel = O.spectrogram(x, 64, 48000, radix2_exp=10, hop=256, data_type=O.DATA_MAG, scale=O.SCALE_MEL, norm_value=0.5)
    assert rel_max(mel, g["mel_mag"]) < TOL
    assert rel_max(O.xxcc(g["mel_mag"], 13), g["mel_cc"]) < TOL


# ---------------- host tables of the product (no GPU needed) ----------------
@pytest.mark.parametrize("num,bpo,fmin", [(12, 12, 32.703196), (12, 24, 32.703196), (12, 36, 55.0), (6, 12, 32.703196),
                                           (24, 24, 65.4), (12, 12, 440.0), (12, 12, 46.25), (12, 12, 61.74)])
def test_chroma_bank(product_lib, num, bpo, fmin):
    length = 7 * bpo
    got = np.zeros((num, length), np.float32)
    assert product_lib.afb200_chromaCqtFilterBank(num, length, bpo, C.c_float(fmin), got.ctypes.data) == 0
    assert np.array_equal(got, O.chroma_cqt_bank(num, length, bpo, fmin))
    assert got.sum() == length                                  # every CQT bin lands in exactly one class


def test_chroma_bank_vs_reference(reference):
    for num, bpo, fmin in [(12, 12, 32.703196), (12, 24, 32.703196), (12, 36, 55.0), (24, 24, 65.4), (12, 12, 440.0),
                           (12, 12, 46.25), (12, 12, 61.74), (4, 12, 100.0)]:
        length = 7 * bpo

        def ref(lib):
            want = np.zeros((num, length), np.float32)
            lib.chroma_cqtFilterBank(num, length, bpo, C.byref(C.c_float(fmin)), want.ctypes.data)
            assert np.array_equal(want, want.astype(np.int8))          # 0 / 1 weights: stored whole as int8
            return want.astype(np.int8)
        want = reference(f"bank{num}-{bpo}-{fmin}", ref)
        assert np.array_equal(want, O.chroma_cqt_bank(num, length, bpo, fmin)), (num, bpo, fmin)


def test_chroma_bank_rejects_bad_division(product_lib):
    got = np.zeros((5, 84), np.float32)
    assert product_lib.afb200_chromaCqtFilterBank(5, 84, 12, C.c_float(32.7), got.ctypes.data) != 0


SPEC_CASES = [
    dict(num=0, samplate=48000, low_fre=100., high_fre=8000., radix2_exp=10, slide_length=256),
    dict(num=0, samplate=32000, radix2_exp=11),
    dict(num=0, samplate=16000, low_fre=7000., high_fre=300., radix2_exp=9),            # high < low -> full band
    dict(num=128, samplate=48000, radix2_exp=11, slide_length=512, filter_bank_type=S.MEL),
    dict(num=64, samplate=32000, radix2_exp=10, filter_bank_type=S.BARK, style_type=ST.ETSI, normal_type=N.AREA),
    dict(num=40, samplate=16000, radix2_exp=10, filter_bank_type=S.ERB, low_fre=50., high_fre=7000.),
    dict(num=84, samplate=32000, radix2_exp=12, filter_bank_type=S.OCTAVE),
    dict(num=48, samplate=32000, radix2_exp=12, filter_bank_type=S.OCTAVE, bin_per_octave=24, low_fre=65.4),
    dict(num=64, samplate=48000, radix2_exp=11, filter_bank_type=S.LINSPACE, low_fre=1000., high_fre=20000.),
    dict(num=64, samplate=48000, radix2_exp=11, filter_bank_type=S.LOG, low_fre=32.703196, high_fre=19000.),
]


@pytest.mark.parametrize("kw", SPEC_CASES)
def test_spectrogram_new_tables_vs_oracle(product_lib, kw):
    s = af.Spectrogram(**kw)
    scale = af.enum_value(kw.get("filter_bank_type", S.LINEAR))
    p = O.spectrogram_params(kw["num"], kw["samplate"], kw.get("low_fre"), kw.get("high_fre"),
                             kw.get("bin_per_octave", 12), kw["radix2_exp"], scale)
    assert s.num == p["num"] == s.get_bin_band_length()
    n = 1 << kw["radix2_exp"]
    hop = kw.get("slide_length", n // 4)
    assert s.cal_time_length(10 * n) == (10 * n - n) // hop + 1
    if scale == 0:
        fre, bins = O.spectrogram_linear_bands(kw["samplate"], kw["radix2_exp"], p["low_idx"], p["num"])
        assert np.array_equal(s.get_bin_band_arr(), bins) and np.array_equal(s.get_fre_band_arr(), fre)
    else:
        _, fre, bins = O.auditory_filterbank(p["num"], n, kw["samplate"], scale,
                                             af.enum_value(kw.get("style_type", ST.SLANEY)),
                                             af.enum_value(kw.get("normal_type", N.NONE)), float(p["low"]), float(p["high"]),
                                             p["bpo"])
        assert np.array_equal(s.get_bin_band_arr(), bins)
        np.testing.assert_allclose(s.get_fre_band_arr(), fre, rtol=2e-6, atol=1e-3)


@pytest.mark.parametrize("kw", SPEC_CASES)
def test_spectrogram_new_tables_vs_reference(product_lib, reference, kw):
    def ref(lib):
        b = af.Spectrogram(_lib=lib, **kw)
        return np.array(b.num), b.get_bin_band_arr(), b.get_fre_band_arr(), np.array(b.cal_time_length(50000))
    num, bins, fre, frames = reference("tables", ref)
    a = af.Spectrogram(**kw)
    assert a.num == num
    assert np.array_equal(a.get_bin_band_arr(), bins)
    np.testing.assert_allclose(*ref_pair(a.get_fre_band_arr(), fre), rtol=2e-6, atol=1e-3)
    assert a.cal_time_length(50000) == frames


def test_spectrogram_new_status_codes(product_lib):
    from audioflux_b200.capi import opt_int
    obj = C.c_void_p()
    none = [None] * 12
    a = list(none); a[4] = opt_int(31)
    assert product_lib.spectrogramObj_new(C.byref(obj), 128, *a) == -100                 # radix2Exp
    a = list(none); a[9] = opt_int(2)
    assert product_lib.spectrogramObj_new(C.byref(obj), 1, *a) == -1                     # num < 2 (mel)
    assert product_lib.spectrogramObj_new(C.byref(obj), 5000, *a) == -1                  # num > n/2+1
    a = list(none); a[9] = opt_int(7)
    assert product_lib.spectrogramObj_new(C.byref(obj), 12, *a) == -2                    # Chroma family: loud
    assert b"not supported" in product_lib.afb200_lastError()
    a = list(none); a[7] = opt_int(1)
    assert product_lib.spectrogramObj_new(C.byref(obj), 12, *a) == 0                     # isContinue: streaming front door
    assert product_lib.spectrogramObj_calTimeLength(obj, 4096) == 1 and product_lib.spectrogramObj_calTimeLength(obj, 100) == 0
    product_lib.spectrogramObj_free(obj)
    a = list(none); a[9] = opt_int(5)
    assert product_lib.spectrogramObj_new(C.byref(obj), 240, *a) == -1                   # Octave overflow
    for ctor, args in (("spectrogramObj_newMel", (128, 48000, 11)), ("spectrogramObj_newBark", (64, 32000, 10)),
                       ("spectrogramObj_newErb", (40, 16000, 10))):
        assert getattr(product_lib, ctor)(C.byref(obj), *args, None) == 0
        assert product_lib.spectrogramObj_getBandNum(obj) == args[0]
        product_lib.spectrogramObj_free(obj)
    assert product_lib.spectrogramObj_newChroma(C.byref(obj), 32000, 12, None) == -2 and not obj.value
    assert product_lib.spectrogramObj_newDeep(C.byref(obj), 84, 32000, 12, None) == -2
    assert product_lib.spectrogramObj_newDeepChroma(C.byref(obj), 32000, 12, None) == -2
    assert b"Chroma / Deep" in product_lib.afb200_lastError()
    assert product_lib.spectrogramObj_newLinear(C.byref(obj), 32000, 11, None) == 0
    assert product_lib.spectrogramObj_getBandNum(obj) == 1025
    product_lib.spectrogramObj_free(obj)


# ---------------- oracle vs the reference itself ----------------
@pytest.mark.parametrize("et,order,cc,rect", [(0, 9, 13, 0), (1, 9, 13, 0), (2, 9, 20, 0), (0, 5, 40, 1), (1, 3, 5, 0),
                                               (0, 4, 13, 0)])
def test_xxcc_standard_vs_reference(reference, et, order, cc, rect):
    rng = np.random.default_rng(7)
    m = (rng.random((37, 64)) ** 4 * 10).astype(np.float32)
    m[3, :5] = 0                                              # exercises the 1e-8 floor
    e = (rng.random(37) * 3).astype(np.float32)
    e[2] = 0
    want = reference("planes", lambda lib: af.XXCC(64, _lib=lib).xxcc_standard_planes(m, e, cc, order, et, rect))
    got = O.xxcc_standard(m, e, cc, order, et, rect)
    for g, w in zip(got, want):
        assert g.shape == w.shape and rel_max(g, w) < TOL


@pytest.mark.parametrize("cn,dt,norm,bpo,num", [(12, 0, 1, 12, 84), (12, 1, 3, 12, 84), (12, 0, 0, 12, 84), (12, 0, 2, 12, 84),
                                                 (12, 1, 4, 12, 84), (12, 0, 1, 24, 96), (24, 0, 1, 24, 96), (6, 1, 3, 12, 48)])
def test_chroma_cqcc_vs_reference(reference, cn, dt, norm, bpo, num):
    x = tones(11, 9000, 32000)
    # the same CQT planes (the oracle's, regenerated wherever the test runs) go into the reference and the oracle
    re, im = (np.ascontiguousarray(a, np.float32) for a in O.cqt(x, num, 32000, bpo=bpo))
    p = (re * re + im * im).astype(np.float32)

    def ref(lib):
        c = af.CQT(num, 32000, bin_per_octave=bpo, _lib=lib)
        assert c.cqt_planes(x)[0].shape == re.shape                    # also sets the object's timeLength
        return c.chroma_planes(re, im, cn, dt, norm), c.cqcc_planes(p, 13)
    want, want_cc = reference("chroma,cqcc", ref)
    got = O.cqt_chroma(re, im, cn, dt, norm, bpo)
    assert rel_max(got, want) < TOL
    assert rel_max(O.xxcc(p, 13), want_cc) < TOL


@pytest.mark.parametrize("kw", SPEC_CASES[:8])
def test_spectrogram_vs_reference(reference, kw):
    x = tones(12, 30000, kw["samplate"])
    for dt, nv in ((D.POWER, 1.0), (D.MAG, 1.0), (D.POWER, 0.7), (D.MAG, 1.5)):
        scale = af.enum_value(kw.get("filter_bank_type", S.LINEAR))

        def ref(lib):
            s = af.Spectrogram(_lib=lib, data_type=dt, **kw)
            if nv != 1.0:
                s.set_data_norm_value(nv)
            return s.spectrogram_planes(x, scale == 0)
        want = reference(f"spec{af.enum_value(dt)}-{nv}", ref)
        got = O.spectrogram(x, kw["num"], kw["samplate"], kw.get("low_fre"), kw.get("high_fre"),
                            kw.get("bin_per_octave", 12), kw["radix2_exp"], hop=kw.get("slide_length"),
                            data_type=af.enum_value(dt), scale=scale,
                            style=af.enum_value(kw.get("style_type", ST.SLANEY)),
                            norm=af.enum_value(kw.get("normal_type", N.NONE)), norm_value=nv, want_phase=scale == 0)
        if scale == 0:
            assert rel_max(got[0], want[0]) < TOL
            m = ref_pair(got[0], want[0])[1] > 1e-7 * ref_absmax(want[0])     # _phase_mask on the stored elements
            g1, w1 = ref_pair(got[1], want[1])
            assert np.abs(g1 - w1)[m].max() < 5e-3
        else:
            assert rel_max(got, want) < TOL


# ---------------- STFT padding modes (SURVEY 8f-4): oracle vs the reference ----------------
PAD_CASES = [(pos, mode, v1, v2, L, n, hop) for pos in (0, 1, 2) for mode in (0, 1, 2)
             for (v1, v2, L, n, hop) in ((0.0, 0.0, 3000, 256, 64), (0.37, -1.6, 2500, 512, 100), (2.9, 0.5, 700, 1024, 256))]


@pytest.mark.parametrize("pos,mode,v1,v2,L,n,hop", PAD_CASES + [(0, 1, 0, 0, 1, 64, 16), (0, 2, 0, 0, 40, 256, 64)])
def test_stft_padding_modes_vs_reference(reference, pos, mode, v1, v2, L, n, hop):
    x = noise(61, L)
    r = int(np.log2(n))

    def ref(lib):
        s = af.STFT(r, af.WindowType.HANN, hop, _lib=lib)
        s.enable_padding(True)
        s.set_padding(pos, mode, v1, v2)
        return s.stft_planes(x)
    re, im = reference("stft", ref)
    re2, im2 = O.stft(x, n, hop, O.fft_window(O.W_HANN, n), True, pos, mode, v1, v2)
    assert re.shape == re2.shape
    scale = max(ref_absmax(re), ref_absmax(im), 1e-30)
    (re2, re), (im2, im) = ref_pair(re2, re), ref_pair(im2, im)
    assert np.abs(re - re2).max() <= TOL * scale and np.abs(im - im2).max() <= TOL * scale


# ---------------- cwtObj_cwtDet (SURVEY 8f-3): oracle vs golden and vs the reference ----------------
def test_oracle_cwt_det_golden(golden):
    g = golden("next_rows.npz")
    re, im = O.cwt(g["xdet"], 12, 10, 48000, O.WAVE_MORLET, O.SCALE_OCTAVE, low=32.703196, det=True)
    scale = max(np.abs(g["det_re"]).max(), np.abs(g["det_im"]).max())
    assert np.abs(re - g["det_re"]).max() <= TOL * scale and np.abs(im - g["det_im"]).max() <= TOL * scale


@pytest.mark.parametrize("wav,pad,r", [(1, False, 12), (0, False, 12), (3, True, 11), (2, False, 10), (4, False, 12), (5, True, 10)])
def test_cwt_det_vs_reference(reference, wav, pad, r):
    x = noise(71, 1 << r)

    def ref(lib):
        w = af.CWT(36, r, 48000, wavelet_type=wav, is_padding=pad, _lib=lib)
        w.enable_det(True)
        w.cwt_planes(x)
        re, im = w.cwt_det_planes(None)                          # reuses the spectrum of the cwt call
        re1, im1 = w.cwt_det_planes(x)
        return re, im, np.array(np.array_equal(re, re1) and np.array_equal(im, im1))
    re, im, same = reference("det", ref)
    assert same
    r2, i2 = O.cwt(x, 36, r, 48000, wav, O.SCALE_OCTAVE, low=32.703196, is_pad=pad, det=True)
    scale = max(ref_absmax(re), ref_absmax(im))
    (r2, re), (i2, im) = ref_pair(r2, re), ref_pair(i2, im)
    assert np.abs(re - r2).max() <= TOL * scale and np.abs(im - i2).max() <= TOL * scale


# ---------------- stftObj_istft: oracle vs the reference ----------------
def istft_conditioned(n, hop, T, window, method):
    """Samples whose window-sum normaliser is not tiny: elsewhere the division amplifies float32 rounding of the
    frames (the reference divides by sums down to 1e-6), so only a loose bound makes sense there."""
    w = np.asarray(window, dtype=np.float64) ** (2 if method == 0 else 1)
    norm = np.zeros((T - 1) * hop + n)
    for t in range(T):
        norm[t * hop:t * hop + n] += w
    return norm > 1e-2


ISTFT_CASES = [(9, 128, 1, 0), (9, 128, 1, 1), (10, 256, 2, 0), (8, 64, 0, 0), (8, 256, 1, 1), (11, 512, 4, 0), (6, 100, 1, 0)]


@pytest.mark.parametrize("r,hop,wt,method", ISTFT_CASES)
def test_istft_vs_reference(reference, r, hop, wt, method):
    n = 1 << r
    x = noise(81, 20 * hop + n)
    # the same STFT planes (the oracle's, regenerated wherever the test runs) go into the reference and the oracle
    re, im = (np.ascontiguousarray(a, np.float32) for a in O.stft(x, n, hop, O.fft_window(wt, n)))

    def ref(lib):
        s = af.STFT(r, wt, hop, _lib=lib)
        assert s.stft_planes(x)[0].shape == re.shape
        z = (re + 1j * im).T[:n // 2 + 1]                # reference-layout front door (complex [n/2+1, T] in)
        return s.istft_planes(re, im, method), s.istft(z, method)
    got, got_z = reference("istft", ref)
    want = O.istft(re, im, n, hop, O.fft_window(wt, n), method)
    assert got.shape == want.shape
    ok = ref_pair(istft_conditioned(n, hop, re.shape[0], O.fft_window(wt, n), method), got)[0]
    scale = np.abs(want).max()
    w, g = ref_pair(want, got)
    assert np.abs(g - w)[ok].max() <= TOL * scale and np.abs(g - w).max() <= 1e-2 * scale
    if hop <= n // 2 and wt in (1, 2):                   # enough overlap: the round trip reproduces the interior
        i = got.index if isinstance(got, RefSample) else np.arange(got.shape[0])
        inner = (i >= n) & (i < got.shape[0] - n)
        assert np.abs(g[inner] - x[i[inner]]).max() < 1e-4
    w, g = ref_pair(want, got_z)
    assert np.abs(g - w)[ok].max() <= TOL * scale


# ---------------- PWT (SURVEY 8f-3): tables and oracle vs the reference ----------------
PWT_CASES = [dict(num=84, samplate=32000, is_padding=False), dict(num=84, samplate=32000, is_padding=True),
             dict(num=40, samplate=16000, scale_type=2, is_padding=False, normal_type=1),
             dict(num=64, samplate=48000, scale_type=3, style_type=1, is_padding=True),
             dict(num=48, samplate=32000, scale_type=5, bin_per_octave=24, low_fre=65.4, is_padding=False),
             dict(num=32, samplate=22050, scale_type=4, style_type=5, normal_type=2, is_padding=False)]


def _pwt_oracle(x, kw, r, det=False):
    return O.pwt(x, kw["num"], r, kw["samplate"], low=kw.get("low_fre"), bpo=kw.get("bin_per_octave", 12),
                 scale=kw.get("scale_type", 5), style=kw.get("style_type", 0), norm=kw.get("normal_type", 0),
                 is_pad=kw["is_padding"], det=det)


@pytest.mark.parametrize("kw", PWT_CASES[:5])
def test_pwt_vs_reference(reference, product_lib, kw):
    x = noise(91, 4096)

    def ref(lib):
        w = af.PWT(radix2_exp=12, _lib=lib, **kw)
        re, im = w.pwt_planes(x)
        w.enable_det(True)
        return (w.get_bin_band_arr(), w.get_fre_band_arr(), re, im) + tuple(w.pwt_det_planes(None))
    bins_r, fre_r, re, im, dr, di = reference("pwt", ref)
    p = af.PWT(radix2_exp=12, **kw)
    assert np.array_equal(bins_r, p.get_bin_band_arr())                           # product tables == reference tables
    np.testing.assert_allclose(*ref_pair(p.get_fre_band_arr(), fre_r), rtol=2e-6, atol=1e-3)
    r2, i2, fre, bins = _pwt_oracle(x, kw, 12)
    scale = max(ref_absmax(re), ref_absmax(im))
    (r2, re), (i2, im) = ref_pair(r2, re), ref_pair(i2, im)
    assert np.abs(re - r2).max() <= TOL * scale and np.abs(im - i2).max() <= TOL * scale
    assert np.array_equal(bins, bins_r)
    d2, e2, _, _ = _pwt_oracle(x, kw, 12, det=True)
    sd = max(ref_absmax(dr), ref_absmax(di))
    (d2, dr), (e2, di) = ref_pair(d2, dr), ref_pair(e2, di)
    assert np.abs(dr - d2).max() <= TOL * sd and np.abs(di - e2).max() <= TOL * sd


def test_pwt_new_status_codes(product_lib):
    obj = C.c_void_p()
    none = [None] * 8
    assert product_lib.pwtObj_new(C.byref(obj), 84, 31, *none) == -100
    assert product_lib.pwtObj_new(C.byref(obj), 1, 12, *none) == -1
    assert product_lib.pwtObj_new(C.byref(obj), 400, 12, *none) == -1                   # octave overflow
    from audioflux_b200.capi import opt_int
    a = list(none); a[4] = opt_int(9)
    assert product_lib.pwtObj_new(C.byref(obj), 84, 12, *a) == 1                        # scale > Log
    a = list(none); a[7] = opt_int(1)
    assert product_lib.pwtObj_new(C.byref(obj), 84, 19, *a) == -2                       # padding -> non power of two
    assert product_lib.pwtObj_new(C.byref(obj), 84, 12, *none) == 0
    product_lib.pwtObj_free(obj)


# ---- synchrosqueezing: the numpy restatement (oracle wsst / synsq) pinned to the reference build -------------------------
def _sq_signal(n, sr, seed):
    t = np.arange(n) / sr
    rng = np.random.default_rng(seed)
    return (0.5 * np.sin(2 * np.pi * (300 + 2000 * t) * t) + 0.2 * np.sin(2 * np.pi * 2500 * t) + 0.01 * rng.standard_normal(n)).astype(np.float32)


def _sq_agree(a, b):
    cols = (np.abs(a - b) > 1e-5 * np.abs(b).max()).any(axis=0)
    return 1.0 - cols.mean(), float(np.linalg.norm(a - b) / np.linalg.norm(b))


@pytest.mark.parametrize("is_pad,scale,wavelet", [(False, O.SCALE_OCTAVE, O.WAVE_MORLET), (True, O.SCALE_OCTAVE, O.WAVE_MORLET),
                                                   (False, O.SCALE_LINEAR, O.WAVE_MORSE), (False, O.SCALE_MEL, O.WAVE_BUMP)])
def test_oracle_wsst_matches_the_reference_build(ref_lib, is_pad, scale, wavelet):
    """row indices are integer outcomes of float32 log2f / divide: a few cells per thousand land one row apart between numpy
    and glibc; the bar is statistical (>= 99 % of time columns identical, Frobenius error <= 5e-3)"""
    import audioflux_b200 as af
    sr, num, radix = 32000, 84, 12
    x = _sq_signal(1 << radix, sr, 1)
    w = af.WSST(num, radix, sr, wavelet_type=af.WaveletContinueType(wavelet), scale_type=af.SpectralFilterBankScaleType(scale),
                is_padding=is_pad, _lib=ref_lib)
    re, im, cr, ci = w.wsst_planes(x)
    o_re, o_im, w_re, w_im = O.wsst(x, num, radix, sr, wavelet=wavelet, scale=scale, is_pad=is_pad, low=w.low_fre, high=w.high_fre)
    assert rel_max(w_re, cr) < 1e-4 and rel_max(w_im, ci) < 1e-4
    for got, want in ((o_re, re), (o_im, im)):
        same, fro = _sq_agree(got, want)
        assert same >= 0.99 and fro <= 5e-3, (same, fro)


@pytest.mark.parametrize("scale", [O.SCALE_OCTAVE, O.SCALE_LINEAR, O.SCALE_BARK])
def test_oracle_synsq_matches_the_reference_build(ref_lib, scale):
    import audioflux_b200 as af
    sr, num, radix = 32000, 84, 12
    x = _sq_signal(1 << radix, sr, 2)
    w_re, w_im = O.cwt(x, num, radix, sr, wavelet=O.WAVE_MORLET, scale=scale, is_pad=False)
    _, fre = O.cwt_filterbank(num, 1 << radix, sr, O.WAVE_MORLET, scale, None, None, 12, None, None, 0)
    fre = np.ascontiguousarray(fre, np.float32)
    want = af.Synsq(num, radix, sr, _lib=ref_lib).synsq_planes(fre, af.SpectralFilterBankScaleType(scale), w_re, w_im)
    got = O.synsq(fre, w_re, w_im, sr, scale)
    for g, w in zip(got, want):
        same, fro = _sq_agree(g, w)
        assert same >= 0.99 and fro <= 1e-2, (same, fro)


# ---- streaming STFT: the oracle's model of __stftObj_dealData pinned to the reference build ----
@pytest.mark.parametrize("r,hop,chunks", [(9, 128, (1000, 37, 500, 3000, 129, 512)), (10, 1024, (700, 700, 2048, 5000, 1)),
                                          (8, 300, (100, 100, 100, 1000, 40, 2000)), (8, 64, (255, 1, 64, 63, 1, 800))])
def test_oracle_stft_streaming_matches_the_reference_build(ref_lib, r, hop, chunks):
    import audioflux_b200 as af
    n = 1 << r
    x = noise(78, sum(chunks))
    q = af.STFT(r, af.WindowType.HANN, hop, is_continue=True, _lib=ref_lib)
    model = O.StftStream(n, hop, O.fft_window(O.W_HANN, n))
    pos = 0
    for c in chunks:
        piece = x[pos:pos + c]
        pos += c
        rr, ri = q.stft_planes(piece)
        wr, wi = model.push(piece)
        assert rr.shape == wr.shape, (c, rr.shape, wr.shape)
        if rr.shape[0]:
            assert rel_max(wr, rr) < 1e-5 and rel_max(wi, ri) < 1e-5


# ---- streaming CQT: the oracle's model of _cqtObj_dealData / right-padded frames pinned to the reference build ----
@pytest.mark.parametrize("chunks", [(3000, 2500, 5000, 1400), (4000, 4000, 2000), (3000, 3000, 3000)])
def test_oracle_cqt_streaming_matches_the_reference_build(ref_lib, chunks):
    import audioflux_b200 as af
    sr = 32000
    x = tones(3, sum(chunks), sr)
    q = af.CQT(84, sr, is_continue=True, _lib=ref_lib)
    model = O.CqtStream(84, sr, norm=O.NORM_AREA)
    pos = 0
    for n in chunks:
        piece = x[pos:pos + n]
        pos += n
        rr, ri = q.cqt_planes(piece)
        wr, wi = model.push(piece)
        assert rr.shape == wr.shape and rr.shape[0] > 0
        assert rel_max(wr, rr) < 1e-5 and rel_max(wi, ri) < 1e-5


@pytest.mark.parametrize("num,sr,beta,norm,bpo", [(84, 32000, 5.0, 0, 12), (48, 44100, 2.0, 1, 12), (72, 22050, 10.0, 2, 12),
                                                   (48, 16000, 3.0, 0, 24)])
def test_oracle_vqt_vs_reference_build(reference, num, sr, beta, norm, bpo):
    """VQT (beta != 0): the oracle's per-octave kernel rows against the reference build"""
    import audioflux_b200 as af
    x = (0.1 * np.random.default_rng(0).standard_normal(30000)).astype(np.float32)

    def ref(lib):
        z = af.CQT(num, sr, bin_per_octave=bpo, beta=beta, normal_type=af.SpectralFilterBankNormalType(norm), _lib=lib).cqt(x)
        return np.ascontiguousarray(z.real), np.ascontiguousarray(z.imag)
    zr, zi = reference("vqt", ref)
    re, im = O.cqt(x, num, sr, bpo=bpo, beta=beta, norm=norm)
    assert rel_max(re.T, zr) < 1e-5 and rel_max(im.T, zi) < 1e-5
