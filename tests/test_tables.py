"""Setup-time tables of libaudioflux_b200 (windows, auditory banks, CQT kernels, wavelet banks,
decimator taps) against the numpy oracle, and against oracle/_ref where present.  No GPU needed:
the builders are host C."""
import ctypes as C

import numpy as np
import pytest

import audioflux_b200 as af
from conftest import ref_pair, ref_window
from oracle import af_oracle as O

S, ST, N, D = (af.SpectralFilterBankScaleType, af.SpectralFilterBankStyleType,
               af.SpectralFilterBankNormalType, af.SpectralDataType)


@pytest.mark.parametrize("wt", range(14))
def test_windows(product_lib, wt):
    for n in (2, 16, 512, 2048):
        w = np.zeros(n, np.float32)
        assert product_lib.afb200_window(wt, n, w.ctypes.data) == 0
        assert np.abs(w - O.fft_window(wt, n)).max() < 1e-6


def _bank(lib, num, n, sr, scale, style, norm, low, high, bpo):
    bank = np.zeros((num, n // 2 + 1), np.float32)
    fb = np.zeros(num, np.float32)
    bb = np.zeros(num, np.int32)
    assert lib.afb200_auditoryFilterBank(num, n, sr, scale, style, norm, low, high, bpo, bank.ctypes.data,
                                         fb.ctypes.data, bb.ctypes.data) == 0
    return bank, fb, bb


@pytest.mark.parametrize("scale", range(1, 7))
@pytest.mark.parametrize("style", (0, 1, 3, 4, 5, 6, 7, 8, 9, 10))
def test_filter_banks(product_lib, scale, style):
    for norm in (0, 1, 2):
        for num, n, sr in ((128, 2048, 48000), (40, 1024, 16000)):
            low = 32.703196 if scale in (5, 6) else None
            high = None
            if scale == 1:
                low, high = 1000.0, sr / 2 - 1000.0
            if scale == 6:
                low, high = 32.703196, sr / 2 * 0.8
            lo, hi, _, _ = O.bft_revise_range(num, n, sr, low, high, scale, 12)
            if scale == 5 and float(hi) > sr / 2:
                continue
            b1, f1, i1 = _bank(product_lib, num, n, sr, scale, style, norm, float(lo), float(hi), 12)
            b2, f2, i2 = O.auditory_filterbank(num, n, sr, scale, style, norm, float(lo), float(hi), 12)
            assert np.array_equal(i1, i2)                       # integer outcomes: exact
            assert np.abs(b1 - b2).max() <= 5e-5 * max(1.0, np.abs(b2).max())
            np.testing.assert_allclose(f1, f2, rtol=2e-6, atol=1e-3)


def test_bank_out_of_range_edges_are_clipped(product_lib):
    # Linspace over the full band revises the edges outside [0, sr/2]; the reference writes out of
    # bounds there, this library must clip (and not crash)
    bank, _, _ = _bank(product_lib, 64, 1024, 16000, 1, 0, 0, 0.0, 8000.0, 12)
    assert np.isfinite(bank).all()


def test_bft_object_tables(product_lib):
    b = af.BFT(128, 11, 48000, slide_length=512, scale_type=S.MEL, data_type=D.POWER)
    assert b.cal_time_length(240000) == 465 and b.cal_time_length(48000) == 90 and b.cal_time_length(2047) == 0
    bank, fre, bins = O.auditory_filterbank(128, 2048, 48000, O.SCALE_MEL, O.STYLE_SLANEY, O.NORM_NONE, 0.0, 24000.0)
    assert np.array_equal(b.get_bin_band_arr(), bins)
    np.testing.assert_allclose(b.get_fre_band_arr(), fre, rtol=2e-6)
    got = b.get_filter_bank_arr()
    assert np.abs(got - bank).max() < 5e-6
    assert int((got != 0).sum()) == 2019                         # SURVEY.md section 3.4


def test_bft_new_status_codes(product_lib):
    import ctypes
    from audioflux_b200.capi import opt_int
    obj = ctypes.c_void_p()
    args = [None] * 12
    assert product_lib.bftObj_new(ctypes.byref(obj), 128, 31, *args) == -100        # radix2Exp
    assert product_lib.bftObj_new(ctypes.byref(obj), 1, 11, *args) == -1            # num < 2
    assert product_lib.bftObj_new(ctypes.byref(obj), 4000, 11, *args) == -1         # num > n/2+1
    a2 = list(args); a2[6] = opt_int(9)
    assert product_lib.bftObj_new(ctypes.byref(obj), 64, 11, *a2) == 1              # scale > Log
    a3 = list(args); a3[10] = opt_int(1)
    assert product_lib.bftObj_new(ctypes.byref(obj), 64, 11, *a3) == 0              # isReassign: supported (bank over the reassigned spectrum)
    product_lib.bftObj_free(obj)
    a4 = list(args); a4[11] = opt_int(1)
    assert product_lib.bftObj_new(ctypes.byref(obj), 64, 11, *a4) == 0              # isTemporal: supported (energy / rms / zcr)
    product_lib.bftObj_free(obj)
    assert product_lib.stftObj_new(ctypes.byref(obj), 0, None, None, None) == -100
    assert product_lib.xxccObj_new(ctypes.byref(obj), 1) == -1
    assert product_lib.cqtObj_newWith(ctypes.byref(obj), 84, None, None, opt_int(10), *([None] * 8)) == -1
    assert product_lib.cqtObj_newWith(ctypes.byref(obj), 80, *([None] * 11)) == -1


def test_cqt_tables(product_lib):
    c = af.CQT(84, 48000)
    assert c.fft_length == 512 and c.slide_length == 128 and c.cal_time_length(240000) == 1876
    kr, ki = c.get_kernel_bank()
    ob = O.cqt_kernel_bank(84, 48000, norm=O.NORM_AREA)
    assert int((kr != 0).sum()) == 104
    assert np.abs(kr - ob["kr"]).max() < 1e-6 and np.abs(ki - ob["ki"]).max() < 1e-6
    np.testing.assert_allclose(c.get_fre_band_arr(), ob["fre"], rtol=1e-7)
    left = np.zeros(32, np.float32)
    right = np.zeros(31, np.float32)
    product_lib.afb200_decimatorTaps(left.ctypes.data, right.ctypes.data)
    l2, r2 = O.decimator_taps()
    assert np.abs(left - l2).max() < 1e-7 and np.abs(right - r2).max() < 1e-7


@pytest.mark.parametrize("num,sr,beta,norm,bpo", [(84, 32000, 5.0, 0, 12), (48, 44100, 2.0, 1, 12), (72, 22050, 10.0, 2, 12),
                                                   (48, 16000, 3.0, 0, 24)])
def test_vqt_tables(product_lib, num, sr, beta, norm, bpo):
    """beta != 0 (VQT, VERDICT r1 missing #5): one kernel row per bin -- every octave from its own float frequencies and the
    integer-halved sample rate (44100 -> ... -> 5512), shortened by beta (cqt_algorithm.c:186-193, 1208-1246)"""
    c = af.CQT(num, sr, bin_per_octave=bpo, beta=beta, normal_type=af.SpectralFilterBankNormalType(norm))
    ob = O.cqt_kernel_bank(num, sr, bpo=bpo, beta=beta, norm=norm)
    assert c.fft_length == ob["fft_length"] and ob["kr"].shape[0] == num
    kr, ki = c.get_kernel_bank()
    scale = max(np.abs(ob["kr"]).max(), np.abs(ob["ki"]).max())
    assert np.abs(kr - ob["kr"]).max() < 2e-5 * scale and np.abs(ki - ob["ki"]).max() < 2e-5 * scale
    assert np.array_equal(kr != 0, ob["kr"] != 0) or np.abs((kr != 0).sum() - (ob["kr"] != 0).sum()) <= 2    # threshold ties


@pytest.mark.parametrize("wav", range(8))
def test_cwt_tables(product_lib, wav):
    w = af.CWT(84, 12, 48000, wavelet_type=af.WaveletContinueType(wav), is_padding=False)
    ob, fre = O.cwt_filterbank(84, 4096, 48000, wav)
    fb = w.get_filter_bank_arr()
    assert np.abs(fb - ob).max() <= 1e-5 * np.abs(ob).max()
    np.testing.assert_allclose(w.get_fre_band_arr(), fre, rtol=1e-6)
    assert abs(w.get_fre_band_arr()[0] - 32.703197) < 1e-4 and abs(w.get_fre_band_arr()[83] - 3951.0667) < 1e-2


def test_tables_against_reference_build(product_lib, reference):
    for wt in range(14):
        w = reference(f"window{wt}", lambda lib: ref_window(lib, wt, 2048))
        w2 = np.zeros(2048, np.float32)
        product_lib.afb200_window(wt, 2048, w2.ctypes.data)
        w2, w = ref_pair(w2, w)
        assert np.abs(w - w2).max() < 1e-6
    for scale, style, norm in ((2, 0, 0), (2, 0, 1), (3, 1, 2), (4, 0, 0), (5, 0, 0)):
        b = af.BFT(96, 11, 44100, scale_type=S(scale), style_type=ST(style), normal_type=N(norm))

        def bands(lib):
            r = af.BFT(96, 11, 44100, scale_type=S(scale), style_type=ST(style), normal_type=N(norm), _lib=lib)
            return r.get_bin_band_arr(), r.get_fre_band_arr()
        bin_band, fre_band = reference(f"bands{scale}{style}{norm}", bands)
        assert np.array_equal(b.get_bin_band_arr(), bin_band)
        np.testing.assert_allclose(b.get_fre_band_arr(), fre_band, rtol=1e-6)


def test_gammatone_bank_matches_golden_and_reference(product_lib, golden):
    g = golden("erb_gammatone.npz")
    b = af.BFT(64, 10, 32000, slide_length=256, scale_type=S.ERB, style_type=ST.GAMMATONE, data_type=D.POWER)
    got = b.get_filter_bank_arr()
    rowmax = np.abs(g["bank"]).max(axis=1, keepdims=True)
    assert (np.abs(got - g["bank"]) / rowmax).max() < 2e-5
    assert np.array_equal(b.get_bin_band_arr(), g["bin_band"])
    np.testing.assert_allclose(b.get_fre_band_arr(), g["fre_band"], rtol=1e-6)


@pytest.mark.parametrize("scale,lo,hi", [(4, 0.0, None), (2, 0.0, None), (3, 0.0, None), (1, 500.0, 7000.0), (6, 32.703196, 7000.0)])
def test_gammatone_banks_against_reference_build(product_lib, ref_lib, scale, lo, hi):
    for norm in (0, 1, 2):
        for num, r, sr in ((128, 11, 48000), (40, 10, 16000)):
            h = sr / 2 if hi is None else hi
            b = af.BFT(num, r, sr, low_fre=lo, high_fre=h, scale_type=S(scale), style_type=ST.GAMMATONE, normal_type=N(norm))
            q = af.BFT(num, r, sr, low_fre=lo, high_fre=h, scale_type=S(scale), style_type=ST.GAMMATONE, normal_type=N(norm), _lib=ref_lib)
            n = 1 << r
            l2, h2, _, _ = O.bft_revise_range(num, n, sr, lo, h, scale, 12)
            ref_bank = np.zeros((num + 4, n // 2 + 1), np.float32)
            fb = np.zeros(num + 2, np.float32)
            bb = np.zeros(num + 2, np.int32)
            ref_lib.auditory_filterBank(num, n, sr, 0, scale, 2, norm, float(l2), float(h2), 12, ref_bank.ctypes.data,
                                        fb.ctypes.data, bb.ctypes.data)
            rowmax = np.abs(ref_bank[:num]).max(axis=1, keepdims=True)
            assert (np.abs(b.get_filter_bank_arr() - ref_bank[:num]) / rowmax).max() < 5e-5
            assert np.array_equal(b.get_bin_band_arr(), q.get_bin_band_arr())
            np.testing.assert_allclose(b.get_fre_band_arr(), q.get_fre_band_arr(), rtol=1e-6)


# ---- planner of the fused MFCC kernel's bank loop: interval ("shared product") form of triangular banks ----
def _interval_plan(lib, bank, gain=None):
    num = bank.shape[0]
    owner = np.zeros(1025, np.int32)
    r = np.zeros(1025, np.float32)
    st = np.zeros(num + 1, np.int32)
    ln = np.zeros(num + 1, np.int32)
    tail = np.zeros(512, np.float32)
    gl = np.zeros(4, np.int32)
    ss = np.zeros(128, np.int32)
    bank = np.ascontiguousarray(bank, np.float32)
    g = None if gain is None else np.ascontiguousarray(gain, np.float32)
    ok = lib.afb200_mfccIntervalPlan(bank.ctypes.data, num, None if g is None else g.ctypes.data, owner.ctypes.data,
                                     r.ctypes.data, st.ctypes.data, ln.ctypes.data, tail.ctypes.data, gl.ctypes.data,
                                     ss.ctypes.data)
    return ok, owner, r, st, ln, tail, gl, ss


def _interval_mel(bank, gain, P, plan):
    """mel_m = g_m (A_m + S_{m+1} - A_{m+1}) exactly as the kernel evaluates it (float64 here)."""
    _, owner, r, st, ln, tail, _, _ = plan
    num = bank.shape[0]
    g = np.ones(num) if gain is None else gain.astype(np.float64)
    A = np.zeros(num + 1)
    S = np.zeros(num + 1)
    m = (owner >= 0) & (owner < num)
    np.add.at(A, owner[m], r[m].astype(np.float64) * P[m])
    np.add.at(S, owner[m], np.where(r[m] > 0, P[m], 0.0))
    U = S - A
    U[num] = sum(float(tail[i]) * P[st[num] + i] for i in range(ln[num]))
    return g * (A[:num] + U[1:num + 1])


@pytest.mark.parametrize("scale,style,norm,num,sr", [(2, 0, 0, 128, 48000), (2, 0, 1, 128, 48000), (2, 0, 2, 128, 48000),
                                                      (3, 1, 1, 64, 48000), (4, 0, 0, 128, 48000), (3, 0, 0, 128, 32000),
                                                      (2, 1, 0, 128, 48000), (2, 0, 0, 40, 16000), (2, 5, 0, 128, 48000),
                                                      (3, 0, 1, 100, 44100), (4, 1, 2, 77, 22050)])
def test_mfcc_interval_plan_reproduces_the_bank(product_lib, scale, style, norm, num, sr):
    lo, hi, _, _ = O.bft_revise_range(num, 2048, sr, None, None, scale, 12)
    bank, _, _ = O.auditory_filterbank(num, 2048, sr, scale, style, norm, float(lo), float(hi), 12)
    gain = None
    if norm:
        unit, _, _ = O.auditory_filterbank(num, 2048, sr, scale, style, 0, float(lo), float(hi), 12)
        pu = unit.max(1)
        gain = np.where(pu > 0, bank.max(1) / np.where(pu > 0, pu, 1), 1).astype(np.float32)
    plan = _interval_plan(product_lib, bank, gain)
    assert plan[0] == 1
    owner, r = plan[1], plan[2]
    assert (np.diff(owner[owner >= 0]) >= 0).all()                 # intervals are runs of consecutive bins
    assert ((r > 0) == (owner >= 0))[owner < num].all()            # every owned bin counts in S_j
    B = bank.astype(np.float64)
    rng = np.random.default_rng(0)
    for _ in range(3):
        P = rng.random(1025) ** 8 * 100
        want = B @ P
        assert np.abs(_interval_mel(bank, gain, P, plan) - want).max() <= 5e-7 * np.abs(want).max()
    eye = np.eye(1025)
    got = np.stack([_interval_mel(bank, gain, eye[k], plan) for k in range(1025)], axis=1)   # = the bank itself
    assert np.abs(got - B).max() <= 3e-7 * max(np.abs(B).max(), 1e-30)


def test_mfcc_interval_plan_rejects_other_banks(product_lib):
    rect, _, _ = O.auditory_filterbank(128, 2048, 48000, 2, 4, 0, 0.0, 24000.0, 12)    # overlapping boxes sum to 2
    assert _interval_plan(product_lib, rect)[0] == 0
    rnd = np.random.default_rng(1).random((16, 1025)).astype(np.float32)               # dense
    assert _interval_plan(product_lib, rnd)[0] == 0
    tri, _, _ = O.auditory_filterbank(128, 2048, 48000, 2, 0, 0, 0.0, 24000.0, 12)
    assert _interval_plan(product_lib, tri)[0] == 1
    bad = tri.copy()
    bad[40, np.nonzero(tri[40])[0][0]] *= 1.01                      # one weight off by 1 %: structure check must fail
    assert _interval_plan(product_lib, bad)[0] == 0
    assert _interval_plan(product_lib, tri, np.full(128, 2.0, np.float32))[0] == 0    # wrong gains


# ---- planner of the second-generation fused kernel (kernels/mfcc_fused2.cu): per-tile interval form with the bank's own weights ----
def _bank_plan2(lib, bank):
    num = bank.shape[0]
    bank = np.ascontiguousarray(bank, np.float32)
    owner = np.zeros(1025, np.int32)
    desc = np.zeros(num + 2, np.uint32)
    table = np.zeros((1408, 4), np.float32)
    piece = np.zeros(256, np.uint32)
    prefix = np.zeros(num + 2, np.uint16)
    assign = np.zeros(2 * 128, np.uint16)
    info = np.zeros(16, np.int32)
    n = lib.afb200_mfccBankPlan2(bank.ctypes.data, num, owner.ctypes.data, desc.ctypes.data, table.ctypes.data,
                                 piece.ctypes.data, prefix.ctypes.data, assign.ctypes.data, info.ctypes.data)
    passes, lanes = int(info[0]), int(info[1])
    plan = dict(n=n, owner=owner, desc=desc, table=table, piece=piece, prefix=prefix, pieces=int(info[2]), lmax=int(info[3]),
                first_pass2=int(info[4]), pass_len=info[5:5 + passes].copy(),
                assign=assign[:passes * lanes].reshape(passes, lanes) if n >= 0 else None)
    return plan


def _plan2_mel(num, P, plan):
    """the helper warps' two bank phases (mfcc_fused2.cu) in float64: per piece the partial sums (rise, fall), then
    mel_m = sum over the pieces of interval m of rise + sum over the pieces of interval m + 1 of fall"""
    Pp = np.concatenate([P, [0.0]])
    S = np.zeros((256, 2))
    seen = np.zeros(256, bool)
    for ps in range(plan["assign"].shape[0]):
        for pc in plan["assign"][ps]:
            if pc == 0xffff:
                continue
            d = int(plan["piece"][int(pc)])
            row, ln, off = d >> 20, (d >> 16) & 15, d & 0xffff
            assert 1 <= ln <= plan["pass_len"][ps] <= plan["lmax"] and not seen[pc]
            assert (int(pc) < plan["first_pass2"]) == (ps == 0)
            if ps == 1:
                assert row >= plan["first_pass2"]          # pass 1 never reads a row that already holds a pass-0 sum
            seen[pc] = True
            for j in range(ln):
                w = plan["table"][off + j].astype(np.float64)
                k = 2 * (row + j)
                S[pc, 0] += Pp[k] * w[0] + Pp[k + 1] * w[1]
                S[pc, 1] += Pp[k] * w[2] + Pp[k + 1] * w[3]
    assert seen[:plan["pieces"]].all() and not seen[plan["pieces"]:].any()
    pre = plan["prefix"].astype(int)
    return np.array([S[pre[m]:pre[m + 1], 0].sum() + S[pre[m + 1]:pre[m + 2], 1].sum() for m in range(num)])


@pytest.mark.parametrize("scale,style,norm,num,sr", [(2, 0, 0, 128, 48000), (2, 0, 1, 128, 48000), (2, 0, 2, 128, 48000),
                                                      (3, 1, 1, 64, 48000), (4, 0, 0, 128, 48000), (3, 0, 0, 128, 32000),
                                                      (2, 1, 0, 128, 48000), (2, 0, 0, 40, 16000), (2, 5, 0, 128, 48000),
                                                      (3, 0, 1, 100, 44100), (4, 1, 2, 77, 22050), (2, 0, 0, 1, 48000),
                                                      (2, 0, 0, 3, 8000)])
def test_mfcc_bank_plan2_reproduces_the_bank(product_lib, scale, style, norm, num, sr):
    lo, hi, _, _ = O.bft_revise_range(num, 2048, sr, None, None, scale, 12)
    bank, _, _ = O.auditory_filterbank(num, 2048, sr, scale, style, norm, float(lo), float(hi), 12)
    plan = _bank_plan2(product_lib, bank)
    assert 0 <= plan["n"] <= 1408 and 1 <= plan["pieces"] <= 256
    owner, desc = plan["owner"], plan["desc"]
    assert (np.diff(owner[owner >= 0]) >= 0).all()                 # intervals are runs of consecutive bins
    # the pieces of an interval tile its table range in order
    pre = plan["prefix"].astype(int)
    for i in range(num + 1):
        off, end, q0 = int(desc[i]) & 0xffff, int(desc[i + 1]) & 0xffff, int(desc[i]) >> 16
        for pc in range(pre[i], pre[i + 1]):
            d = int(plan["piece"][pc])
            assert (d & 0xffff) == off and (d >> 20) == q0 + (off - (int(desc[i]) & 0xffff))
            off += (d >> 16) & 15
        assert off == end
    if num == 128 and scale == 2:                                  # the headline bank: balanced, half-warps start in distinct bank pairs
        assert plan["lmax"] <= 4 and plan["assign"].shape[0] == 2
        for ps in range(plan["assign"].shape[0]):
            for h in range(plan["assign"].shape[1] // 16):
                pcs = [int(v) for v in plan["assign"][ps, 16 * h:16 * h + 16] if v != 0xffff]
                res = [(int(plan["piece"][v]) >> 20) & 15 for v in pcs]
                assert len(res) - len(set(res)) <= 4
    B = bank.astype(np.float64)
    rng = np.random.default_rng(0)
    for _ in range(2):
        P = rng.random(1025) ** 8 * 100
        want = B @ P
        got = _plan2_mel(num, P, plan)
        assert np.abs(got - want).max() <= 1e-12 * max(np.abs(want).max(), 1e-300)
    eye = np.eye(1025)
    got = np.stack([_plan2_mel(num, eye[k], plan) for k in range(0, 1025, 7)], axis=1)      # = the bank's own float weights
    assert np.array_equal(got, B[:, 0:1025:7])


def test_mfcc_bank_plan2_rejects_other_banks(product_lib):
    rnd = np.random.default_rng(1).random((16, 1025)).astype(np.float32)               # dense
    assert _bank_plan2(product_lib, rnd)["n"] == -1
    tri, _, _ = O.auditory_filterbank(128, 2048, 48000, 2, 0, 0, 0.0, 24000.0, 12)
    assert _bank_plan2(product_lib, tri)["n"] > 0
    bad = tri.copy()
    bad[10, 900] = 0.5                                              # a third filter on a high bin
    assert _bank_plan2(product_lib, bad)["n"] == -1


def test_mfcc_bank_plan2_random_banks(product_lib):
    """the fused kernel's host planner on 150 random banks of fftLength 2048 (every scale / style / normalisation the bank
    builder knows, 1 .. 128 bands, odd ranges): whenever it accepts a bank, its pieces, passes and lane assignment reproduce
    B . P exactly as the helper warps evaluate them; banks it declines go to the v1 / general kernels"""
    rng = np.random.default_rng(77)
    accepted = 0
    for _ in range(150):
        scale = int(rng.integers(1, 7))
        style = int(rng.choice([0, 0, 1, 3, 4, 5]))
        norm = int(rng.integers(0, 3))
        sr = int(rng.choice([8000, 16000, 22050, 32000, 44100, 48000]))
        num = int(rng.integers(1, 129))
        if scale == 5:
            num = int(rng.choice([12, 24, 36, 48, 60, 72, 84]))
        low = float(rng.choice([0.0, 20.0, 100.0, 300.0])) if scale not in (5, 6) else 32.703196
        high = float(rng.choice([sr / 2, 0.45 * sr, sr / 4]))
        try:
            lo, hi, _, _ = O.bft_revise_range(num, 2048, sr, low, high, scale, 12)
            bank, _, _ = O.auditory_filterbank(num, 2048, sr, scale, style, norm, float(lo), float(hi), 12)
        except (IndexError, ValueError, ZeroDivisionError):
            continue                                               # (band edges beyond Nyquist: no one-sided bank)
        if not np.isfinite(bank).all() or not bank.any():
            continue
        plan = _bank_plan2(product_lib, np.ascontiguousarray(bank, np.float32))
        if plan["n"] < 0:
            continue
        accepted += 1
        assert plan["n"] <= 1408 and 1 <= plan["pieces"] <= 256
        B = bank.astype(np.float64)
        P = rng.random(1025) ** 6 * 50
        want, got = B @ P, _plan2_mel(num, P, plan)
        assert np.abs(got - want).max() <= 1e-12 * max(np.abs(want).max(), 1e-300), (scale, style, norm, num, sr, low, high)
    assert accepted >= 40, accepted
