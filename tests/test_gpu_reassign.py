"""Reassignment on the GPU (reassignObj_reassign / reassignObj_reassignBatch, kernels/reassign.cu) against the numpy
oracle and the reference build.  Parity bar as in tests/test_reassign_cpu.py (indices are roundf() of float32 divides):
>= 99.5 % of the cells identical to 1e-5 of the maximum and relative Frobenius error <= 5e-3 for the reassigned planes,
1e-4 for the plain half spectrum; the GPU scatter is bit-stable across runs (64-bit fixed-point accumulation)."""
import numpy as np
import pytest

from conftest import ref_pair, rel_max
from oracle import af_oracle as O
from test_reassign_cpu import _signal, agree, CASES

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("radix,sr,window,hop,re_type,thresh,pad,order,result_type", CASES)
def test_reassign_vs_oracle(cuda_device, radix, sr, window, hop, re_type, thresh, pad, order, result_type):
    import audioflux_b200 as af
    x = _signal(20000, sr, radix)
    r = af.Reassign(radix, sr, af.WindowType(window), hop, af.ReassignType(re_type), thresh, bool(pad))
    r.set_order(order)
    got = r.reassign_planes(x, result_type)
    want = O.reassign(x, radix, sr, window, hop, re_type, thresh, bool(pad), order, result_type)
    assert rel_max(got[2], want[2]) < 1e-4 and rel_max(got[3], want[3]) < 1e-4
    for k in ((0,) if result_type else (0, 1)):
        same, fro = agree(got[k], want[k])
        assert same >= 0.995 and fro <= 5e-3, (k, same, fro)
    if result_type:
        assert not got[1].any()                                   # the imaginary plane is left alone in amplitude mode


def test_reassign_vs_reference_build_and_python_layout(cuda_device, reference):
    import audioflux_b200 as af
    x = _signal(30000, 32000, 11)
    got = af.Reassign(10, 32000).reassign_planes(x)
    want = reference("planes", lambda lib: af.Reassign(10, 32000, _lib=lib).reassign_planes(x))
    assert rel_max(got[2], want[2]) < 1e-4 and rel_max(got[3], want[3]) < 1e-4
    for g, w in zip(got[:2], want[:2]):
        same, fro = agree(*ref_pair(g, w))
        assert same >= 0.995 and fro <= 5e-3, (same, fro)
    m1, m2 = af.Reassign(10, 32000).reassign(np.stack([x, x[::-1].copy()]))
    assert m1.shape == (2, 513, got[0].shape[0]) and np.iscomplexobj(m1)
    assert np.allclose(m1[0].T.real, got[0]) and np.allclose(m2[0].T.imag, got[3])


def test_reassign_none_and_accumulation_and_bit_stability(cuda_device):
    import audioflux_b200 as af
    from audioflux_b200.base import np_ptr
    x = _signal(12000, 16000, 4)
    r0 = af.Reassign(9, 16000, re_type=af.ReassignType.NONE)
    a = r0.reassign_planes(x)
    want = O.reassign(x, 9, 16000, re_type=O.REASSIGN_NONE)
    assert rel_max(a[0], want[0]) < 1e-4 and rel_max(a[1], want[1]) < 1e-4
    r = af.Reassign(9, 16000)
    one = r.reassign_planes(x)
    two = r.reassign_planes(x)
    assert all(np.array_equal(p, q) for p, q in zip(one, two))            # bit-stable
    T, W = one[0].shape
    re = np.full((T, W), 2.0, np.float32)
    im = np.full((T, W), -1.0, np.float32)
    r._lib.reassignObj_reassign(r._obj, np_ptr(x), len(x), np_ptr(re), np_ptr(im), None, None)
    assert np.allclose(re, one[0] + np.float32(2.0), rtol=0, atol=1e-5 * np.abs(one[0]).max())   # ADDED to the caller's planes
    assert np.allclose(im, one[1] - np.float32(1.0), rtol=0, atol=1e-5 * np.abs(one[1]).max())


def test_reassign_batch_host_and_device_match_single_clips(cuda_device):
    import torch
    import audioflux_b200 as af
    xs = np.stack([_signal(16000, 16000, s) * (s + 1) for s in range(5)])
    r = af.Reassign(9, 16000, slide_length=100)
    single = [r.reassign_planes(x) for x in xs]
    host = r.reassign_batch(xs)
    dev = r.reassign_batch(torch.from_numpy(xs).cuda())
    torch.cuda.synchronize()
    for k in range(4):
        want = np.stack([s[k] for s in single])
        assert np.array_equal(host[k], want)
        assert np.array_equal(dev[k].cpu().numpy(), want)


@pytest.mark.parametrize("result_type,data_type", [(1, 0), (1, 1), (0, 0), (0, 1)])
def test_bft_with_reassign_vs_reference_build(cuda_device, reference, result_type, data_type):
    """bftObj_new(isReassign = 1): the bank over the reassigned spectrum.  Compared with the FIRST call of a fresh
    reference object (from its second call on the reference keeps adding into its cached planes)."""
    import audioflux_b200 as af
    S, D = af.SpectralFilterBankScaleType, af.SpectralDataType
    x = _signal(16000, 16000, 21)
    def bft(lib):
        b = af.BFT(64, 9, 16000, slide_length=128, scale_type=S.MEL, data_type=D(data_type), is_reassign=True, _lib=lib)
        out = b.bft(x, result_type=result_type)
        # a complex result as its interleaved (re, im) float32 view: the same Frobenius norm, and sampled when stored
        return (np.ascontiguousarray(out).view(np.float32) if np.iscomplexobj(out) else out), np.abs(out)
    (got, got_abs), (want, want_abs) = bft(None), reference("bft,abs", bft)
    assert got.shape == want.shape
    g, w = ref_pair(got, want)
    err = np.linalg.norm(g - w) / np.linalg.norm(w)
    assert err <= 1e-2, err                      # cells within an ulp of a rounding boundary move by one bin (see above)
    assert rel_max(got_abs, want_abs) < 5e-2


def test_bft_temporal_descriptors_vs_reference_build(cuda_device, reference):
    """bftObj_new(isTemporal = 1): energy / rms / zero-crossing rate of the windowed frames (src/temporal_algorithm.c:93-146)"""
    import audioflux_b200 as af
    S = af.SpectralFilterBankScaleType
    x = _signal(20000, 16000, 31)
    def temporal(lib):
        b = af.BFT(64, 10, 16000, slide_length=200, scale_type=S.MEL, is_temporal=True, _lib=lib)
        b.bft(x, result_type=1)
        return b.get_temporal_data(len(x))
    outs = [temporal(None), reference("temporal", temporal)]
    for g, w in zip(*outs):
        assert g.shape == w.shape and g.shape[0] == (20000 - 1024) // 200 + 1
        assert rel_max(g, w) < 1e-5
    w = O.fft_window(O.W_HANN, 1024).astype(np.float64)
    fr = np.stack([x[t * 200:t * 200 + 1024] * w for t in range(outs[0][0].shape[0])])
    assert rel_max(outs[0][0], (fr ** 2).sum(1)) < 1e-5
    assert np.array_equal(outs[0][2], ((fr[:, 1:] * fr[:, :-1] < 0).sum(1) / 1024).astype(np.float32))
