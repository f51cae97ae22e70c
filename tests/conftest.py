import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.realpath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on the B200 box)")


def rel_max(a, b):
    """max|a-b| / max|b|: the parity metric of BASELINE.md (pure element-wise relative error is
    meaningless near the 1e-8 log floor and for coefficients near zero).  `b` may be a RefSample: then
    the difference is taken on its elements and divided by the max|b| of the whole array."""
    if isinstance(b, RefSample):
        a = np.asarray(a, dtype=np.float64)
        assert a.shape == b.shape, (a.shape, b.shape)
        return float(np.abs(a.reshape(-1)[b.index] - b.values).max() / max(b.absmax, 1e-30))
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def ref_pair(a, b):
    """(a, b) as they are, or, when b is a RefSample, the elements of a at its sample and b's values."""
    if isinstance(b, RefSample):
        assert np.shape(a) == b.shape, (np.shape(a), b.shape)
        return np.asarray(a).reshape(-1)[b.index], b.values
    return a, b


def ref_absmax(b):
    """max |b| of a reference result, stored whole or as a RefSample"""
    return b.absmax if isinstance(b, RefSample) else float(np.abs(b).max())


def ref_window(lib, wt, n):
    """window_calFFTWindow of a library (reference build or product), copied out"""
    import ctypes as C
    p = lib.window_calFFTWindow(wt, n)
    return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_float)), shape=(n,)).copy()


# ---- results of the reference build, stored so that the comparisons run where it cannot be built ----
REF_GOLDEN = os.path.join(GOLDEN, "ref")
REF_RECORD = os.environ.get("AFB200_REF_RECORD")    # a directory: the reference results of this session are written there
REF_WHOLE = 256                                     # float arrays up to this many elements are stored whole
REF_AXIS = 96                                       # larger ones: up to this many indices of every axis, first and last
REF_EXTRA = 32                                      # included, + this many elements spread over the whole array
_recorded, _stored = {}, {}


def _sample_index(shape):
    """Flat indices of the stored sample of an array of `shape` (pure integer arithmetic: the same on every machine).
    Every index of an axis of up to REF_AXIS entries, and REF_AXIS evenly spaced ones of a longer axis (its first and
    last included), lies in at least one sampled element -- so every frame of a transform of up to REF_AXIS frames, and
    its first and last frame always; the other coordinates walk their axes at different strides.  REF_EXTRA more
    elements are spread evenly over the array, one per stratum."""
    shape = tuple(int(n) for n in shape)
    size = int(np.prod(shape))
    picks = [np.array([0, size - 1])]
    for d, n in enumerate(shape):
        k = np.unique(np.arange(min(n, REF_AXIS), dtype=np.int64) * (n - 1) // max(1, min(n, REF_AXIS) - 1))
        coords = [k if e == d else (k * (2 * e + 3) + 7 * d) % m for e, m in enumerate(shape)]
        picks.append(np.ravel_multi_index(coords, shape))
    j = np.arange(REF_EXTRA, dtype=np.int64)
    picks.append(j * size // REF_EXTRA + j * 7919 % max(1, size // REF_EXTRA))
    return np.unique(np.concatenate(picks))


class RefSample:
    """A fixed sample of a stored reference array: its shape, the values at _sample_index(shape) and the max |x| of the
    whole array (what rel_max divides by)."""

    def __init__(self, shape, values, absmax):
        self.shape, self.values, self.absmax = tuple(int(s) for s in shape), values.astype(np.float64), float(absmax)
        self.index = _sample_index(self.shape)


def _ref_store(key, a, out):
    a = np.asarray(a)
    if a.dtype.kind == "f" and a.size > REF_WHOLE:                 # one float32 member: ndim, shape, max |a|, sample
        head = [a.ndim, *a.shape, np.abs(a).max()]
        out[key + ".sample"] = np.concatenate((head, a.reshape(-1)[_sample_index(a.shape)])).astype(np.float32)
    else:
        out[key] = a


def _ref_load(key, st):
    if key in st:
        return st[key]
    if key + ".sample" in st:
        v = st[key + ".sample"]
        n = int(v[0])
        return RefSample(v[1:1 + n].astype(np.int64), v[2 + n:], v[1 + n])
    if key + "#n" in st:
        return tuple(_ref_load(f"{key}#{i}", st) for i in range(int(st[key + "#n"])))
    raise KeyError(key)


def _pack(arrays):
    """a module's stored arrays as two npz members -- a JSON manifest (key -> dtype, shape, byte offset) and one byte
    blob -- instead of one zip member and npy header per array"""
    manifest, blobs, pos = {}, [], 0
    for key, a in arrays.items():
        raw = np.ascontiguousarray(a).tobytes()
        manifest[key] = [np.asarray(a).dtype.str, list(np.shape(a)), pos]
        blobs.append(raw)
        pos += len(raw)
    return {"manifest": np.frombuffer(json.dumps(manifest).encode(), np.uint8), "data": np.frombuffer(b"".join(blobs), np.uint8)}


def _unpack(npz):
    manifest, data = json.loads(npz["manifest"].tobytes()), npz["data"].tobytes()
    return {key: np.frombuffer(data, np.dtype(dt), int(np.prod(shape)), pos).reshape(shape).copy()
            for key, (dt, shape, pos) in manifest.items()}


@pytest.fixture
def reference(request):
    """reference(name, fn) -> fn(reference library): computed by the reference build (oracle/_ref) where it is present;
    elsewhere read back from tests/golden/ref/<module>.npz, which a run with AFB200_REF_RECORD=<dir> and the reference
    build writes.  A stored float array larger than REF_WHOLE elements comes back as a RefSample; tuples stay tuples."""
    from oracle import ref_lib as R
    lib = R.get_ref_lib() if R.available() else None
    module = request.module.__name__.rsplit(".", 1)[-1]
    path = os.path.join(REF_GOLDEN, module + ".npz")

    def get(name, fn):
        key = f"{request.node.name}::{name}"
        if lib is not None:
            val = fn(lib)
            if REF_RECORD:
                _recorded.setdefault(module, {})[key] = val
            return val
        if module not in _stored:
            _stored[module] = _unpack(np.load(path)) if os.path.exists(path) else {}
        try:
            return _ref_load(key, _stored[module])
        except KeyError:
            pytest.fail(f"no stored reference result {key} in {os.path.relpath(path, ROOT)}")
    return get


def pytest_sessionfinish(session):
    if not (REF_RECORD and _recorded):
        return
    os.makedirs(REF_RECORD, exist_ok=True)
    for module, results in _recorded.items():
        out = {}
        for key, val in results.items():
            if isinstance(val, (tuple, list)):
                out[key + "#n"] = np.array(len(val))
                for i, v in enumerate(val):
                    _ref_store(f"{key}#{i}", v, out)
            else:
                _ref_store(key, val, out)
        np.savez_compressed(os.path.join(REF_RECORD, module + ".npz"), **_pack(out))


def noise(seed, n):
    return (0.1 * np.random.default_rng(seed).standard_normal(n)).astype(np.float32)


def tones(seed, n, sr):
    t = np.arange(n) / sr
    x = 0.3 * (np.sin(2 * np.pi * 220 * t) + np.sin(2 * np.pi * 880 * t) + np.sin(2 * np.pi * 3520 * t))
    return (x + 0.01 * np.random.default_rng(seed).standard_normal(n)).astype(np.float32)


@pytest.fixture(scope="session")
def golden():
    def load(name):
        return np.load(os.path.join(GOLDEN, name))
    return load


@pytest.fixture(scope="session")
def ref_lib():
    from oracle import ref_lib as R
    if not R.available():
        pytest.skip("oracle/_ref/libaudioflux_ref.so not built (needs /root/reference: make -C oracle)")
    return R.get_ref_lib()


@pytest.fixture(scope="session")
def product_lib():
    from audioflux_b200 import lib as L
    try:
        return L.get_lib()
    except L.LibraryNotBuilt:
        import __graft_entry__ as g
        g.build()
        return L.get_lib()


@pytest.fixture(scope="session")
def cuda_device(product_lib):
    if product_lib.afb200_deviceCount() <= 0:
        pytest.fail("no CUDA device visible to libaudioflux_b200 (gpu-marked test on a CPU box?)")
    return 0
