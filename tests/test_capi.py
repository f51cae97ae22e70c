"""The C-ABI library loads, exports every symbol include/*.h declares, and fails loudly
(status + message, no CPU fallback) when no GPU is usable.  No compute calls here."""
import ctypes
import os
import re

import numpy as np

import audioflux_b200 as af
from audioflux_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.realpath(__file__)))


def declared_symbols():
    names = set()
    for f in sorted(os.listdir(os.path.join(ROOT, "include"))):
        src = open(os.path.join(ROOT, "include", f)).read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        for m in re.finditer(r"\b([A-Za-z_][A-Za-z0-9_]*)\s*\(", src):
            n = m.group(1)
            if re.match(r"(stftObj_|bftObj_|xxccObj_|cqtObj_|cwtObj_|pwtObj_|wsstObj_|synsqObj_|reassignObj_|spectrogramObj_|afb200_)", n):
                names.add(n)
    return names


def test_every_declared_symbol_is_exported(product_lib):
    names = declared_symbols()
    assert len(names) > 50
    missing = [n for n in sorted(names) if not hasattr(product_lib, n)]
    assert not missing, missing


def test_binding_table_matches_headers(product_lib):
    declared = declared_symbols()
    for table in (capi.REFERENCE_API, capi.EXTENSION_API):
        for name in table:
            assert name in declared, f"{name} bound in capi.py but not declared in include/"


def test_reference_build_exports_the_same_c_api(reference):
    exported = reference("exported", lambda lib: np.array([hasattr(lib, name) for name in capi.REFERENCE_API]))
    assert len(exported) == len(capi.REFERENCE_API)
    for name, present in zip(capi.REFERENCE_API, exported):
        assert present, name


def test_no_gpu_means_loud_failure(product_lib):
    if product_lib.afb200_deviceCount() > 0:
        return
    b = af.BFT(128, 11, 48000, slide_length=512, scale_type=af.SpectralFilterBankScaleType.MEL)
    x = np.zeros((2, 48000), np.float32)
    try:
        b.mfcc_batch(x, 40)
        raised = False
    except af.lib.AfB200Error as e:
        raised = "no CUDA device" in str(e)
    assert raised
    # legacy void entry point: output untouched, message recorded
    out = np.full((90, 128), 7.0, np.float32)
    im = np.zeros_like(out)
    product_lib.bftObj_bft(b._obj, x[0].ctypes.data, 48000, out.ctypes.data, im.ctypes.data)
    assert (out == 7.0).all()
    assert b"no CUDA device" in product_lib.afb200_lastError()


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "audioflux_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".c", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "import oracle" not in src and "from oracle" not in src and "oracle/" not in src.replace("oracle/_ref", ""), f
