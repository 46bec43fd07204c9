"""The C-ABI library builds, loads without a GPU, and exports every symbol include/hipac_b200.h declares."""
import ctypes as C
import os
import re

import numpy as np

from conftest import ROOT
from oracle import hipac_oracle as orc


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "hipac_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(hipac_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(built_lib):
    from ss25_hierarchical_multiscale_image_classification_b200 import _lib
    syms = _declared_symbols()
    assert set(syms) == set(_lib.EXPORTS)
    for s in syms:
        assert hasattr(built_lib, s), s
    assert built_lib.hipac_abi_version() == 2


def test_pillow_coeff_tables_equal_oracle(built_lib):
    for scale in (2, 4, 8):
        a, b, c = (C.c_int32 * 16)(), (C.c_int32 * 12)(), (C.c_int32 * 12)()
        assert built_lib.hipac_pillow_coeffs(scale, a, b, c) == 0
        _, cnt, kk = orc.pil_bilinear_coeffs(224 * scale, 224)
        assert list(a)[:2 * scale] == list(kk[1, :2 * scale])
        assert list(b)[:cnt[0]] == list(kk[0, :cnt[0]])
        assert list(c)[:cnt[-1]] == list(kk[-1, :cnt[-1]])
    assert built_lib.hipac_pillow_coeffs(3, a, b, c) != 0
    assert b"scale" in built_lib.hipac_last_error()


def test_normalize_lut_equals_oracle(built_lib):
    lut = np.zeros((256, 3), dtype=np.uint16)
    assert built_lib.hipac_normalize_lut_bf16(lut.ctypes.data_as(C.c_void_p)) == 0
    assert np.array_equal(lut, orc.to_bf16_bits(orc.normalize_lut()))


def test_argument_validation_without_gpu(built_lib):
    assert built_lib.hipac_tile_scan_workspace_bytes(100, 100, 225, 224, 0, 1, 0) == 0
    assert b"patch size" in built_lib.hipac_last_error()
    assert built_lib.hipac_tile_scan_workspace_bytes(1000, 1000, 224, 224, 0, 5, 0) > 0
    assert built_lib.hipac_tile_scan_workspace_bytes(1000, 1000, 224, 224, 0, 6, 0) == 0
