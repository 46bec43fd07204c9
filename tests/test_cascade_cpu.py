"""Coarse-to-fine cascade without a GPU: the oracle's closed-form ROI test against painted footprints, the margin threshold
against the softmax rule, and the library's argument checks."""
import ctypes as C

import numpy as np
import pytest

from oracle import cascade as oc

PATCH = {0: 1792, 1: 896, 2: 448, 3: 224}


def _painted_truth(fine_xy, pf, lf, roi, lc):
    """Paint every set cell's footprint at level-0 resolution, then ask each fine footprint (level-0 pixels) whether it
    covers a painted pixel (summed-area table)."""
    ny, nx = roi.grid.shape
    ext = max(((nx - 1) * roi.stride + roi.patch) << lc, ((int(fine_xy[:, 0].max()) + pf) << lf) + 1,
              ((ny - 1) * roi.stride + roi.patch) << lc, ((int(fine_xy[:, 1].max()) + pf) << lf) + 1)
    paint = np.zeros((ext, ext), np.uint8)
    for j, i in zip(*np.nonzero(roi.grid)):
        x0, y0 = (int(i) * roi.stride) << lc, (int(j) * roi.stride) << lc
        paint[y0:y0 + (roi.patch << lc), x0:x0 + (roi.patch << lc)] = 1
    sat = np.zeros((ext + 1, ext + 1), np.int32)
    sat[1:, 1:] = paint.cumsum(0, dtype=np.int32).cumsum(1, dtype=np.int32)
    out = []
    for x, y in fine_xy:
        a0, b0, a1, b1 = int(x) << lf, int(y) << lf, (int(x) + pf) << lf, (int(y) + pf) << lf
        out.append(sat[b1, a1] - sat[b0, a1] - sat[b1, a0] + sat[b0, a0] > 0)
    return np.array(out)


@pytest.mark.parametrize("lc,lf", [(3, 0), (3, 1), (2, 0), (1, 0)])
@pytest.mark.parametrize("stride_kind", ["cli", "nonoverlap"])
def test_closed_form_roi_test_equals_painted_footprints(lc, lf, stride_kind):
    rng = np.random.default_rng(lc * 10 + lf + (0 if stride_kind == "cli" else 100))
    w0, h0 = 5000 + 37 * lc, 4300 + 11 * lf                       # level-0 size: not multiples of any stride
    wc, hc, wf, hf = w0 >> lc, h0 >> lc, w0 >> lf, h0 >> lf
    sc = 224 if stride_kind == "cli" else PATCH[lc]
    sf = 224 if stride_kind == "cli" else PATCH[lf]
    pc, pf = PATCH[lc], PATCH[lf]
    nxc, nyc = -(-wc // sc), -(-hc // sc)
    cc = np.array([(i * sc, j * sc) for i in range(nxc) for j in range(nyc)], np.int32)
    fine = np.array([(x, y) for x in range(0, wf, sf) for y in range(0, hf, sf)], np.int64)   # border candidates included
    for dilate in (0, 1, 2):
        for frac in (0.0, 0.15, 0.5):
            scores = rng.standard_normal(len(cc)).astype(np.float32)
            thr = np.quantile(scores, 1 - frac) if frac else np.inf
            roi = oc.Roi(oc.roi_grid(cc, scores, thr, sc, nxc, nyc, dilate), lc, sc, pc)
            got = np.array([oc.in_roi(x, y, pf, roi, lc - lf) for x, y in fine])
            want = _painted_truth(fine, pf, lf, roi, lc)
            assert np.array_equal(got, want), (lc, lf, stride_kind, dilate, frac)
            if frac == 0.0:
                assert not got.any()
            res = {"coords": fine.astype(np.int32), "labels": np.arange(len(fine)) % 2, "candidates": len(fine)}
            r = oc.restrict(res, roi, lf, stride=sf)
            assert np.array_equal(r["coords"], fine[want]) and r["candidates"] == len(fine)


def test_roi_grid_dilation_is_chebyshev_and_clipped():
    cc = np.array([[0, 0], [224 * 5, 224 * 3], [224 * 9, 224 * 9]], np.int32)
    s = np.array([1.0, 1.0, -1.0], np.float32)
    g = oc.roi_grid(cc, s, 0.0, 224, 8, 6, dilate=2)
    want = np.zeros((6, 8), np.uint8)
    want[0:3, 0:3] = 1
    want[1:6, 3:8] = 1
    assert np.array_equal(g, want)


def test_threshold_of_matches_softmax_rule():
    from ss25_hierarchical_multiscale_image_classification_b200.cascade import threshold_of
    rng = np.random.default_rng(3)
    logits = (rng.standard_normal((20000, 2)) * 4).astype(np.float32)
    margin = logits[:, 1] - logits[:, 0]                        # fp32 subtraction, as tumor_margin
    l64 = logits.astype(np.float64)
    p1 = 1.0 / (1.0 + np.exp(l64[:, 0] - l64[:, 1]))
    for tau in (0.01, 0.1, 0.3, 0.5, 0.7, 0.9, 0.99, 0.999):
        theta = threshold_of(tau)
        assert np.float32(theta) == theta
        away = np.abs(p1 - tau) > 1e-5
        assert away.sum() > 100
        assert np.array_equal((margin >= np.float32(theta))[away], (p1 >= tau)[away]), tau
    assert threshold_of(0.5) == 0.0
    for bad in (0.0, 1.0, -0.1, 1.5):
        with pytest.raises(ValueError):
            threshold_of(bad)


def _scan_roi(lib, fine_level=0, coarse_level=3, S=224, mode=0, roi_stride=224, roi_patch=224, tissue_scale=0):
    fake = C.c_void_p(1 << 20)                                    # never dereferenced: validation fails first
    P = PATCH[fine_level]
    return lib.hipac_tile_scan_roi(fake, 4000, 4000, 4000 * 3, None, 0, P, S, 0, 18, fake, fake, None, fake, 2, fake, 100,
                                   fake, 1 << 30, mode, None, 0, 0, 0, tissue_scale, 0, fake, 3, 3,
                                   coarse_level - fine_level, roi_stride, roi_patch, 0, None)


def test_library_refuses_bad_roi_arguments_without_gpu(built_lib):
    lib = built_lib
    assert _scan_roi(lib, fine_level=0, coarse_level=0) == -1            # Lc <= Lf
    assert b"coarser level" in lib.hipac_last_error()
    assert _scan_roi(lib, fine_level=1, coarse_level=0) == -1
    assert b"coarser level" in lib.hipac_last_error()
    assert _scan_roi(lib, roi_stride=0) == -1
    assert b"roi_stride" in lib.hipac_last_error()
    assert _scan_roi(lib, roi_patch=-224) == -1
    assert b"roi_patch" in lib.hipac_last_error()
    assert _scan_roi(lib, S=0) == -1                                     # the fine level's stride
    assert b"stride must be positive" in lib.hipac_last_error()
    assert _scan_roi(lib, mode=0x100) == -1                              # HIPAC_SCAN_KEEP_ALL
    assert b"KEEP_ALL" in lib.hipac_last_error()
    assert _scan_roi(lib, tissue_scale=3) == -1
    assert b"tissue_scale" in lib.hipac_last_error()
    fake = C.c_void_p(1 << 20)
    assert lib.hipac_roi_grid(fake, fake, fake, 10, C.c_float(0.0), 0, 4, 4, 0, fake, None) == -1
    assert b"stride" in lib.hipac_last_error()
    assert lib.hipac_roi_grid(fake, fake, fake, 10, C.c_float(0.0), 224, 4, 4, -1, fake, None) == -1
    assert b"dilate" in lib.hipac_last_error()
    assert lib.hipac_roi_grid(fake, fake, fake, 10, C.c_float(0.0), 224, 0, 4, 0, fake, None) == -1
    assert lib.hipac_roi_grid_bytes(0, 5) == 0 and lib.hipac_roi_grid_bytes(7, 5) == 35
    assert lib.hipac_tile_scan_roi_workspace_bytes(1000, 1000, 224, 224, 0, 5, 0, 0) == \
        lib.hipac_tile_scan_workspace_bytes(1000, 1000, 224, 224, 0, 5, 0)
    assert lib.hipac_tile_scan_roi_workspace_bytes(1000, 1000, 224, 224, 0, 5, 0, 8) == \
        lib.hipac_tile_scan_tissue_workspace_bytes(1000, 1000, 224, 224, 0, 5, 0, 8)

