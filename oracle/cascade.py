"""numpy restatement of the coarse-to-fine cascade (csrc/cascade.cu, include/hipac_b200.h "Coarse-to-fine cascade").

``roi_grid``  cell (i, j) of the coarse candidate grid is set iff a survivor with ``score >= threshold`` (fp32) at coarse
              coordinates (i*S_c, j*S_c) lies within Chebyshev distance ``dilate`` cells.
``in_roi``    a fine candidate at fine pixel (x, y) (y global) is in the ROI iff its footprint [x, x+P_f) x [y, y+P_f)
              overlaps with positive area the footprint [i*S_c << d, (i*S_c + P_c) << d) x (same on y) of a set cell,
              d = Lc - Lf, closed form per axis (cells outside the grid are not set).
``restrict``  the rows of an unfiltered result whose candidates are in the ROI.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from . import hipac_oracle as orc


@dataclass
class Roi:
    grid: np.ndarray      # uint8 [ny, nx]
    level: int
    stride: int
    patch: int


def roi_grid(coords: np.ndarray, scores: np.ndarray, threshold: float, stride: int, nx: int, ny: int, dilate: int = 0) -> np.ndarray:
    grid = np.zeros((ny, nx), np.uint8)
    coords = np.asarray(coords, np.int64).reshape(-1, 2)
    pos = np.asarray(scores, np.float32) >= np.float32(threshold)
    for x, y in coords[pos]:
        if x < 0 or y < 0:
            continue
        i, j = int(x) // stride, int(y) // stride
        if i >= nx or j >= ny:
            continue
        grid[max(j - dilate, 0):j + dilate + 1, max(i - dilate, 0):i + dilate + 1] = 1
    return grid


def cell_range(v: int, p: int, a: int, b: int, n: int):
    """Cells [c0, c1] whose extent [c*a, c*a + b) overlaps [v, v + p) with positive area."""
    return max((v - b) // a + 1, 0), min((v + p - 1) // a, n - 1)


def in_roi(x: int, y: int, patch: int, roi: Roi, shift: int) -> bool:
    ny, nx = roi.grid.shape
    a, b = roi.stride << shift, roi.patch << shift
    i0, i1 = cell_range(int(x), patch, a, b, nx)
    j0, j1 = cell_range(int(y), patch, a, b, ny)
    if i0 > i1 or j0 > j1:
        return False
    return bool(roi.grid[j0:j1 + 1, i0:i1 + 1].any())


def roi_mask(coords: np.ndarray, level: int, roi: Roi, stride=None, y_origin: int = 0) -> np.ndarray:
    """bool [n]: which fine candidates at ``coords`` (level pixels of ``level``, rows relative to ``y_origin``) are in the ROI."""
    p, _ = orc.patch_and_stride(level, stride)
    c = np.asarray(coords, np.int64).reshape(-1, 2)
    return np.array([in_roi(x, y + y_origin, p, roi, roi.level - level) for x, y in c], dtype=bool)


def restrict(result: dict, roi: Roi, level: int, stride=None, y_origin: int = 0) -> dict:
    """The rows of an unfiltered result (a dict with ``coords`` and other per-row arrays) whose candidates are in the ROI;
    entries that are not per-row arrays (e.g. ``candidates``) are kept as they are."""
    coords = np.asarray(result["coords"])
    keep = roi_mask(coords, level, roi, stride, y_origin)
    n = len(coords)
    return {k: (v[keep] if isinstance(v, np.ndarray) and v.ndim >= 1 and v.shape[0] == n else v) for k, v in result.items()}
