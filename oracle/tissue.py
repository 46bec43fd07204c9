"""CPU oracle of the tissue segmentation and the tissue-mask patch filter -- TEST INFRASTRUCTURE, NOT PRODUCT.

A numpy restatement of OpenCV 4.13's 8-bit code paths for the CLAM-style thumbnail segmentation
``cv2.cvtColor(RGB2HSV)[..., 1] -> cv2.medianBlur(S, k) -> cv2.threshold(BINARY | OTSU)`` and of the filter rule of
``hipac_tile_scan_tissue``.  ``tests/test_tissue_oracle.py`` pins every function here against the installed ``cv2``;
``tests/test_tissue_gpu.py`` compares the kernels with these functions bit for bit.
"""
from __future__ import annotations

import numpy as np

from . import hipac_oracle as orc

FLT_EPSILON = float(np.finfo(np.float32).eps)
# OpenCV's RGB2HSV 8-bit saturation table: sdiv[i] = round(255 * 4096 / i) (no entry falls on a .5)
SDIV = np.array([0] + [int(round((255 << 12) / i)) for i in range(1, 256)], dtype=np.int64)


def saturation(img: np.ndarray) -> np.ndarray:
    """uint8 [H, W] HSV saturation of a uint8 [H, W, 3] image (RGB or BGR: max and min do not care)."""
    v = img.max(axis=2).astype(np.int64)
    d = v - img.min(axis=2).astype(np.int64)
    return ((d * SDIV[v] + (1 << 11)) >> 12).astype(np.uint8)


def median_blur(x: np.ndarray, k: int) -> np.ndarray:
    """k x k median with replicated borders (``cv2.medianBlur``), any image size."""
    if k == 1:
        return x.copy()
    r = k // 2
    h, w = x.shape
    p = np.pad(x, r, mode="edge")
    out = np.empty_like(x)
    for y0 in range(0, h, 256):          # bounded memory: k*k shifted copies of a band of rows
        y1 = min(h, y0 + 256)
        st = np.stack([p[y0 + dy:y1 + dy, dx:dx + w] for dy in range(k) for dx in range(k)], 0)
        out[y0:y1] = np.partition(st, k * k // 2, axis=0)[k * k // 2]
    return out


def otsu_threshold(x: np.ndarray) -> int:
    """OpenCV ``getThreshVal_Otsu_8u``: fp64, i ascending, no fused multiply-add."""
    h = np.bincount(x.ravel(), minlength=256)
    n = x.size
    scale = 1.0 / n
    mu = 0.0
    for i in range(256):
        mu += i * float(h[i])
    mu *= scale
    q1 = mu1 = max_sigma = 0.0
    t = 0
    for i in range(256):
        p = float(h[i]) * scale
        mu1 *= q1
        q1 += p
        q2 = 1.0 - q1
        if min(q1, q2) < FLT_EPSILON or max(q1, q2) > 1.0 - FLT_EPSILON:
            continue
        mu1 = (mu1 + i * p) / q1
        mu2 = (mu - q1 * mu1) / q2
        sigma = q1 * q2 * (mu1 - mu2) * (mu1 - mu2)
        if sigma > max_sigma:
            max_sigma = sigma
            t = i
    return t


def segment(img: np.ndarray, ksize: int = 7, threshold: int | None = None):
    """(mask uint8 [H, W] of 0 / 255, t, blurred saturation plane)."""
    blur = median_blur(saturation(img), ksize)
    t = otsu_threshold(blur) if threshold is None else int(threshold)
    return np.where(blur > t, 255, 0).astype(np.uint8), t, blur


def min_tissue_pixels(min_tissue, patch: int, scale: int) -> int:
    """ceil(min_tissue * (P/m)^2) in exact rational arithmetic."""
    from fractions import Fraction
    import math
    return math.ceil(Fraction(min_tissue) * (patch // scale) ** 2)


def tissue_count(tissue: np.ndarray, x: int, y: int, p: int, m: int) -> int:
    """Mask pixels > 0 in [y/m, (y+P)/m) x [x/m, (x+P)/m); outside the mask's extent counts as background."""
    return int(np.count_nonzero(tissue[y // m:(y + p) // m, x // m:(x + p) // m]))


def extract_patches_tissue_oracle(level_img: np.ndarray, mask: np.ndarray | None, level: int, tissue: np.ndarray, scale: int,
                                  min_tissue=0.5, stride=None, want_images: bool = True, row_range=None):
    """``hipac_oracle.extract_patches_oracle`` with the tissue-mask rule in place of ``mean > 240``."""
    h, w = level_img.shape[:2]
    p, s, grid = orc.candidate_grid(w, h, level, stride)
    need = min_tissue_pixels(min_tissue, p, scale)
    coords, labels, images = [], [], []
    n_cand = 0
    for x, y in grid:
        x, y = int(x), int(y)
        if row_range is not None and not (row_range[0] <= y // s < row_range[1]):
            continue
        n_cand += 1
        if tissue_count(tissue, x, y, p, scale) < need:
            continue
        coords.append((x, y))
        labels.append(orc.lesion_label(mask, x, y, p))
        if want_images:
            images.append(orc.pil_resize_bilinear(orc.padded_patch(level_img, x, y, p)))
    return dict(
        coords=np.asarray(coords, dtype=np.int32).reshape(-1, 2),
        labels=np.asarray(labels, dtype=np.uint8),
        images=(np.stack(images) if images else np.zeros((0, orc.OUT, orc.OUT, 3), np.uint8)) if want_images else None,
        candidates=n_cand, patch=p, stride=s)
