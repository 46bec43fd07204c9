"""Coarse-to-fine cascade over the pyramid: classify a coarse level everywhere, then tile and classify a finer level only
inside the footprints the coarse classifier flagged (the recipe of CAMELYON16 detection pipelines).

``roi_grid`` turns a coarse level's survivors and their scores into an ``RoiGrid``: a uint8 grid over the coarse level's
candidate grid, cell ``(i, j)`` set iff a survivor with ``score >= threshold`` sits at ``(i*S_c, j*S_c)`` or within
Chebyshev distance ``dilate`` cells of it (``hipac_roi_grid``, two kernels, the survivor count read on the device).  Passed
as ``roi=`` to ``extract_patches_tensor`` / ``process_level`` / ``process_level_exchanged`` of a finer level, it keeps a
candidate only if its footprint overlaps with positive area the footprint of a set cell, both taken at the finer level's
resolution (``hipac_tile_scan_roi``); the rejected candidates never reach the resample or the network.
``process_cascade`` chains the two steps over a list of levels.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from . import pipeline as _pipeline
from .preprocessing.tensor_api import grid_shape, patch_and_stride


@dataclass
class RoiGrid:
    """Region of interest on a coarse level's candidate grid."""
    grid: torch.Tensor    # uint8 [ny, nx] on the device, 1 = set
    level: int            # the coarse level
    stride: int           # S_c
    patch: int            # P_c
    nx: int
    ny: int


def tumor_margin(logits: torch.Tensor) -> torch.Tensor:
    """Score of a binary classifier: ``logits[:, 1] - logits[:, 0]`` (one fp32 subtraction)."""
    return logits[:, 1] - logits[:, 0]


def threshold_of(tau: float) -> float:
    """The margin threshold of a probability threshold ``tau`` in (0, 1): ``float32(log(tau) - log1p(-tau))``, computed in
    fp64.  ``tumor_margin(logits) >= threshold_of(tau)`` is the cascade's rule; it equals ``softmax(logits)[:, 1] >= tau``
    up to rounding (the two can differ only when the probability is within a few ulps of ``tau``)."""
    tau = float(tau)
    if not 0.0 < tau < 1.0:
        raise ValueError(f"tau must lie in (0, 1), got {tau}")
    return float(np.float32(math.log(tau) - math.log1p(-tau)))


def roi_grid(coords: torch.Tensor, scores: torch.Tensor, level: int, width: int, height: int, stride=None,
             threshold: float = 0.0, dilate: int = 0, count: torch.Tensor | None = None) -> RoiGrid:
    """ROI of the coarse level ``level`` (a ``width`` x ``height`` image tiled at ``stride``) from its survivors.

    ``coords``: int32 ``[n, 2]`` survivor coordinates (level pixels), ``scores``: float32 ``[n]`` on the same device, e.g.
    ``tumor_margin(logits)`` with ``threshold = threshold_of(tau)``, or ``labels.float()`` with ``threshold = 0.5`` for
    lesion-guided mining.  ``count``: optional int32 device counter (element 0); then ``min(count[0], n)`` rows are read
    on the device and nothing waits on the host.  ``dilate`` >= 0 grows every positive cell by that many cells."""
    P, S = patch_and_stride(level, stride)
    nx, ny = grid_shape(int(width), int(height), S)
    if not (coords.is_cuda and coords.dtype == torch.int32 and coords.dim() == 2 and coords.shape[1] == 2):
        raise ValueError("coords must be a CUDA int32 tensor of shape [n, 2]")
    if not (scores.is_cuda and scores.dtype == torch.float32 and scores.dim() == 1 and scores.device == coords.device):
        raise ValueError("scores must be a float32 [n] tensor on the device of coords")
    n = int(coords.shape[0])
    if int(scores.shape[0]) < n:
        raise ValueError(f"{int(scores.shape[0])} scores for {n} coordinates")
    if int(dilate) < 0:
        raise ValueError("dilate must be >= 0")
    dev = coords.device
    l = _lib.lib()
    if l.hipac_roi_grid_bytes(nx, ny) == 0:
        raise ValueError(l.hipac_last_error().decode())
    st = torch.cuda.current_stream(dev)
    with torch.cuda.device(dev):
        coords, scores = coords.contiguous(), scores.contiguous()
        if count is None:
            count = torch.tensor([n], dtype=torch.int32, device=dev)
        elif not (count.is_cuda and count.dtype == torch.int32 and count.device == dev):
            raise ValueError("count must be an int32 tensor on the device of coords")
        grid = torch.empty((ny, nx), dtype=torch.uint8, device=dev)
        _lib.check(l.hipac_roi_grid(coords.data_ptr() if n else None, scores.data_ptr() if n else None, count.data_ptr(), n,
                                    float(threshold), S, nx, ny, int(dilate), grid.data_ptr(), st.cuda_stream), "hipac_roi_grid")
    return RoiGrid(grid, int(level), S, P, nx, ny)


def process_cascade(levels: dict, packed, order=(3, 0), tau: float = 0.5, dilate: int = 0, stride=None, tissue=None,
                    tissue_level: int | None = None, min_tissue=0.5, chunk: int = 8192, tta: bool = False,
                    stain=None) -> dict:
    """Coarse-to-fine cascade over the levels in ``order`` (strictly decreasing, e.g. ``(3, 0)`` or the chain ``(3, 1, 0)``).

    ``levels`` maps a level number to ``(img, lesion_mask)`` on the device (``lesion_mask`` may be None); ``packed`` is one
    ``PackedResNet18`` with a head of at least two classes, or a dict of them per level.  The first level is processed in
    full; every later level only inside the ROI of the previous one, whose positive survivors are those with
    ``tumor_margin(logits) >= threshold_of(tau)`` (dilated by ``dilate`` cells).  ``tissue``: optional tissue mask of level
    ``tissue_level`` (e.g. ``segment_tissue`` of the thumbnail), used at scale ``2 ** (tissue_level - L)`` for every level
    ``L`` in place of the ``mean > 240`` rule.  ``tta``: every level is classified with the D4 test-time augmentation
    (``process_level(tta=True)``), so each ROI is scored on the averaged logits.  ``stain``: one ``StainNormalizer`` for
    every level (one slide, one stain), applied to every survivor before the network.  Returns ``{level: LevelResult}``; each fine result equals the full
    ``process_level`` of that level restricted to the ROI."""
    order = tuple(int(L) for L in order)
    if not order or any(a <= b for a, b in zip(order, order[1:])):
        raise ValueError(f"order {order} must list levels from coarse to fine (strictly decreasing)")
    if tissue is not None and (tissue_level is None or tissue_level < order[0]):
        raise ValueError("a tissue mask needs its tissue_level, at or above the coarsest level of the cascade")
    theta = threshold_of(tau)
    results, roi = {}, None
    for k, L in enumerate(order):
        img, mask = levels[L]
        net = packed[L] if isinstance(packed, dict) else packed
        tis = {} if tissue is None else dict(tissue=tissue, tissue_scale=1 << (tissue_level - L), min_tissue=min_tissue)
        r = _pipeline.process_level(img, mask, L, net, stride=stride, chunk=chunk, roi=roi, tta=tta, stain=stain, **tis)
        results[L] = r
        if k + 1 < len(order):
            if r.logits is None or r.logits.shape[1] < 2:
                raise ValueError(f"the classifier of level {L} needs at least two classes to score the cascade")
            roi = roi_grid(r.coords, tumor_margin(r.logits), L, int(img.shape[1]), int(img.shape[0]), stride=stride,
                           threshold=theta, dilate=dilate)
    return results
