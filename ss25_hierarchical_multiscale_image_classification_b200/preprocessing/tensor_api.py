"""In-HBM patch extraction: the fast path under the reference's ``extract_patches``.

``extract_patches_tensor`` replaces the hot loop of the reference's ``extract_patches``
(``src/main.py:682-727``) and the ``Resize/ToTensor/Normalize`` of its feature-extraction
transform (``src/main.py:812-818``) for one level image already resident in device memory.
All arithmetic happens in ``libhipac_b200.so`` (``hipac_tile_scan``); this module only sizes
buffers and moves pointers.  There is no CPU fallback.
"""
from __future__ import annotations

import math
import threading
from dataclasses import dataclass
from fractions import Fraction

import torch

from .. import _lib

PATCH_SIZES = {0: 1792, 1: 896, 2: 448, 3: 224}   # reference src/main.py:614
OUT = 224
S2D16_WIDTH = 115   # 112 + explicit zero columns (2 left, 1 right), include/hipac_b200.h

_LAYOUTS = {"nhwc3": _lib.LAYOUT_NHWC3_BF16, "s2d16": _lib.LAYOUT_S2D16_BF16}
_MODES = {"auto": _lib.SCAN_AUTO, "direct": _lib.SCAN_DIRECT, "fused": _lib.SCAN_FUSED,
          "fused_legacy": _lib.SCAN_FUSED | _lib.SCAN_NO_STREAM}   # cp.async kernels instead of the TMA streaming pass


_count_host = threading.local()


def _pinned_count():
    """Per-thread pinned int32[2] registered with the library for the early survivor count."""
    buf = getattr(_count_host, "buf", None)
    if buf is None:
        buf = torch.zeros(2, dtype=torch.int32).pin_memory()
        _lib.check(_lib.lib().hipac_tile_scan_set_count_buffer(buf.data_ptr()), "hipac_tile_scan_set_count_buffer")
        _count_host.buf = buf
    return buf


def patch_and_stride(level: int, stride=None, patch_size: int = 224):
    """``stride = stride or patch_size`` happens BEFORE the level map overwrites the patch size
    (reference ``src/main.py:611`` vs ``614-615``), so the CLI stride is 224 at every level."""
    s = stride or patch_size
    return PATCH_SIZES.get(level, 224), int(s)


def grid_shape(width: int, height: int, stride: int):
    """(nx, ny) of the candidate grid ``range(0,W,S) x range(0,H,S)`` (reference ``src/main.py:682-686``)."""
    return (width + stride - 1) // stride, (height + stride - 1) // stride


@dataclass
class PatchBatch:
    """Survivors of one ``hipac_tile_scan`` call, in the reference's emission order (x outer, y inner)."""
    coords: torch.Tensor            # int32 [N,2] (x, y) in level pixels
    labels: torch.Tensor            # uint8 [N] 1 = tumor, 0 = normal
    batch: torch.Tensor | None      # bf16 [N,224,224,3] ("nhwc3") or [N,112,115,16] ("s2d16")
    images_u8: torch.Tensor | None  # uint8 [N,224,224,3] Pillow-exact resized patches
    layout: str | None
    candidates: int
    patch: int
    stride: int
    level: int

    def __len__(self):
        return int(self.coords.shape[0])


@dataclass
class PendingPatchBatch:
    """A tile scan that has been enqueued but whose survivor count has not been read on the host yet: capacity-sized
    tensors plus the device counter.  ``resolve()`` waits for the count only (not for the kernels) and slices."""
    coords: torch.Tensor
    labels: torch.Tensor
    batch: torch.Tensor | None
    images_u8: torch.Tensor | None
    count: torch.Tensor             # int32 [2] on the device: {survivors, candidates}
    capacity: int
    layout: str | None
    patch: int
    stride: int
    level: int
    seq: int = 0                    # position in this thread's sequence of scans (the pinned count buffer is shared)

    def resolve(self) -> "PatchBatch":
        l = _lib.lib()
        if self.seq == getattr(_count_host, "seq", 0):
            # fast path: this is the thread's most recent scan, its count is (or will be) in the pinned buffer
            _lib.check(l.hipac_tile_scan_wait_count(), "hipac_tile_scan_wait_count")
            h = _pinned_count()
            n, n_c = int(h[0]), int(h[1])
        else:
            # a later scan has reused the pinned buffer: read this scan's own device counter (synchronises)
            n, n_c = (int(v) for v in self.count.cpu().tolist())
        if n > self.capacity:
            raise RuntimeError(f"{n} survivors exceed capacity {self.capacity}; pass a smaller row_range or a larger capacity")
        return PatchBatch(coords=self.coords[:n], labels=self.labels[:n],
                          batch=self.batch[:n] if self.batch is not None else None,
                          images_u8=self.images_u8[:n] if self.images_u8 is not None else None, layout=self.layout,
                          candidates=n_c, patch=self.patch, stride=self.stride, level=self.level)


def alloc_level_image(height: int, width: int, device, channels: int = 3) -> torch.Tensor:
    """uint8 ``[H, W, 3]`` (``channels=3``) or ``[H, W]`` (``channels=1``, lesion mask) device tensor whose row pitch is a
    multiple of 16 bytes -- what the read-once TMA streaming pass of ``hipac_tile_scan`` needs (``3 * W`` usually is
    not).  A view of a ``[H, pitch]`` buffer; index / slice it like any tensor."""
    pitch = (width * channels + 15) // 16 * 16
    buf = torch.empty((height, pitch), dtype=torch.uint8, device=device)
    if channels == 1:
        return buf[:, :width]
    return buf.as_strided((height, width, channels), (pitch, channels, 1))


def upload_level_rows(dst: torch.Tensor, src_host, r0: int = 0, stream: torch.cuda.Stream | None = None) -> int:
    """Copy host rows ``src_host`` (``uint8 [n, W, 3]`` or ``[n, W]``, numpy or CPU tensor, row-contiguous) into rows
    ``[r0, r0 + n)`` of a (possibly pitched) device image with ONE 2-D DMA (``hipac_upload_rows``); asynchronous when
    the host memory is pinned.  Returns the number of payload bytes."""
    src = torch.as_tensor(src_host)
    if src.dtype != torch.uint8 or src.is_cuda:
        raise ValueError("src_host must be uint8 host memory")
    n = int(src.shape[0])
    if n == 0:
        return 0
    row_bytes = int(src[0].numel())
    if src.dim() >= 2 and src[0].numel() and not src[0].is_contiguous():
        src = src.contiguous()
    view = dst[r0:r0 + n]
    if int(view.shape[0]) != n or int(view[0].numel()) != row_bytes:
        raise ValueError(f"rows [{r0}, {r0 + n}) x {row_bytes} bytes do not fit the destination {tuple(dst.shape)}")
    st = stream or torch.cuda.current_stream(dst.device)
    with torch.cuda.device(dst.device):
        _lib.check(_lib.lib().hipac_upload_rows(view.data_ptr(), int(dst.stride(0)), src.data_ptr(), int(src.stride(0)) if n > 1 else row_bytes,
                                                row_bytes, n, st.cuda_stream), "hipac_upload_rows")
    return row_bytes * n


def _pitched16(t: torch.Tensor, channels: int) -> torch.Tensor:
    """``t`` itself when its rows already start on 16-byte boundaries, else a device-side copy into a pitched buffer (one
    extra read + write of the image: callers that own the upload should use ``alloc_level_image`` instead)."""
    if int(t.stride(0)) % 16 == 0 and t.data_ptr() % 16 == 0:
        return t
    out = alloc_level_image(int(t.shape[0]), int(t.shape[1]), t.device, channels)
    out.copy_(t)
    return out


def batch_shape(n: int, layout: str):
    return (n, OUT, OUT, 3) if layout == "nhwc3" else (n, OUT // 2, S2D16_WIDTH, 16)


def extract_patches_tensor(level_img: torch.Tensor, lesion_mask: torch.Tensor | None, level: int,
                           stride=None, row_range=None, patch_size: int = 224, layout: str | None = "s2d16",
                           want_u8: bool = False, mode: str = "auto", capacity: int | None = None,
                           stream: torch.cuda.Stream | None = None, keep_all: bool = False, tissue: torch.Tensor | None = None,
                           tissue_scale: int = 1, min_tissue=0.5, roi=None, roi_y_origin: int = 0, stain=None) -> PatchBatch:
    """``extract_patches_enqueue(...).resolve()``: see there."""
    return extract_patches_enqueue(level_img, lesion_mask, level, stride=stride, row_range=row_range, patch_size=patch_size,
                                   layout=layout, want_u8=want_u8, mode=mode, capacity=capacity, stream=stream,
                                   keep_all=keep_all, tissue=tissue, tissue_scale=tissue_scale, min_tissue=min_tissue,
                                   roi=roi, roi_y_origin=roi_y_origin, stain=stain).resolve()


def extract_patches_enqueue(level_img: torch.Tensor, lesion_mask: torch.Tensor | None, level: int,
                            stride=None, row_range=None, patch_size: int = 224, layout: str | None = "s2d16",
                            want_u8: bool = False, mode: str = "auto", capacity: int | None = None,
                            stream: torch.cuda.Stream | None = None, keep_all: bool = False, tissue: torch.Tensor | None = None,
                            tissue_scale: int = 1, min_tissue=0.5, roi=None, roi_y_origin: int = 0,
                            stain=None) -> PendingPatchBatch:
    """Tile one level image (uint8 ``[H,W,3]`` on a CUDA device) exactly as the reference does.

    ``lesion_mask``: uint8 ``[H,W]`` (>0 = lesion, the rasterised ``parse_xml_mask`` output,
    reference ``src/main.py:372-410``) or ``None`` -> every patch "normal" (``src/main.py:714-716``).
    ``row_range=(i0,i1)`` restricts to candidate grid rows ``y//stride in [i0,i1)`` -- the
    multi-GPU shard unit.  ``keep_all`` disables the tissue rejection (used on stacks of already
    extracted patches).

    ``tissue``: a tissue mask (uint8 ``[h, w]`` CUDA tensor, > 0 = tissue, e.g. ``tissue.segment_tissue`` of a coarser
    level) at ``tissue_scale`` m in {1, 2, 4, 8, 16, 32}: mask pixel ``(u, v)`` covers level pixels ``[u*m, u*m+m) x
    [v*m, v*m+m)`` of ``level_img``.  A candidate then survives iff at least ``ceil(min_tissue * (P/m)^2)`` mask pixels of
    its footprint are tissue (mask pixels beyond the mask count as background), instead of the reference's ``mean > 240``
    rule; ``keep_all`` still overrides.

    ``roi``: a ``cascade.RoiGrid`` of a coarser level (the coarse-to-fine cascade).  After the ``mean > 240`` or tissue-mask
    rule, a candidate survives only if its footprint overlaps with positive area the footprint of a set ROI cell, both taken
    at this level's resolution.  ``roi_y_origin`` is the level row of ``level_img``'s row 0 (a shard's slab).  Cannot be
    combined with ``keep_all``.

    ``stain``: a ``preprocessing.StainNormalizer`` (Macenko).  The survivors' resized uint8 patches are normalised
    (``hipac_stain_apply``) before ToTensor/Normalize: ``batch`` and ``images_u8`` hold the normalised patches.  Grid,
    tissue test, ROI, labels and survivor order are decided on the raw pixels and do not change.

    Nothing blocks: the call returns capacity-sized tensors and the device-side survivor counter; ``resolve()`` waits only
    until the count is known (after the compaction kernel) and slices, and ``features.classify_tensor(...,
    count=pending.count)`` consumes the batch without any host round trip.
    """
    l = _lib.lib()
    if not (level_img.is_cuda and level_img.dtype == torch.uint8 and level_img.dim() == 3 and level_img.shape[2] == 3):
        raise ValueError("level_img must be a CUDA uint8 tensor of shape [H, W, 3]")
    if level_img.stride(2) != 1 or level_img.stride(1) != 3:
        level_img = level_img.contiguous()
    H, W = int(level_img.shape[0]), int(level_img.shape[1])
    pitch = int(level_img.stride(0))
    if lesion_mask is not None:
        if not (lesion_mask.is_cuda and lesion_mask.dtype == torch.uint8 and tuple(lesion_mask.shape) == (H, W)):
            raise ValueError("lesion_mask must be a CUDA uint8 tensor of shape [H, W]")
        if lesion_mask.stride(1) != 1:
            lesion_mask = lesion_mask.contiguous()
    P, S = patch_and_stride(level, stride, patch_size)
    if roi is not None:
        if keep_all:
            raise ValueError("keep_all cannot be combined with an ROI")
        if roi.level <= level:
            raise ValueError(f"the ROI of level {roi.level} must come from a level coarser than {level}")
        if not (roi.grid.is_cuda and roi.grid.device == level_img.device and roi.grid.dtype == torch.uint8
                and tuple(roi.grid.shape) == (roi.ny, roi.nx) and roi.grid.is_contiguous()):
            raise ValueError("roi.grid must be a contiguous uint8 [ny, nx] tensor on the level image's device")
        if int(roi_y_origin) < 0:
            raise ValueError("roi_y_origin must be >= 0")
    if stain is not None and stain.device != level_img.device:
        raise ValueError("the stain normaliser lives on another device than the level image")
    if tissue is not None:
        if not (tissue.is_cuda and tissue.dtype == torch.uint8 and tissue.dim() == 2 and tissue.device == level_img.device):
            raise ValueError("tissue must be a uint8 [h, w] tensor on the level image's device")
        if tissue_scale not in (1, 2, 4, 8, 16, 32) or S % tissue_scale or P % tissue_scale:
            raise ValueError(f"tissue_scale {tissue_scale} must be a power of two up to 32 dividing the stride {S} and patch {P}")
        if not 0 <= min_tissue <= 1:
            raise ValueError("min_tissue must be a fraction in [0, 1]")
        if tissue.stride(1) != 1:
            tissue = tissue.contiguous()
        min_pixels = math.ceil(Fraction(min_tissue) * (P // tissue_scale) ** 2)
    if P > OUT and mode != "direct":
        # the read-once streaming pass wants 16-byte aligned rows; anything else would silently take the two-pass kernels
        with torch.cuda.device(level_img.device), torch.cuda.stream(stream or torch.cuda.current_stream(level_img.device)):
            level_img = _pitched16(level_img, 3)
            if lesion_mask is not None:
                lesion_mask = _pitched16(lesion_mask, 1)
        pitch = int(level_img.stride(0))
    nx, ny_all = grid_shape(W, H, S)
    i0, i1 = (0, ny_all) if row_range is None else (int(row_range[0]), int(row_range[1]))
    if not (0 <= i0 <= i1 <= ny_all):
        raise ValueError(f"row_range {row_range} outside the candidate grid rows [0, {ny_all}]")
    n_cand = nx * (i1 - i0)
    cap = n_cand if capacity is None else int(capacity)
    dev = level_img.device
    st = stream or torch.cuda.current_stream(dev)
    with torch.cuda.device(dev), torch.cuda.stream(st):
        coords = torch.empty((max(cap, 1), 2), dtype=torch.int32, device=dev)
        labels = torch.empty((max(cap, 1),), dtype=torch.uint8, device=dev)
        count = torch.zeros((2,), dtype=torch.int32, device=dev)
        batch = torch.empty(batch_shape(max(cap, 1), layout), dtype=torch.bfloat16, device=dev) if layout else None
        u8 = torch.empty((max(cap, 1), OUT, OUT, 3), dtype=torch.uint8, device=dev) if want_u8 else None
        # with a normaliser stage 1 writes only the uint8 patches (into a scratch buffer unless they are wanted) and the
        # apply kernel writes the batch from them
        scan_u8 = u8 if stain is None or want_u8 else torch.empty((max(cap, 1), OUT, OUT, 3), dtype=torch.uint8, device=dev)
        scan_batch = batch if stain is None else None
        m = _MODES[mode] | (_lib.SCAN_KEEP_ALL if keep_all else 0)
        if roi is not None:
            ws_bytes = l.hipac_tile_scan_roi_workspace_bytes(H, W, P, S, i0, i1, m, tissue_scale if tissue is not None else 0)
        elif tissue is None:
            ws_bytes = l.hipac_tile_scan_workspace_bytes(H, W, P, S, i0, i1, m)
        else:
            ws_bytes = l.hipac_tile_scan_tissue_workspace_bytes(H, W, P, S, i0, i1, m, tissue_scale)
        if ws_bytes == 0:
            raise RuntimeError("hipac_tile_scan_workspace_bytes: " + l.hipac_last_error().decode())
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        h_count = _pinned_count()
        args = (level_img.data_ptr(), H, W, pitch,
                lesion_mask.data_ptr() if lesion_mask is not None else None,
                int(lesion_mask.stride(0)) if lesion_mask is not None else 0,
                P, S, i0, i1, coords.data_ptr(), labels.data_ptr(),
                scan_u8.data_ptr() if scan_u8 is not None else None,
                scan_batch.data_ptr() if scan_batch is not None else None, _LAYOUTS[layout] if scan_batch is not None else 0,
                count.data_ptr(), cap, ws.data_ptr(), ws_bytes, m)
        if tissue is not None:
            th, tw = int(tissue.shape[0]), int(tissue.shape[1])
            tis = (tissue.data_ptr() if th * tw else None, th, tw, int(tissue.stride(0)), tissue_scale, min_pixels)
        if roi is not None:
            _lib.check(l.hipac_tile_scan_roi(*args, *(tis if tissue is not None else (None, 0, 0, 0, 0, 0)), roi.grid.data_ptr(),
                                             roi.nx, roi.ny, roi.level - level, roi.stride, roi.patch, int(roi_y_origin),
                                             st.cuda_stream), "hipac_tile_scan_roi")
        elif tissue is None:
            _lib.check(l.hipac_tile_scan(*args, st.cuda_stream), "hipac_tile_scan")
        else:
            _lib.check(l.hipac_tile_scan_tissue(*args, *tis, st.cuda_stream), "hipac_tile_scan_tissue")
        ws.record_stream(st)
        if stain is not None and (batch is not None or want_u8):
            stain.apply(scan_u8, layout, count=count, out_u8=u8, out=batch, stream=st)
            scan_u8.record_stream(st)
    del h_count   # registered with the library; read in resolve()
    _count_host.seq = getattr(_count_host, "seq", 0) + 1
    return PendingPatchBatch(coords=coords, labels=labels, batch=batch, images_u8=u8, count=count, capacity=cap,
                             layout=layout, patch=P, stride=S, level=level, seq=_count_host.seq)
