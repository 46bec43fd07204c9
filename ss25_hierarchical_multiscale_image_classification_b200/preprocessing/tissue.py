"""Tissue segmentation on the GPU: the CLAM-style background rejection of CAMELYON16 pipelines.

``segment_tissue`` thresholds the HSV saturation of a low-resolution level (a "thumbnail") after a median blur, exactly as
``cv2.cvtColor(RGB2HSV)`` -> ``cv2.medianBlur(S, ksize)`` -> ``cv2.threshold(BINARY | OTSU)`` (or a fixed threshold) do in
OpenCV 4.13, bit for bit (``hipac_tissue_segment``, ``csrc/tissue.cu``).  Its mask is what ``extract_patches_tensor(...,
tissue=mask, tissue_scale=m)`` and ``pipeline.process_level(..., tissue=mask, tissue_scale=m)`` filter the candidates of a
finer level with: segment coarse, tile fine.
"""
from __future__ import annotations

import torch

from .. import _lib


def segment_tissue(img: torch.Tensor, ksize: int = 7, threshold: int | None = None, stream: torch.cuda.Stream | None = None,
                   with_blur: bool = False):
    """Tissue mask of a CUDA uint8 ``[H, W, 3]`` image (any row pitch).

    Returns ``(mask, t)``: uint8 ``[H, W]`` CUDA tensor of 0 / 255 and the threshold used as a CUDA int32 ``[1]`` tensor
    (Otsu's value when ``threshold`` is ``None``).  ``with_blur`` also returns the median-blurred saturation plane.
    Nothing waits on the host."""
    if not (img.is_cuda and img.dtype == torch.uint8 and img.dim() == 3 and img.shape[2] == 3):
        raise ValueError("img must be a CUDA uint8 tensor of shape [H, W, 3]")
    if ksize not in (1, 3, 5, 7):
        raise ValueError("ksize must be 1, 3, 5 or 7")
    if threshold is not None and not 0 <= int(threshold) <= 255:
        raise ValueError("threshold must be None (Otsu) or in [0, 255]")
    if img.stride(2) != 1 or img.stride(1) != 3:
        img = img.contiguous()
    H, W = int(img.shape[0]), int(img.shape[1])
    l = _lib.lib()
    dev = img.device
    st = stream or torch.cuda.current_stream(dev)
    with torch.cuda.device(dev), torch.cuda.stream(st):
        mask = torch.empty((H, W), dtype=torch.uint8, device=dev)
        t = torch.empty((1,), dtype=torch.int32, device=dev)
        blur = torch.empty((H, W), dtype=torch.uint8, device=dev) if with_blur else None
        ws_bytes = l.hipac_tissue_workspace_bytes(H, W)
        if ws_bytes == 0:
            raise RuntimeError("hipac_tissue_workspace_bytes: " + l.hipac_last_error().decode())
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        _lib.check(l.hipac_tissue_segment(img.data_ptr(), H, W, int(img.stride(0)), int(ksize),
                                          -1 if threshold is None else int(threshold), mask.data_ptr(), W, t.data_ptr(),
                                          blur.data_ptr() if blur is not None else None, W, ws.data_ptr(), ws_bytes,
                                          st.cuda_stream), "hipac_tissue_segment")
        ws.record_stream(st)
    return (mask, t, blur) if with_blur else (mask, t)
