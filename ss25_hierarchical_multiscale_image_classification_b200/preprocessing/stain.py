"""Macenko stain normalisation on the GPU: the colour standardisation of CAMELYON16 pipelines.

CAMELYON16 slides come from two centres whose H&E staining differs visibly.  ``estimate_stain`` finds a slide's
haematoxylin and eosin optical-density vectors and its stain concentration scale from a thumbnail, exactly as torchstain's
``NumpyMacenkoNormalizer`` (``Io = 240``, ``alpha = 1``, ``beta = 0.15``) does, up to fp64 rounding
(``hipac_stain_estimate``, ``csrc/stain.cu``).  ``StainNormalizer`` re-expresses every pixel of a patch batch in a
reference stain (torchstain's by default): the uint8 result equals torchstain's ``normalize`` with the slide's matrix, and
the bf16 batch is stage 1's ToTensor/Normalize of it (``hipac_stain_apply``).  ``extract_patches_tensor(..., stain=)``,
``pipeline.process_level(..., stain=)`` and ``cascade.process_cascade(..., stain=)`` run it on every survivor.
Nothing here waits on the host except ``Stain.valid()``.
"""
from __future__ import annotations

import numpy as np
import torch

from .. import _lib

_LAYOUTS = {"nhwc3": _lib.LAYOUT_NHWC3_BF16, "s2d16": _lib.LAYOUT_S2D16_BF16}
HE_REF = ((0.5626, 0.2159), (0.7201, 0.8012), (0.4062, 0.5581))   # torchstain's target
MAXC_REF = (1.9705, 1.0308)


class Stain:
    """A stain block on the device: fp64 ``[16]`` = HE row-major ``[3][2]`` (haematoxylin, eosin columns), maxC ``[2]``,
    valid, n_hat (include/hipac_b200.h)."""

    def __init__(self, block: torch.Tensor):
        if not (block.is_cuda and block.dtype == torch.float64 and block.shape == (_lib.STAIN_BLOCK_DOUBLES,) and block.is_contiguous()):
            raise ValueError(f"a stain block is a contiguous CUDA float64 [{_lib.STAIN_BLOCK_DOUBLES}] tensor")
        self.block = block

    @property
    def he(self) -> torch.Tensor:
        return self.block[:6].view(3, 2)

    @property
    def max_c(self) -> torch.Tensor:
        return self.block[6:8]

    @property
    def n_hat(self) -> torch.Tensor:
        return self.block[9]

    def valid(self) -> bool:
        """Whether the estimate succeeded (at least two stained pixels, a non-singular matrix, a positive scale).  Waits
        for the block."""
        return bool(self.block[8].item() != 0)

    @property
    def device(self):
        return self.block.device

    @staticmethod
    def from_matrix(he, max_c, device) -> "Stain":
        """A valid block holding a given ``he`` [3, 2] and ``max_c`` [2]."""
        he, max_c = np.asarray(he, dtype=np.float64), np.asarray(max_c, dtype=np.float64)
        if he.shape != (3, 2) or max_c.shape != (2,):
            raise ValueError("he must be [3, 2] and max_c [2]")
        b = np.zeros(_lib.STAIN_BLOCK_DOUBLES)
        b[:6], b[6:8], b[8] = he.reshape(-1), max_c, 1.0
        return Stain(torch.from_numpy(b).to(device))

    @staticmethod
    def reference(device) -> "Stain":
        """torchstain's target stain."""
        return Stain.from_matrix(HE_REF, MAXC_REF, device)


def estimate_stain(rgb: torch.Tensor, io: int = 240, alpha: float = 1.0, beta: float = 0.15,
                   stream: torch.cuda.Stream | None = None) -> Stain:
    """The Macenko stain of a CUDA uint8 ``[H, W, 3]`` image (any row pitch), e.g. a slide thumbnail.  Asynchronous; the
    result is the same bits on every run and every device."""
    if not (rgb.is_cuda and rgb.dtype == torch.uint8 and rgb.dim() == 3 and rgb.shape[2] == 3):
        raise ValueError("rgb must be a CUDA uint8 tensor of shape [H, W, 3]")
    if rgb.stride(2) != 1 or rgb.stride(1) != 3:
        rgb = rgb.contiguous()
    H, W = int(rgb.shape[0]), int(rgb.shape[1])
    l = _lib.lib()
    dev = rgb.device
    st = stream or torch.cuda.current_stream(dev)
    with torch.cuda.device(dev), torch.cuda.stream(st):
        ws_bytes = l.hipac_stain_workspace_bytes(H, W)
        if ws_bytes == 0:
            raise ValueError("hipac_stain_workspace_bytes: " + l.hipac_last_error().decode())
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        block = torch.empty((_lib.STAIN_BLOCK_DOUBLES,), dtype=torch.float64, device=dev)
        _lib.check(l.hipac_stain_estimate(rgb.data_ptr(), H, W, int(rgb.stride(0)), int(io), float(alpha), float(beta),
                                          block.data_ptr(), ws.data_ptr(), ws_bytes, st.cuda_stream), "hipac_stain_estimate")
        ws.record_stream(st)
    return Stain(block)


class StainNormalizer:
    """Maps the stain ``source`` (a slide's ``estimate_stain``) to ``target`` (default: torchstain's reference).  With an
    invalid source or target the normaliser passes pixels through unchanged."""

    def __init__(self, source: Stain, target: Stain | None = None, io: int = 240):
        if target is not None and target.device != source.device:
            raise ValueError("source and target stains live on different devices")
        l = _lib.lib()
        dev = source.device
        with torch.cuda.device(dev):
            self.params = torch.empty((_lib.STAIN_PARAMS_DOUBLES,), dtype=torch.float64, device=dev)
            _lib.check(l.hipac_stain_normalizer(source.block.data_ptr(), target.block.data_ptr() if target is not None else None,
                                                int(io), self.params.data_ptr(), torch.cuda.current_stream(dev).cuda_stream),
                       "hipac_stain_normalizer")
        self.source, self.target, self.io = source, target, int(io)

    @property
    def device(self):
        return self.params.device

    def apply(self, images_u8: torch.Tensor, layout: str | None = "s2d16", count: torch.Tensor | None = None, base: int = 0,
              out_u8: torch.Tensor | None = None, out: torch.Tensor | None = None, stream: torch.cuda.Stream | None = None):
        """Normalise a CUDA uint8 ``[N, 224, 224, 3]`` patch batch.

        ``layout`` "s2d16" / "nhwc3": returns the bf16 batch of the normalised patches (into ``out`` if given), ready for
        ``features.classify_tensor``; ``None``: returns the normalised uint8 patches.  ``out_u8`` also receives the uint8
        patches (``images_u8`` itself for in place).  ``count`` (int32 device tensor): only patches
        ``< clamp(count[0] - base, 0, N)`` are read and written (device-count mode), nothing waits on the host."""
        if not (images_u8.is_cuda and images_u8.dtype == torch.uint8 and images_u8.dim() == 4
                and tuple(images_u8.shape[1:]) == (224, 224, 3) and images_u8.is_contiguous()):
            raise ValueError("images_u8 must be a contiguous CUDA uint8 tensor [N, 224, 224, 3]")
        if images_u8.device != self.device:
            raise ValueError("images and normaliser live on different devices")
        n = int(images_u8.shape[0])
        if layout is not None and layout not in _LAYOUTS:
            raise ValueError(f"layout must be 's2d16', 'nhwc3' or None, got {layout!r}")
        if count is not None and not (count.is_cuda and count.dtype == torch.int32 and count.numel() >= 1):
            raise ValueError("count must be a CUDA int32 tensor")
        dev = images_u8.device
        st = stream or torch.cuda.current_stream(dev)
        with torch.cuda.device(dev), torch.cuda.stream(st):
            if layout is None and out_u8 is None:
                out_u8 = torch.empty_like(images_u8)
            if out_u8 is not None and not (out_u8.dtype == torch.uint8 and out_u8.shape == images_u8.shape
                                           and out_u8.is_contiguous() and out_u8.device == dev):
                raise ValueError("out_u8 must be a contiguous uint8 tensor shaped like images_u8 on its device")
            if layout is not None:
                shape = (n, 224, 224, 3) if layout == "nhwc3" else (n, 112, 115, 16)
                if out is None:
                    out = torch.empty(shape, dtype=torch.bfloat16, device=dev)
                elif not (out.dtype == torch.bfloat16 and tuple(out.shape) == shape and out.is_contiguous() and out.device == dev):
                    raise ValueError(f"out must be a contiguous bf16 tensor of shape {shape} on {dev}")
            if n == 0:
                return out if layout is not None else out_u8
            _lib.check(_lib.lib().hipac_stain_apply(images_u8.data_ptr(), n, count.data_ptr() if count is not None else None,
                                                    int(base), self.params.data_ptr(),
                                                    out_u8.data_ptr() if out_u8 is not None else None,
                                                    out.data_ptr() if layout is not None else None,
                                                    _LAYOUTS[layout] if layout is not None else 0, st.cuda_stream),
                       "hipac_stain_apply")
        return out if layout is not None else out_u8
