"""Tensor-level ResNet18 feature extraction / classification on the CUDA path.

Replaces the model forward of the reference's ``extract_features`` hot loop
(``src/main.py:867-871``: ``feats = model(imgs.to(device))``) and the classifier forward of
``evaluate_resnet_classifier`` (``src/main.py:1004-1009``).  Weights come from a torchvision
``resnet18`` module / state dict (the reference's wrappers in ``src/models/resnet.py`` are thin
shells around exactly that); eval-mode BatchNorm is folded in ``hipac_resnet18_pack``.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib

_BLOCKS = [("layer1", 0, False), ("layer1", 1, False), ("layer2", 0, True), ("layer2", 1, False),
           ("layer3", 0, True), ("layer3", 1, False), ("layer4", 0, True), ("layer4", 1, False)]


def conv_bn_names():
    """(conv, bn) module-name pairs in the C ABI's layer order (torchvision state-dict order)."""
    names = [("conv1", "bn1")]
    for layer, blk, ds in _BLOCKS:
        p = f"{layer}.{blk}"
        names += [(f"{p}.conv1", f"{p}.bn1"), (f"{p}.conv2", f"{p}.bn2")]
        if ds:
            names.append((f"{p}.downsample.0", f"{p}.downsample.1"))
    return names


class PackedResNet18:
    """Folded + re-laid-out weights resident on one device."""

    def __init__(self, blob: torch.Tensor, num_classes: int):
        self.blob = blob
        self.num_classes = num_classes

    @property
    def device(self):
        return self.blob.device


def pack_resnet18(state_dict: dict, device, prefix: str = "", bn_eps: float = 1e-5) -> PackedResNet18:
    """Pack a torchvision-style resnet18 state dict (keys ``{prefix}conv1.weight`` ...).

    A present ``{prefix}fc.weight`` of shape ``[k,512]`` becomes the classifier head."""
    l = _lib.lib()
    tensors = []
    for conv, bn in conv_bn_names():
        for key in (f"{conv}.weight", f"{bn}.weight", f"{bn}.bias", f"{bn}.running_mean", f"{bn}.running_var"):
            tensors.append(state_dict[prefix + key].detach().to("cpu", torch.float32).contiguous())
    fcw = state_dict.get(prefix + "fc.weight")
    num_classes = 0
    if fcw is not None and fcw.dim() == 2 and fcw.shape[1] == 512:
        num_classes = int(fcw.shape[0])
        tensors.append(fcw.detach().to("cpu", torch.float32).contiguous())
        tensors.append(state_dict[prefix + "fc.bias"].detach().to("cpu", torch.float32).contiguous())
    ptrs = (C.c_void_p * 102)(*([t.data_ptr() for t in tensors] + [None] * (102 - len(tensors))))
    nbytes = l.hipac_resnet18_packed_bytes(num_classes)
    host = np.zeros(nbytes, dtype=np.uint8)
    _lib.check(l.hipac_resnet18_pack(ptrs, 102, num_classes, bn_eps, host.ctypes.data_as(C.c_void_p), nbytes),
               "hipac_resnet18_pack")
    return PackedResNet18(torch.from_numpy(host).to(device), num_classes)


_LAYOUT_BY_SHAPE = {(224, 224, 3): _lib.LAYOUT_NHWC3_BF16, (112, 115, 16): _lib.LAYOUT_S2D16_BF16}


def _forward(batch: torch.Tensor, packed: PackedResNet18, want_logits: bool, chunk: int, stream=None,
             count: torch.Tensor | None = None, tta: bool = False):
    """``count``: int32 device tensor whose element 0 is the number of valid patches in ``batch`` (device-count mode:
    ``batch.shape[0]`` is only the capacity; nothing here waits for the value).  ``tta``: the D4 test-time augmentation
    (``hipac_resnet18_forward_d4``)."""
    l = _lib.lib()
    if not (batch.is_cuda and batch.dtype == torch.bfloat16 and batch.dim() == 4 and tuple(batch.shape[1:]) in _LAYOUT_BY_SHAPE):
        raise ValueError("batch must be a CUDA bf16 tensor [N,224,224,3] or [N,112,115,16]")
    if batch.device != packed.device:
        raise ValueError("batch and packed weights live on different devices")
    if want_logits and packed.num_classes == 0:
        raise ValueError("packed weights have no classifier head")
    batch = batch.contiguous()
    n = int(batch.shape[0])
    dev = batch.device
    st = stream or torch.cuda.current_stream(dev)
    with torch.cuda.device(dev), torch.cuda.stream(st):
        feats = torch.empty((n, 512), dtype=torch.float32, device=dev)
        logits = torch.empty((n, packed.num_classes), dtype=torch.float32, device=dev) if want_logits else None
        if n == 0:
            return feats, logits
        ws_bytes = l.hipac_resnet18_workspace_bytes(n, chunk)
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        if count is not None and not (count.is_cuda and count.dtype == torch.int32 and count.numel() >= 1):
            raise ValueError("count must be a CUDA int32 tensor")
        if tta:
            rc = l.hipac_resnet18_forward_d4(packed.blob.data_ptr(), packed.num_classes, batch.data_ptr(),
                                             _LAYOUT_BY_SHAPE[tuple(batch.shape[1:])], n,
                                             count.data_ptr() if count is not None else None, feats.data_ptr(),
                                             logits.data_ptr() if logits is not None else None, ws.data_ptr(), ws_bytes,
                                             chunk, st.cuda_stream)
        elif count is None:
            rc = l.hipac_resnet18_forward(packed.blob.data_ptr(), packed.num_classes, batch.data_ptr(),
                                          _LAYOUT_BY_SHAPE[tuple(batch.shape[1:])], n, feats.data_ptr(),
                                          logits.data_ptr() if logits is not None else None, ws.data_ptr(), ws_bytes,
                                          chunk, st.cuda_stream)
        else:
            rc = l.hipac_resnet18_forward_dcount(packed.blob.data_ptr(), packed.num_classes, batch.data_ptr(),
                                                 _LAYOUT_BY_SHAPE[tuple(batch.shape[1:])], n, count.data_ptr(),
                                                 feats.data_ptr(), logits.data_ptr() if logits is not None else None,
                                                 ws.data_ptr(), ws_bytes, chunk, st.cuda_stream)
        _lib.check(rc, "hipac_resnet18_forward")
        ws.record_stream(st)
    return feats, logits


def extract_features_tensor(batch: torch.Tensor, packed: PackedResNet18, chunk: int = 4096, stream=None,
                            count: torch.Tensor | None = None, *, tta: bool = False) -> torch.Tensor:
    """float32 ``[N,512]`` pooled trunk features of a bf16 patch batch (asynchronous).

    ``tta=True``: rotation/flip test-time augmentation.  Each patch's features are the mean of the features of its eight
    views under the dihedral group D4 (``d4_view``), summed in fp32 in view order 0..7 and multiplied by 0.125, so they do
    not depend on the patch's orientation.  Costs eight forwards."""
    return _forward(batch, packed, False, chunk, stream, count, tta)[0]


def classify_tensor(batch: torch.Tensor, packed: PackedResNet18, chunk: int = 4096, stream=None,
                    count: torch.Tensor | None = None, *, tta: bool = False):
    """(features float32 ``[N,512]``, logits float32 ``[N,k]``) of a bf16 patch batch (asynchronous).  ``tta=True``: the
    features of ``extract_features_tensor(..., tta=True)`` and the head applied to them (which, the head being affine,
    is the mean of the eight views' logits up to rounding)."""
    return _forward(batch, packed, True, chunk, stream, count, tta)


def d4_view(batch: torch.Tensor, view: int, *, count: torch.Tensor | None = None, base: int = 0,
            out: torch.Tensor | None = None) -> torch.Tensor:
    """View ``view`` = 4 f + k (0..7) of a bf16 patch batch (``[N,224,224,3]`` or ``[N,112,115,16]``) under the dihedral
    group D4, as the S2D16 batch ``[N,112,115,16]`` the network reads: the S2D16 form of
    ``torch.rot90(torch.flip(x, dims=[2]) if f else x, k, dims=(1, 2))`` for the NHWC image ``x``.  The padding columns and
    channels 12..15 of the output are zero.  ``count`` / ``base`` / ``out``: device-count mode and in-place output as for
    ``conv_layer``."""
    if not (batch.is_cuda and batch.dtype == torch.bfloat16 and batch.dim() == 4 and tuple(batch.shape[1:]) in _LAYOUT_BY_SHAPE):
        raise ValueError("batch must be a CUDA bf16 tensor [N,224,224,3] or [N,112,115,16]")
    l = _lib.lib()
    batch = batch.contiguous()
    n = int(batch.shape[0])
    out = _hook_out(out, (n, 112, 115, 16), batch.device)
    d_count, n_base = _launch_state(count, base)
    rc = l.hipac_batch_d4_view(batch.data_ptr(), _LAYOUT_BY_SHAPE[tuple(batch.shape[1:])], n, int(view), out.data_ptr(),
                               d_count, n_base, torch.cuda.current_stream(batch.device).cuda_stream)
    _lib.check(rc, "hipac_batch_d4_view")
    return out


def _launch_state(count: torch.Tensor | None, base: int):
    """The trailing (d_count, n_base) arguments of the test hooks: host count when ``count`` is None."""
    if count is None:
        return None, int(base)
    if not (count.is_cuda and count.dtype == torch.int32 and count.numel() >= 1):
        raise ValueError("count must be a CUDA int32 tensor")
    return count.data_ptr(), int(base)


def _hook_out(out: torch.Tensor | None, shape, device) -> torch.Tensor:
    if out is None:
        return torch.empty(shape, dtype=torch.bfloat16, device=device)
    if not (out.dtype == torch.bfloat16 and tuple(out.shape) == tuple(shape) and out.is_contiguous() and out.device == device):
        raise ValueError(f"out must be a contiguous bf16 tensor of shape {tuple(shape)} on {device}")
    return out


def conv_layer(packed: PackedResNet18, layer: int, x: torch.Tensor, residual: torch.Tensor | None, relu: bool, *,
               reverse: bool = False, count: torch.Tensor | None = None, base: int = 0, out: torch.Tensor | None = None):
    """Test hook: run one conv(+folded BN)(+residual)(+ReLU) layer on bf16 NHWC input.  Layers 0 and 7 exist only fused
    (``stem``, ``conv_ds_fused``): the library refuses them, and out-of-range indices, with a RuntimeError.

    The keywords give the kernel the launch state the forward uses: ``reverse`` walks the tiles from the last to the
    first; ``count`` (int32 device tensor) switches to device-count mode, where the kernel works on
    ``clamp(count[0] - base, 0, n)`` patches and leaves the other rows of ``out`` untouched; ``out`` is written in
    place instead of a fresh tensor."""
    l = _lib.lib()
    cout_hout = {**{i: (64, 56) for i in range(1, 5)}, **{i: (128, 28) for i in range(5, 10)},
                 **{i: (256, 14) for i in range(10, 15)}, **{i: (512, 7) for i in range(15, 20)}}
    cout, hout = cout_hout.get(layer, (1, 1))   # placeholder output for a layer the library refuses
    n = int(x.shape[0])
    out = _hook_out(out, (n, hout, hout, cout), x.device)
    d_count, n_base = _launch_state(count, base)
    st = torch.cuda.current_stream(x.device)
    rc = l.hipac_resnet18_conv_layer(packed.blob.data_ptr(), packed.num_classes, layer, x.contiguous().data_ptr(),
                                     residual.contiguous().data_ptr() if residual is not None else None,
                                     out.data_ptr(), n, int(relu), st.cuda_stream, int(reverse), d_count, n_base)
    _lib.check(rc, "hipac_resnet18_conv_layer")
    return out


def stem(packed: PackedResNet18, x: torch.Tensor, *, reverse: bool = False, count: torch.Tensor | None = None, base: int = 0,
         out: torch.Tensor | None = None) -> torch.Tensor:
    """Test hook: fused conv1 + BN + ReLU + max pool on an S2D16 batch -> bf16 ``[n,56,56,64]`` (keywords: ``conv_layer``)."""
    l = _lib.lib()
    n = int(x.shape[0])
    out = _hook_out(out, (n, 56, 56, 64), x.device)
    d_count, n_base = _launch_state(count, base)
    rc = l.hipac_resnet18_stem(packed.blob.data_ptr(), packed.num_classes, x.contiguous().data_ptr(), out.data_ptr(), n,
                               torch.cuda.current_stream(x.device).cuda_stream, int(reverse), d_count, n_base)
    _lib.check(rc, "hipac_resnet18_stem")
    return out


def conv_ds_fused(packed: PackedResNet18, stage: int, x: torch.Tensor, block_in: torch.Tensor, *, reverse: bool = False,
                  count: torch.Tensor | None = None, base: int = 0, out: torch.Tensor | None = None) -> torch.Tensor:
    """Test hook: conv2 of layer{2,3,4}.0 + fused 1x1/s2 projection shortcut + ReLU (stage 0/1/2; keywords: ``conv_layer``)."""
    l = _lib.lib()
    n, cout, hout = int(x.shape[0]), (128, 256, 512)[stage], (28, 14, 7)[stage]
    out = _hook_out(out, (n, hout, hout, cout), x.device)
    d_count, n_base = _launch_state(count, base)
    rc = l.hipac_resnet18_conv_ds_fused(packed.blob.data_ptr(), packed.num_classes, stage, x.contiguous().data_ptr(),
                                        block_in.contiguous().data_ptr(), out.data_ptr(), n,
                                        torch.cuda.current_stream(x.device).cuda_stream, int(reverse), d_count, n_base)
    _lib.check(rc, "hipac_resnet18_conv_ds_fused")
    return out
