"""Drop-in mirrors of the reference's ResNet18 wrappers (``src/models/resnet.py:22-91``).

Same class names, constructor arguments and -- crucially -- the same state-dict key names
(``features.N.*`` for the feature extractor, ``model.*`` for the classifiers, ``encoder.*`` for
the SimCLR variant), so reference checkpoints load unchanged.  The parameters live in ordinary
torchvision modules; ``forward`` on a CUDA tensor does not run them through cuDNN but through the
sm_100a tcgen05 kernels (``hipac_resnet18_forward``), after folding eval-mode BatchNorm.  There is
no fallback: a CPU input raises.

Differences from the reference, on purpose:
  * ``ResNet18Classifier()`` does not download ImageNet weights (``pretrained=True`` at
    ``src/models/resnet.py:63-65`` cannot work offline); it starts from random init like
    ``ResNet18FeatureExtractor`` does when its checkpoint is missing.
  * inference only (eval-mode BatchNorm); training is out of scope (SURVEY.md section 2).
"""
from __future__ import annotations

import os

import torch
import torch.nn as nn
from torchvision import models

from .. import features as _features


class _HipacForwardMixin:
    """Caches the packed weights and routes forward() through the CUDA library."""

    _tv_prefix = ""          # where the torchvision resnet18 keys live inside state_dict()
    _wants_logits = False

    def _tv_state(self):
        raise NotImplementedError

    def _packed(self, device):
        params = list(self.parameters()) + list(self.buffers())
        key = (str(device), tuple(p._version for p in params), tuple(p.data_ptr() for p in params))
        if getattr(self, "_pack_key", None) != key:
            self._pack = _features.pack_resnet18(self._tv_state(), device)
            self._pack_key = key
        return self._pack

    def _run(self, x: torch.Tensor, chunk: int = 4096, tta: bool = False):
        if self.training:
            raise RuntimeError("the B200 path is inference-only: call .eval() first (training is out of scope)")
        if not x.is_cuda:
            raise RuntimeError("the HiPAC B200 path needs a CUDA tensor; there is no CPU fallback")
        if x.dim() == 4 and x.shape[1] == 3 and x.dtype != torch.bfloat16:
            # reference signature: float [B,3,224,224] NCHW, already normalised (src/main.py:815-816)
            x = x.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)
        packed = self._packed(x.device)
        if packed.num_classes > 0 and self._wants_logits:
            return _features.classify_tensor(x, packed, chunk, tta=tta)[1]
        return _features.extract_features_tensor(x, packed, chunk, tta=tta)

    def forward_batch(self, batch: torch.Tensor, chunk: int = 4096, tta: bool = False):
        """Native entry: bf16 ``[N,224,224,3]`` or ``[N,112,115,16]`` batch from ``extract_patches_tensor``.  ``tta=True``:
        the mean over the eight D4 rotations / flips of each patch (``features.extract_features_tensor(..., tta=True)``)."""
        return self._run(batch, chunk, tta)


def _sequential_to_tv(sd: dict, prefix: str = "features.") -> dict:
    """``features.{0,1,4,5,6,7}.*`` (Sequential over resnet.children()[:-1]) -> torchvision names."""
    names = {0: "conv1", 1: "bn1", 4: "layer1", 5: "layer2", 6: "layer3", 7: "layer4"}
    out = {}
    for k, v in sd.items():
        if not k.startswith(prefix):
            continue
        idx, rest = k[len(prefix):].split(".", 1)
        if int(idx) in names:
            out[f"{names[int(idx)]}.{rest}"] = v
    return out


class ResNet18FeatureExtractor(_HipacForwardMixin, nn.Module):
    """512-d trunk features (reference ``src/models/resnet.py:22-40``)."""

    def __init__(self, weight_path="resnet18_patch_classifier.pth"):
        super().__init__()
        resnet = models.resnet18(weights=None)
        weight_path = os.path.join(os.getcwd(), "src", "models", weight_path)
        if weight_path and os.path.exists(weight_path):
            state_dict = torch.load(weight_path, map_location="cpu")
            state_dict = {k: v for k, v in state_dict.items() if "fc" not in k}
            resnet.load_state_dict(state_dict, strict=False)
        else:
            print("[WARNING] Using ImageNet weights (not fine-tuned)")   # reference's (inaccurate) message, kept
        self.features = nn.Sequential(*list(resnet.children())[:-1])
        self.eval()

    def _tv_state(self):
        return _sequential_to_tv(self.state_dict())

    def forward(self, x):
        return self._run(x)


class UnifiedResNet(_HipacForwardMixin, nn.Module):
    """Reference ``src/models/resnet.py:42-55``: ``model.*`` keys, optional 2-class head."""

    def __init__(self, pretrained_weights_path=None, classifier=False):
        super().__init__()
        self.model = models.resnet18(weights=None)
        self.model.fc = nn.Identity()
        if pretrained_weights_path and os.path.exists(pretrained_weights_path):
            state_dict = torch.load(pretrained_weights_path, map_location="cpu")
            state_dict = {k: v for k, v in state_dict.items() if "fc" not in k}
            self.model.load_state_dict(state_dict, strict=False)
        if classifier:
            self.model.fc = nn.Linear(512, 2)
        self._wants_logits = bool(classifier)
        self.eval()

    def _tv_state(self):
        return {k[len("model."):]: v for k, v in self.state_dict().items() if k.startswith("model.")}

    def forward(self, x):
        return self._run(x)


class ResNet18Classifier(_HipacForwardMixin, nn.Module):
    """Binary patch classifier (reference ``src/models/resnet.py:57-77``), ``model.*`` keys."""

    _wants_logits = True

    def __init__(self):
        super().__init__()
        self.model = models.resnet18(weights=None)   # reference asks for pretrained=True (needs network)
        num_ftrs = self.model.fc.in_features
        self.model.fc = nn.Linear(num_ftrs, 2)
        self.eval()

    def _tv_state(self):
        return {k[len("model."):]: v for k, v in self.state_dict().items() if k.startswith("model.")}

    def forward(self, x):
        return self._run(x)


class ResNet18ClassifierSIMCLR(_HipacForwardMixin, nn.Module):
    """Reference ``src/models/resnet.py:80-91``: ``encoder.*`` keys, SimCLR-pretrained trunk + linear head."""

    _wants_logits = True

    def __init__(self, pretrained_weights_path=None, num_classes=2):
        super().__init__()
        self.encoder = models.resnet18(weights=None)
        in_features = self.encoder.fc.in_features
        if pretrained_weights_path:
            state_dict = torch.load(pretrained_weights_path, map_location="cpu")
            self.encoder.fc = nn.Identity()
            self.encoder.load_state_dict(state_dict, strict=False)
        self.encoder.fc = nn.Linear(in_features, num_classes)
        self.eval()

    def _tv_state(self):
        return {k[len("encoder."):]: v for k, v in self.state_dict().items() if k.startswith("encoder.")}

    def forward(self, x):
        return self._run(x)
