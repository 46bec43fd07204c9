"""B200-native HiPAC hot path: multiscale patch extraction + ResNet18 features.

Mirrors the reference's entry points (anacarsi/ss25_Hierarchical_Multiscale_Image_Classification,
``src/main.py`` / ``src/models`` / ``src/datasets``) on top of hand-written sm_100a CUDA kernels
reached through the C ABI in ``include/hipac_b200.h``.
"""
from . import _lib  # noqa: F401
from .cascade import RoiGrid, process_cascade, roi_grid, threshold_of, tumor_margin  # noqa: F401
from .preprocessing.stain import Stain, StainNormalizer, estimate_stain  # noqa: F401

__version__ = "0.1.0"
