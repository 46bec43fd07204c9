"""Patch extraction (the reference's ``src/preprocessing`` / ``extract_patches`` home)."""
from .extract import extract_patches, extract_patches_per_slide, parse_xml_mask, scan_slide  # noqa: F401
from .tensor_api import (PatchBatch, PendingPatchBatch, alloc_level_image, extract_patches_enqueue,  # noqa: F401
                         extract_patches_tensor, grid_shape, patch_and_stride, upload_level_rows)
from .tissue import segment_tissue  # noqa: F401
from .stain import Stain, StainNormalizer, estimate_stain  # noqa: F401
