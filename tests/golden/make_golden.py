"""Generate tests/golden/*.npz.

    python tests/golden/make_golden.py            # stage-1 and stage-2 fixtures: needs the reference checkout
    python tests/golden/make_golden.py config0    # the configs[0] fixture: needs only this repository

Each stage-1 fixture freezes what the reference's own ``extract_patches``
(src/main.py:609-732) emitted for one synthetic slide / level / stride:
patch coordinates in emission order, labels, a CRC32 of every patch after the
reference's ``transforms.Resize((224,224))`` (src/main.py:814) and a few full
224x224x3 images.  The stage-2 fixture freezes features of the reference's
``ResNet18FeatureExtractor`` (src/models/resnet.py:22-40) fed through its own
transform chain, for seeded weights.

The configs[0] fixture freezes the whole BASELINE configs[0] (see ``config0_case``) as computed by the CPU oracle, whose
stage 1 the fixtures above pin to the reference and whose fp32 ResNet18 is the reference's feature extractor.
"""
from __future__ import annotations

import os
import sys
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import hipac_oracle as orc  # noqa: E402
from oracle import ref_harness as rh  # noqa: E402
from ss25_hierarchical_multiscale_image_classification_b200.synthetic import SyntheticSlide  # noqa: E402
sys.path.insert(0, os.path.dirname(HERE))
from conftest import make_slide  # noqa: E402

# name -> (w0, h0, seed, level, stride, with_mask)
CASES = {
    "l3_default":      (12000, 9000, 1234, 3, None, True),    # P=S=224, ragged border
    "l2_cli_stride":   (12000, 9000, 1234, 2, None, True),    # P=448, S=224 (reference CLI semantics)
    "l2_nonoverlap":   (12000, 9000, 1234, 2, 448, True),
    "l1_cli_stride":   (6000, 5000, 77, 1, None, True),       # P=896, S=224
    "l1_odd_stride":   (6000, 5000, 77, 1, 300, True),        # stride not a multiple of the 4x scale
    "l0_cli_stride":   (4000, 3000, 5, 0, None, True),        # P=1792, S=224: 252 candidates (SURVEY §8c)
    "l0_nonoverlap":   (4000, 3000, 5, 0, 1792, True),
    "l3_no_mask":      (9000, 7000, 99, 3, None, False),      # no annotation -> all "normal"
    "l0_tiny_slide":   (1000, 800, 3, 0, None, True),         # slide smaller than one patch
    "l2_exact_fit":    (3584 * 4 // 4, 1792, 11, 2, 448, True),  # level dims multiple of P: no padding
    # slide smaller than one patch WITH survivors: every patch is mostly white padding, the dark content decides
    # (seed < 0 selects conftest.dark_level: uniform noise in [40, 170) instead of the synthetic tissue layout)
    "l0_tiny_dark":    (1500, 1400, -7, 0, None, True),
    "l1_tiny_dark":    (1300, 1000, -9, 1, None, True),       # level-1 image 650 x 500 < P = 896
}
N_FULL = 4   # full resized images kept per case


def stage1_case(name):
    w0, h0, seed, level, stride, with_mask = CASES[name]
    slide = make_slide(w0, h0, seed, with_mask)
    ref = rh.run_reference_extract_patches(slide, level, stride=stride, with_mask=with_mask)
    coords = np.asarray([(r[1], r[2]) for r in ref], dtype=np.int32).reshape(-1, 2)
    labels = np.asarray([r[3] for r in ref], dtype=np.uint8)
    crcs = np.zeros(len(ref), dtype=np.uint32)
    full_idx = sorted(set(np.linspace(0, max(len(ref) - 1, 0), N_FULL).astype(int).tolist())) if ref else []
    full = []
    for i, r in enumerate(ref):
        img = rh.run_reference_resize_u8(r[4])
        crcs[i] = zlib.crc32(img.tobytes())
        if i in full_idx:
            full.append(img)
    names = np.asarray([r[0] for r in ref])
    return dict(w0=w0, h0=h0, seed=seed, level=level, stride=-1 if stride is None else stride,
                with_mask=int(with_mask), coords=coords, labels=labels, crc32=crcs,
                full_idx=np.asarray(full_idx, dtype=np.int64),
                full=np.stack(full) if full else np.zeros((0, 224, 224, 3), np.uint8), names=names)


def stage2_case():
    import torch
    net = orc.make_resnet18(seed=0, classifier=True)
    sd = rh.torchvision_to_feature_extractor_keys(net.state_dict())
    patches, src = [], []
    for name, take in (("l3_default", 4), ("l2_cli_stride", 3), ("l0_nonoverlap", 1)):
        w0, h0, seed, level, stride, with_mask = CASES[name]
        slide = SyntheticSlide(w0, h0, seed=seed, with_lesion=with_mask)
        ref = rh.run_reference_extract_patches(slide, level, stride=stride, with_mask=with_mask)
        for i in np.linspace(0, len(ref) - 1, take).astype(int):
            patches.append(ref[i][4])
            src.append((name, int(ref[i][1]), int(ref[i][2])))
    feats = rh.run_reference_features(patches, sd)
    u8 = np.stack([rh.run_reference_resize_u8(p) for p in patches])
    with torch.no_grad():
        logits = net.fc(torch.from_numpy(feats)).numpy()
    wsum = float(sum(v.double().abs().sum() for v in net.state_dict().values()))
    return dict(images=u8, features=feats.astype(np.float32), logits=logits.astype(np.float32),
                src_case=np.asarray([s[0] for s in src]), src_xy=np.asarray([(s[1], s[2]) for s in src], np.int32),
                weight_abs_sum=wsum, seed=0)


CONFIG0 = dict(size0=32768, slide_seed=1234, level=3, weight_seed=0)   # bench.py --config 0's slide: 361 candidates


def config0_case():
    """Every survivor of BASELINE configs[0]: the 4096 x 4096 level-3 image of a 32768^2 synthetic slide, P = S = 224,
    tissue filter + lesion labels + fp32 ResNet18 features and logits of the seeded weights.  The unmodified reference
    kept 116 of the 361 candidates of this slide (profiles/r02_bench_config0.json)."""
    c = CONFIG0
    slide = SyntheticSlide(c["size0"], c["size0"], seed=c["slide_seed"])
    want = orc.extract_patches_oracle(slide.level_array(c["level"]), slide.lesion_mask(c["level"]), c["level"])
    assert want["candidates"] == 361 and len(want["coords"]) == 116, (want["candidates"], len(want["coords"]))
    net = orc.make_resnet18(seed=c["weight_seed"], classifier=True)
    feats, logits = orc.resnet18_features_fp32(net, want["images"])
    wsum = float(sum(v.double().abs().sum() for v in net.state_dict().values()))
    return dict(**c, candidates=want["candidates"], coords=want["coords"], labels=want["labels"],
                features=feats.astype(np.float32), logits=logits.astype(np.float32), weight_abs_sum=wsum)


def main():
    only = sys.argv[1:]
    if only == ["config0"]:
        d = config0_case()
        np.savez_compressed(os.path.join(HERE, "config0.npz"), **d)
        print(f"config0: {len(d['coords'])} survivors of {d['candidates']} candidates, {int(d['labels'].sum())} tumor")
        return
    assert rh.reference_available(), "needs the reference checkout (HIPAC_REFERENCE_ROOT)"
    for name in CASES:
        if only and name not in only:
            continue
        d = stage1_case(name)
        np.savez_compressed(os.path.join(HERE, f"stage1_{name}.npz"), **d)
        print(f"{name}: {len(d['coords'])} survivors, {int(d['labels'].sum())} tumor")
    if only and "stage2" not in only:
        return
    d = stage2_case()
    np.savez_compressed(os.path.join(HERE, "stage2_features.npz"), **d)
    print("stage2:", d["features"].shape, "weight_abs_sum", d["weight_abs_sum"])


if __name__ == "__main__":
    main()
