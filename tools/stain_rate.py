"""Cost of the Macenko stain normalisation (stain=) on the bench workload; one JSON line on stdout.

Workload: the bench's synthetic 16384 x 16384 level-0 image (seed 1234, P = 1792 on the 224-px grid) with its lesion mask,
its 2048 x 2048 level-3 thumbnail, and the seeded ResNet18 with a two-class head.  Reports the card and its power limit;
the estimation time on the thumbnail (CUDA events around each call, and the per-kernel profile of one call); the apply
kernel alone on the level-0 survivors' uint8 patches (330 MB, larger than L2) in both layouts, with its bandwidth on the
algorithmic bytes (150 528 B read plus 412 160 B (S2D16) or 301 056 B (NHWC3) written per survivor) as a share of
7.7 TB/s; and the level-0 process_level step plain and with stain=, alternated step by step.  Checks that the normalised
step keeps the plain step's coordinates and labels.

    python tools/stain_rate.py [--steps 10] [--out profiles/r06_stain_rate.json]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from tta_rate import alternate, card, profiled  # noqa: E402

SEED, WIDTH, COARSE = 1234, 16384, 3
PEAK_TB_S = 7.7


def events_ms(fn, reps: int):
    """Median / min of `reps` calls, each bracketed by CUDA events (after two warm-up calls)."""
    import torch
    for _ in range(2):
        fn()
    t = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        t.append(a.elapsed_time(b))
    return {"median_ms": round(statistics.median(t), 4), "min_ms": round(min(t), 4), "reps": reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10, help="timed steps per variant (after 2 warm-up steps each)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    import torch
    from ss25_hierarchical_multiscale_image_classification_b200 import _lib, features, pipeline
    from ss25_hierarchical_multiscale_image_classification_b200.preprocessing import (StainNormalizer, alloc_level_image,
                                                                                      estimate_stain, extract_patches_tensor,
                                                                                      upload_level_rows)
    from ss25_hierarchical_multiscale_image_classification_b200.synthetic import make_lesion_mask, make_level, seeded_resnet18

    _lib.build()
    torch.cuda.set_device(0)
    wc = WIDTH >> COARSE
    out = {"card": card(), "workload": f"synthetic seed {SEED}: level 0 {WIDTH}^2 (P=1792, S=224) with its lesion mask, "
                                       f"level {COARSE} {wc}^2 as the thumbnail, seeded ResNet18 with a 2-class head"}
    img0 = alloc_level_image(WIDTH, WIDTH, "cuda")
    msk0 = alloc_level_image(WIDTH, WIDTH, "cuda", channels=1)
    for r in range(0, WIDTH, 2048):
        upload_level_rows(img0, make_level(SEED, 0, WIDTH, WIDTH, r, r + 2048), r)
        upload_level_rows(msk0, make_lesion_mask(SEED, 0, WIDTH, WIDTH, r, r + 2048), r)
    img3 = torch.from_numpy(make_level(SEED, COARSE, wc, wc)).cuda()
    torch.cuda.synchronize()
    packed = features.pack_resnet18(seeded_resnet18(0, True).state_dict(), "cuda")

    stain = estimate_stain(img3)
    norm = StainNormalizer(stain)
    out["stain"] = {"valid": stain.valid(), "n_hat": int(stain.n_hat), "he": stain.he.cpu().tolist(),
                    "max_c": stain.max_c.cpu().tolist()}
    out["estimate_thumbnail"] = {**events_ms(lambda: estimate_stain(img3), 20), "pixels": wc * wc,
                                 "profile": profiled(lambda: estimate_stain(img3))}

    pb = extract_patches_tensor(img0, msk0, 0, layout=None, want_u8=True)
    n = len(pb)
    u8 = pb.images_u8.contiguous()
    apply = {"survivors": n}
    for layout, wbytes in (("s2d16", 412160), ("nhwc3", 301056)):
        shape = (n, 112, 115, 16) if layout == "s2d16" else (n, 224, 224, 3)
        batch = torch.empty(shape, dtype=torch.bfloat16, device="cuda")
        t = events_ms(lambda: norm.apply(u8, layout, out=batch), 20)
        nbytes = n * (150528 + wbytes)
        t.update(algorithmic_bytes=nbytes, tb_per_s=round(nbytes / (t["median_ms"] * 1e-3) / 1e12, 3),
                 share_of_7_7_tb_s=round(nbytes / (t["median_ms"] * 1e-3) / 1e12 / PEAK_TB_S, 3))
        apply[layout] = t
    out["apply_kernel"] = apply

    plain = pipeline.process_level(img0, msk0, 0, packed)
    normed = pipeline.process_level(img0, msk0, 0, packed, stain=norm)
    out["level0"] = {"candidates": plain.candidates, "survivors": len(plain),
                     "stain_keeps_coords_and_labels": bool(torch.equal(plain.coords, normed.coords)
                                                           and torch.equal(plain.labels, normed.labels))}
    steps = alternate({"plain": lambda: pipeline.process_level(img0, msk0, 0, packed),
                       "stain": lambda: pipeline.process_level(img0, msk0, 0, packed, stain=norm)}, args.steps)
    steps["stain_minus_plain_ms"] = round(steps["stain"]["median_ms"] - steps["plain"]["median_ms"], 3)
    out["process_level_level0"] = steps
    prof = profiled(lambda: pipeline.process_level(img0, msk0, 0, packed, stain=norm))
    out["process_level_stain_apply_profile"] = prof.get("stain_apply")
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
