"""Cost and yield of the coarse-to-fine cascade 3 -> 0 on the bench workload; one JSON line on stdout.

Workload: the bench's synthetic 16384 x 16384 level-0 image (seed 1234, P = 1792 on the 224-px grid) and its 2048 x 2048
level 3, each with its synthetic lesion mask, and the seeded ResNet18 with a two-class head.  Reports the card and its
power limit, the full process_level of level 0, and the cascade at three thresholds taken from quantiles of the coarse
margins (about 10 / 25 / 50 % of the coarse survivors positive) plus the lesion-guided ROI (coarse labels >= 0.5).  For each
run: fine candidates and survivors, set ROI cells, the fine step's device time (CUDA events, warm-up excluded), the coarse
time (level-3 process_level + ROI grid), and whether the cascade's fine rows equal the full run restricted by
oracle/cascade.py bit for bit.

    python tools/cascade_rate.py [--steps 10] [--out profiles/r04_cascade_rate.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SEED, WIDTH, COARSE = 1234, 16384, 3


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, timeout=30).stdout.strip()
    name, power, clock = (s.strip() for s in q.split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def events_ms(fn, reps):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10, help="timed steps per run (after 2 warm-up steps)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    import numpy as np
    import torch
    from oracle import cascade as oc
    from ss25_hierarchical_multiscale_image_classification_b200 import _lib, features, pipeline
    from ss25_hierarchical_multiscale_image_classification_b200.cascade import roi_grid, tumor_margin
    from ss25_hierarchical_multiscale_image_classification_b200.preprocessing import alloc_level_image, upload_level_rows
    from ss25_hierarchical_multiscale_image_classification_b200.synthetic import make_lesion_mask, make_level, seeded_resnet18

    _lib.build()
    torch.cuda.set_device(0)
    wc = WIDTH >> COARSE
    out = {"card": card(), "workload": f"synthetic seed {SEED}: level 0 {WIDTH}^2 (P=1792, S=224) and level {COARSE} {wc}^2 "
                                       f"(P=224, S=224), synthetic lesion masks, seeded ResNet18 with a 2-class head"}
    img0 = alloc_level_image(WIDTH, WIDTH, "cuda")
    msk0 = alloc_level_image(WIDTH, WIDTH, "cuda", channels=1)
    for r in range(0, WIDTH, 2048):
        upload_level_rows(img0, make_level(SEED, 0, WIDTH, WIDTH, r, r + 2048), r)
        upload_level_rows(msk0, make_lesion_mask(SEED, 0, WIDTH, WIDTH, r, r + 2048), r)
    img3 = torch.from_numpy(make_level(SEED, COARSE, wc, wc)).cuda()
    msk3 = torch.from_numpy(make_lesion_mask(SEED, COARSE, wc, wc)).cuda()
    torch.cuda.synchronize()
    packed = features.pack_resnet18(seeded_resnet18(0, True).state_dict(), "cuda")

    def timed(fn):
        for _ in range(2):
            r = fn()
        return r, round(events_ms(fn, args.steps), 3)

    full, full_ms = timed(lambda: pipeline.process_level(img0, msk0, 0, packed))
    out["full_level0"] = {"candidates": full.candidates, "survivors": len(full), "ms": full_ms}
    coarse, coarse_ms = timed(lambda: pipeline.process_level(img3, msk3, COARSE, packed))
    margin = tumor_margin(coarse.logits)
    out["coarse_level3"] = {"candidates": coarse.candidates, "survivors": len(coarse), "ms": coarse_ms}
    full_np = {k: getattr(full, k).cpu().numpy() for k in ("coords", "labels", "features", "logits")}
    m_np = margin.cpu().numpy()
    runs = {}
    cases = [(f"margin_top_{int(f * 100)}pct", margin, float(np.quantile(m_np, 1 - f))) for f in (0.10, 0.25, 0.50)]
    cases.append(("lesion_guided", coarse.labels.float(), 0.5))
    for name, scores, theta in cases:
        roi = roi_grid(coarse.coords, scores, COARSE, wc, wc, threshold=theta)
        grid_ms = round(events_ms(lambda: roi_grid(coarse.coords, scores, COARSE, wc, wc, threshold=theta), args.steps), 4)
        fine, fine_ms = timed(lambda: pipeline.process_level(img0, msk0, 0, packed, roi=roi))
        want = oc.restrict(full_np, oc.Roi(roi.grid.cpu().numpy(), COARSE, roi.stride, roi.patch), 0)
        parity = all(np.array_equal(getattr(fine, k).cpu().numpy().view(np.uint8), want[k].view(np.uint8))
                     for k in ("coords", "labels", "features", "logits"))
        runs[name] = {"threshold": theta, "positive_coarse": int((scores >= theta).sum()), "roi_cells": int(roi.grid.sum()),
                      "fine_candidates": fine.candidates, "fine_survivors": len(fine), "fine_ms": fine_ms,
                      "coarse_ms": round(coarse_ms + grid_ms, 3), "roi_grid_ms": grid_ms,
                      "cascade_ms": round(coarse_ms + grid_ms + fine_ms, 3), "parity_with_full_restricted": parity}
    out["cascade_3_to_0"] = runs
    out["parity"] = all(r["parity_with_full_restricted"] for r in runs.values())
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
