"""Cost of the rotation/flip test-time augmentation (tta=True) on the bench workload; one JSON line on stdout.

Workload: the bench's synthetic 16384 x 16384 level-0 image (seed 1234, P = 1792 on the 224-px grid) and its 2048 x 2048
level 3, each with its synthetic lesion mask, and the seeded ResNet18 with a two-class head.  Reports the card and its power
limit; the level-0 process_level step plain and with tta=True, alternated step by step (CUDA events around each step,
warm-up excluded); the per-kernel times of one step of each from the library's profiler (the view kernel is `d4_view`);
and the cascade 3 -> 0 with and without TTA at one tau (the 75th percentile of the TTA level-3 margins), alternated.
Checks that the TTA step keeps the plain step's coordinates and labels.

    python tools/tta_rate.py [--steps 10] [--out profiles/r05_tta_rate.json]
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
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


def step_ms(fn):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    r = fn()
    b.record()
    b.synchronize()
    return r, a.elapsed_time(b)


def alternate(fns: dict, steps: int):
    """Each function warmed up twice, then `steps` rounds calling them in turn: {name: summary of its step times}."""
    for fn in fns.values():
        for _ in range(2):
            step_ms(fn)
    times = {k: [] for k in fns}
    for _ in range(steps):
        for k, fn in fns.items():
            times[k].append(step_ms(fn)[1])
    return {k: {"median_ms": round(statistics.median(t), 3), "min_ms": round(min(t), 3), "max_ms": round(max(t), 3),
                "steps": len(t)} for k, t in times.items()}


def profiled(fn):
    """Per-kernel {name: {launches, ms, work}} of one call (the profiler brackets every library launch with events)."""
    from ss25_hierarchical_multiscale_image_classification_b200 import _lib
    _lib.profile_report()
    _lib.profile(True)
    try:
        fn()
        rep = _lib.profile_report()
    finally:
        _lib.profile(False)
    return {k: {"launches": v["launches"], "ms": round(v["ms"], 4), "work": v["work"]} for k, v in sorted(rep.items())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10, help="timed steps per variant (after 2 warm-up steps each)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    import numpy as np
    import torch
    from ss25_hierarchical_multiscale_image_classification_b200 import _lib, features, pipeline
    from ss25_hierarchical_multiscale_image_classification_b200.cascade import process_cascade, tumor_margin
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

    plain = pipeline.process_level(img0, msk0, 0, packed)
    tta = pipeline.process_level(img0, msk0, 0, packed, tta=True)
    out["level0"] = {"candidates": plain.candidates, "survivors": len(plain),
                     "tta_keeps_coords_and_labels": bool(torch.equal(plain.coords, tta.coords) and torch.equal(plain.labels, tta.labels))}
    steps = alternate({"plain": lambda: pipeline.process_level(img0, msk0, 0, packed),
                       "tta": lambda: pipeline.process_level(img0, msk0, 0, packed, tta=True)}, args.steps)
    steps["tta_over_plain"] = round(steps["tta"]["median_ms"] / steps["plain"]["median_ms"], 3)
    out["process_level_level0"] = steps
    prof = {"plain": profiled(lambda: pipeline.process_level(img0, msk0, 0, packed)),
            "tta": profiled(lambda: pipeline.process_level(img0, msk0, 0, packed, tta=True))}
    view = prof["tta"].get("d4_view", {"launches": 0, "ms": 0.0, "work": 0.0})
    out["view_kernel"] = {"launches": view["launches"], "ms_total": view["ms"],
                          "ms_per_launch": round(view["ms"] / max(view["launches"], 1), 4),
                          "bytes": view["work"], "tb_per_s": round(view["work"] / (view["ms"] * 1e-3) / 1e12, 3) if view["ms"] else None}
    out["kernel_ms_sum"] = {k: round(sum(v["ms"] for v in p.values()), 3) for k, p in prof.items()}
    out["profile"] = prof

    coarse = pipeline.process_level(img3, msk3, COARSE, packed, tta=True)
    theta = float(np.quantile(tumor_margin(coarse.logits).cpu().numpy().astype(np.float64), 0.75))
    tau = 1.0 / (1.0 + math.exp(-theta))
    levels = {COARSE: (img3, msk3), 0: (img0, msk0)}
    res = {k: process_cascade(levels, packed, order=(COARSE, 0), tau=tau, tta=k == "tta") for k in ("plain", "tta")}
    casc = alternate({k: (lambda t=(k == "tta"): process_cascade(levels, packed, order=(COARSE, 0), tau=tau, tta=t))
                      for k in ("plain", "tta")}, args.steps)
    for k in ("plain", "tta"):
        casc[k].update(coarse_survivors=len(res[k][COARSE]), fine_candidates=res[k][0].candidates, fine_survivors=len(res[k][0]))
    out["cascade_3_to_0"] = {"tau": tau, "note": "tau = sigmoid(75th percentile of the TTA level-3 margins); both runs "
                                                 "score their ROI with their own logits", **casc}
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
