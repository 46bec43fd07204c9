"""Cost of the tissue segmentation and the tissue-mask filter on the bench workload; one JSON line on stdout.

Workload: the bench's synthetic 16384 x 16384 level-0 image (seed 1234, P = 1792 on the 224-px grid, no lesion mask) and
its 2048 x 2048 level-3 thumbnail, segmented with the default recipe (7 x 7 median, Otsu) and used at scale m = 8 with
min_tissue = 0.5.  Reports the card and its power limit, per-kernel times from the library's event profiler for segmenting
the thumbnail and the whole 16384^2 level, their bytes against a device-to-device copy rate measured in the same run,
the process_level step time and survivors with the default mean > 240 rule and with the tissue filter, and launch counts.

    python tools/tissue_rate.py [--reps 20] [--steps 10] [--out profiles/r03_tissue_rate.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SEED, WIDTH, THUMB, M = 1234, 16384, 2048, 8
STAGE1 = ("scan_planes", "cell_votes", "cell_stats", "patch_flags", "stats_direct", "tissue_cells", "tissue_flags", "compact",
          "downsample_planes", "gather", "resample_direct", "sat_median", "otsu", "binarize")


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


def copy_gbs():
    """Device-to-device copy of 4 GiB (read + write), larger than L2: the HBM rate this run can reach."""
    import torch
    src = torch.empty(1 << 32, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    dst.copy_(src)
    ms = events_ms(lambda: dst.copy_(src), 10)
    return 2 * src.numel() / ms / 1e6


def kernel_profile(fn, reps):
    from ss25_hierarchical_multiscale_image_classification_b200 import _lib
    import torch
    torch.cuda.synchronize()
    _lib.profile(True)
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    rep = _lib.profile_report()
    _lib.profile(False)
    return {k: {"launches": v["launches"] // reps, "ms": round(v["ms"] / reps, 5), "bytes": v["work"] / reps} for k, v in rep.items()}


def launches(fn):
    from ss25_hierarchical_multiscale_image_classification_b200 import _lib
    l = _lib.lib()
    l.hipac_launch_count(1)
    fn()
    return int(l.hipac_launch_count(1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20, help="segmentation calls per profiled window")
    ap.add_argument("--steps", type=int, default=10, help="timed process_level steps per variant (after 3 warm-up steps)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    import torch
    from ss25_hierarchical_multiscale_image_classification_b200 import _lib, features, pipeline
    from ss25_hierarchical_multiscale_image_classification_b200.preprocessing import alloc_level_image, segment_tissue, upload_level_rows
    from ss25_hierarchical_multiscale_image_classification_b200.synthetic import make_level, seeded_resnet18

    _lib.build()
    torch.cuda.set_device(0)
    out = {"card": card(), "workload": f"synthetic seed {SEED}: level 0 {WIDTH}^2 (P=1792, S=224, no lesion mask), "
                                       f"level-3 thumbnail {THUMB}^2, ksize 7, Otsu, tissue_scale {M}, min_tissue 0.5"}
    thumb = torch.from_numpy(make_level(SEED, 3, THUMB, THUMB)).cuda()
    level = alloc_level_image(WIDTH, WIDTH, "cuda")
    for r in range(0, WIDTH, 2048):
        upload_level_rows(level, make_level(SEED, 0, WIDTH, WIDTH, r, r + 2048), r)
    torch.cuda.synchronize()
    peak = copy_gbs()
    out["hbm_copy_gbs_measured"] = round(peak, 1)

    def seg_record(img, name):
        H, W = int(img.shape[0]), int(img.shape[1])
        segment_tissue(img)
        prof = kernel_profile(lambda: segment_tissue(img), args.reps)
        ms = events_ms(lambda: segment_tissue(img), args.reps)
        # bytes the algorithm must move: RGB in, blurred plane out and back in, mask out
        need = H * W * 3 + H * W + H * W + H * W
        k_ms = sum(v["ms"] for v in prof.values())
        out[name] = {"shape": [H, W], "kernels": prof, "call_ms": round(ms, 5), "kernel_ms": round(k_ms, 5),
                     "algorithmic_bytes": need, "gbs": round(need / k_ms / 1e6, 1), "frac_of_copy_rate": round(need / k_ms / 1e6 / peak, 4),
                     "launches": launches(lambda: segment_tissue(img))}

    seg_record(thumb, "segment_thumbnail")
    seg_record(level, "segment_level0")
    mask, t = segment_tissue(thumb)
    out["otsu_threshold"] = int(t.item())
    out["thumbnail_tissue_fraction"] = round(float((mask > 0).float().mean()), 4)

    net = seeded_resnet18(0, True)
    packed = features.pack_resnet18(net.state_dict(), "cuda")
    variants = {
        "default_rule": lambda: pipeline.process_level(level, None, 0, packed),
        "tissue_filter": lambda: pipeline.process_level(level, None, 0, packed, tissue=mask, tissue_scale=M),
        "segment_and_filter": lambda: pipeline.process_level(level, None, 0, packed, tissue=segment_tissue(thumb)[0], tissue_scale=M),
    }
    steps = {}
    for name, fn in variants.items():
        for _ in range(3):
            r = fn()
        steps[name] = {"survivors": len(r), "candidates": r.candidates, "launches": launches(fn)}
    for _ in range(2):                         # alternate the variants: the shared host drifts
        for name, fn in variants.items():
            steps[name].setdefault("ms", []).append(round(events_ms(fn, args.steps), 3))
    for name, fn in variants.items():
        prof = kernel_profile(fn, 2)
        steps[name]["stage1_kernels"] = {k: v for k, v in prof.items() if k in STAGE1}
    out["process_level"] = steps
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
