#!/usr/bin/env python
"""HiPAC hot-path benchmark: patches/sec through tile + tissue/lesion mask + ResNet18 features.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): a synthetic level-0 image, 16384 x 16384 RGB per GPU, tiled
into 1792^2 patches on the reference CLI's 224-px grid (src/main.py:611 -> stride 224 at every
level), white-padded borders, mean>240 tissue rejection, lesion-mask labels, Pillow-exact resize to
224^2, ImageNet normalisation, then ResNet18 512-d features + 2-class logits for every survivor.
A "step" is one pass over the whole level image.  With N > 1 the slide is N x 16384 rows tall and is
sharded by candidate tile-row range across the ranks (weak scaling: per-GPU work fixed); the only
collective is the NCCL all-gather of survivor counts / coordinates / labels / features.

Prints ONE JSON line (rank 0).  `value` = survivors (patches that get features) per second over all
ranks with the image resident in HBM; `e2e` = same through host buffers (pinned H2D of the image and
mask, D2H of coords / labels / features inside the timed region).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LEVEL, PATCH, STRIDE = 0, 1792, 224
WIDTH, ROWS_PER_GPU = 16384, 16384
SEED = 1234
FLOP_PER_PATCH = 3.627e9          # SURVEY.md section 2.2 (conv 2*MAC + fc)
# SURVEY.md section 8(d): algorithmic stage-1 output per survivor = the bf16 NHWC 224x224x3 image + coords (8) + label (1)
ALGO_OUT_BYTES = 224 * 224 * 3 * 2 + 9
# what the kernels really write per survivor: the S2D16 operand layout of conv1 (16 of 12 channels, 115 of 112 columns)
S2D_BYTES = 112 * 115 * 16 * 2
REF_STRIDE_MULT = 20              # --impl reference: the reference's own stride argument = 224 * this (every 20th grid column/row)
DUMP_LIMIT_BYTES = 64_000_000     # --dump-outputs: larger patch sets are reduced to a fixed, seeded sample of rows


def dump_outputs(out_dir: str, res: dict):
    """Write the patch set a caller of the timed path receives (coords, labels, features, logits) as
    ``out_dir/<name>.npy`` in float32 (coordinates and labels are small integers, exact in float32).  If the set exceeds
    DUMP_LIMIT_BYTES, the same seeded sample of rows (kept in canonical order) is taken from every array, and its row
    indices are written as ``rows.npy``; otherwise every row is written."""
    n = int(res["coords"].shape[0])
    row_bytes = sum(4 * int(np.prod(v.shape[1:])) for v in res.values())
    if n * row_bytes + 1024 * len(res) <= DUMP_LIMIT_BYTES:
        rows = None
    else:                                                  # + 8 bytes per row for rows.npy, 1 KB per .npy header
        keep = (DUMP_LIMIT_BYTES - 1024 * (len(res) + 1)) // (row_bytes + 8)
        rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for k, v in res.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), np.ascontiguousarray((v if rows is None else v[rows]).astype(np.float32)))
    if rows is not None:
        np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))


def ncu_traffic():
    """DRAM bytes per step from the newest committed ncu capture (profiles/r*_traffic.json), or {} if absent.  This is a
    COMMITTED CONSTANT of the capture named in its "source" field, not measured in this run (ncu replays kernels ~40x, so it
    cannot run inside the timed bench); `traffic_source` in the JSON line says so."""
    try:
        pd = os.path.join(ROOT, "profiles")
        names = sorted(f for f in os.listdir(pd) if f.endswith("_traffic.json"))
        d = json.load(open(os.path.join(pd, names[-1])))
        d["file"] = "profiles/" + names[-1]
        return d
    except Exception:
        return {}


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region: NVML in-process every 10 ms
    (nvidia-smi every 200 ms as the fallback)."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.sm, self.flags, self.max_mhz, self._stop = index, [], set(), None, threading.Event()
        self.source = "nvml"
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run_nvml(self):
        import pynvml as nv
        nv.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[self.index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else self.index
        h = nv.nvmlDeviceGetHandleByIndex(phys)
        self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
        while not self._stop.is_set():
            self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
            self.flags.update(n for n, bit in names.items() if r & bit)
            self._stop.wait(0.01)

    def _run_smi(self):
        self.source = "nvidia-smi"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    c = [v.strip() for v in out.split(",")]
                    self.sm.append(float(c[0]))
                    self.max_mhz = float(c[1])
                    self.flags.update(n for i, n in enumerate(names) if c[2 + i].lower().startswith("active"))
            except Exception:
                pass
            self._stop.wait(0.2)

    def _run(self):
        try:
            self._run_nvml()
        except Exception:
            self._run_smi()

    def __enter__(self):
        self._t.start()
        time.sleep(0.03)
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": statistics.median(self.sm), "sm_min_mhz": min(self.sm), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.flags), "samples": len(self.sm), "source": self.source}


def bind_near_gpu(index: int):
    """Pin this process to the host cores NVML reports as local to GPU `index` (its NUMA node), BEFORE any pinned host
    buffer is allocated: first-touch then places the staging memory next to the GPU's PCIe root, which is what the e2e
    leg's H2D rate depends on when several ranks upload at once.  Best effort: returns the cpu count or None."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
        h = nv.nvmlDeviceGetHandleByIndex(phys)
        words = nv.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        near = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
        allowed = near & os.sched_getaffinity(0)
        if len(allowed) >= 2:
            os.sched_setaffinity(0, allowed)
            return len(allowed)
    except Exception:
        pass
    return None


_period_mask = None


def lesion_polygons(world: int = 1):
    """The slide's lesion ANNOTATIONS: the synthetic lesion ellipses as 720-vertex integer polygons, one copy per 16384-row
    period of the N x 16384-row slide (what a CAMELYON16 XML holds, after parse_xml_mask's int(x * scale) truncation,
    reference src/main.py:388-405)."""
    from ss25_hierarchical_multiscale_image_classification_b200.synthetic import _geometry
    _, lesion, _, _ = _geometry(SEED, LEVEL, WIDTH, ROWS_PER_GPU)
    t = np.linspace(0.0, 2.0 * np.pi, 720, endpoint=False)
    base = [np.stack([(cx + rx * np.cos(t)).astype(np.int64), (cy + ry * np.sin(t)).astype(np.int64)], 1).astype(np.int32)
            for cx, cy, rx, ry in lesion]
    return [p + np.array([0, k * ROWS_PER_GPU], np.int32) for k in range(world) for p in base]


def period_mask():
    """uint8 [16384, 16384] lesion mask of one period, rasterised on the HOST the way the reference does it:
    ImageDraw.polygon(coords, outline=255, fill=255) per annotation (src/main.py:392-409).  Input of the CPU arms and the
    cross-check of the device rasteriser."""
    global _period_mask
    if _period_mask is None:
        from PIL import Image, ImageDraw
        im = Image.new("L", (WIDTH, ROWS_PER_GPU), 0)
        d = ImageDraw.Draw(im)
        for p in lesion_polygons(1):
            d.polygon([(int(x), int(y)) for x, y in p], outline=255, fill=255)
        _period_mask = np.array(im)
    return _period_mask


def shard_rows(ny_total: int, world: int, rank: int):
    """Contiguous candidate tile-row range of `rank` (balanced by row count)."""
    base, rem = divmod(ny_total, world)
    i0 = rank * base + min(rank, rem)
    return i0, i0 + base + (1 if rank < rem else 0)


def build_slab(world: int, rank: int, pinned: bool = True):
    """Pinned host tensors of this rank's row slab (+ halo) of the N x 16384-row synthetic slide.

    The slide's content repeats every 16384 rows (row y shows row y mod 16384 of the N = 1 slide), so the per-GPU
    work really is fixed as N grows: every rank tiles the same tissue layout; only the last rank sees the slide's
    bottom edge (white-padded patches), exactly like the single rank at N = 1."""
    import torch
    from ss25_hierarchical_multiscale_image_classification_b200.synthetic import make_level
    H = ROWS_PER_GPU * world
    pm = period_mask()
    ny_total = (H + STRIDE - 1) // STRIDE
    i0, i1 = shard_rows(ny_total, world, rank)
    y0, y1 = i0 * STRIDE, min(H, (i1 - 1) * STRIDE + PATCH)
    img = torch.empty((y1 - y0, WIDTH, 3), dtype=torch.uint8)
    msk = torch.empty((y1 - y0, WIDTH), dtype=torch.uint8)
    if pinned:
        img, msk = img.pin_memory(), msk.pin_memory()
    inp, mnp = img.numpy(), msk.numpy()

    def fill(r):
        r1 = min(r + 256, y1)
        while r < r1:                                   # split at period boundaries
            q = r % ROWS_PER_GPU
            n = min(r1 - r, ROWS_PER_GPU - q)
            inp[r - y0:r - y0 + n] = make_level(SEED, LEVEL, WIDTH, ROWS_PER_GPU, q, q + n)
            mnp[r - y0:r - y0 + n] = pm[q:q + n]
            r += n

    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max(1, min(16, (os.cpu_count() or 8) // max(1, world)))) as ex:
        list(ex.map(fill, range(y0, y1, 256)))
    return img, msk, (i0, i1, y0, H)


def run_ours(args):
    import torch
    import torch.distributed as dist
    import __graft_entry__ as ge
    from ss25_hierarchical_multiscale_image_classification_b200 import _lib, features, pipeline, sharding
    from ss25_hierarchical_multiscale_image_classification_b200.synthetic import seeded_resnet18

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    cpus_before = len(os.sched_getaffinity(0))
    near_cpus = bind_near_gpu(local) if world > 1 else None
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # torchrun exports OMP_NUM_THREADS=1; the e2e leg's host work (block-max scan of the lesion mask) wants this
    # rank's share of the host cores
    ranks_sharing = max(1, round(world * len(os.sched_getaffinity(0)) / cpus_before))   # ranks bound to the same cores
    host_threads = max(1, min(16, len(os.sched_getaffinity(0)) // ranks_sharing))
    torch.set_num_threads(host_threads)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ge.build()
    net = seeded_resnet18(seed=0, classifier=True)                        # random-init weights (BASELINE config)
    packed = features.pack_resnet18(net.state_dict(), dev)
    img_h, msk_h, (i0, i1, y0, H) = build_slab(world, rank)
    # the lesion mask is born on the GPU: hipac_polygon_fill rasterises the annotation polygons (bit-exact against the
    # Pillow call of the reference's parse_xml_mask); msk_h -- the same polygons rasterised by Pillow on the host -- is
    # what the CPU arms read and the cross-check below
    from ss25_hierarchical_multiscale_image_classification_b200.preprocessing import lesion_mask as lm
    polys = lm.PolygonSet(lesion_polygons(world), dev)
    img_d = img_h.to(dev)
    msk_d = lm.rasterize_polygons(polys, WIDTH, H, dev, y_begin=y0, n_rows=int(img_h.shape[0]))
    mask_equal = bool(torch.equal(msk_d.cpu(), msk_h))
    rows = (0, i1 - i0)
    n_cand = ((WIDTH + STRIDE - 1) // STRIDE) * (i1 - i0)
    pipe = pipeline.HostPipeline(int(img_h.shape[0]), WIDTH, dev, with_mask=True, num_classes=2)

    nx = (WIDTH + STRIDE - 1) // STRIDE
    # the exchange step (csrc/exchange.cu + one NCCL all-gather): capacity = the largest per-rank candidate count
    ny_total = (ROWS_PER_GPU * world + STRIDE - 1) // STRIDE
    seg_cap = nx * max(shard_rows(ny_total, world, r)[1] - shard_rows(ny_total, world, r)[0] for r in range(world))
    xchg = sharding.SurvivorExchange(dev, seg_cap, 2, nx, STRIDE) if world > 1 else None
    gb = pipeline.upload_group_bounds(0, seg_cap // nx, args.groups)        # e2e leg: one segment per upload row group
    xchg_e2e = sharding.SurvivorExchange(dev, nx * (max(b - a for a, b in zip(gb, gb[1:])) + 1), 2, nx, STRIDE,
                                         segs_per_rank=len(gb) - 1) if world > 1 else None
    last_gathered = {}

    def step_resident():
        if world == 1:
            r = pipeline.process_level(img_d, msk_d, LEVEL, packed, stride=None, row_range=rows, chunk=args.chunk)
            last_gathered["out"] = {"coords": r.coords, "labels": r.labels, "features": r.features, "logits": r.logits}
            return len(r), len(r)
        # tile scan + ResNet18 enqueued without a host wait, then the one exchange step: pack (device count) ->
        # all-gather -> index + scatter into canonical (x, y) order; the only host read of the step is the final total
        seg = pipeline.process_level_enqueue(img_d, msk_d, LEVEL, packed, stride=None, row_range=rows, chunk=args.chunk)
        xchg.pack(0, seg.pend.coords, seg.pend.labels, seg.features, seg.logits, seg.count, y_offset=y0)
        xchg.merge()
        out = xchg.result()
        last_gathered["out"] = out
        return int(out["coords"].shape[0]), None

    def step_e2e():
        # host buffers in, host buffers out: pinned H2D of image + mask (overlapped with compute by row groups),
        # D2H of coords / labels / features / logits; process_level_host synchronises before returning
        r = pipeline.process_level_host(img_h, polys, LEVEL, packed, pipe, stride=None, row_range=rows,
                                        groups=args.groups, chunk=args.chunk, exchange=xchg_e2e, y_offset=y0, polygon_window=(H, y0))
        return len(r), len(r)

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            total, pb = fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            total, pb = fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / steps, total, pb

    _lib.lib().hipac_launch_count(1)
    with ClockSampler(local) as clk:
        ms_step, total_surv, pb = timed(step_resident, args.steps, args.warmup)
    launches = int(_lib.lib().hipac_launch_count(1)) // (args.steps + args.warmup)
    # the gathered, canonically sorted patch set of the last resident step (every rank holds the same one)
    res = {k: v.cpu().numpy() for k, v in last_gathered["out"].items()}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res)
    order = np.lexsort((res["coords"][:, 1], res["coords"][:, 0]))
    canonical = bool(np.array_equal(order, np.arange(len(order))))     # the exchange already delivers (x, y) order
    import zlib
    crc = 0
    for k in ("coords", "labels", "features", "logits"):
        crc = zlib.crc32(np.ascontiguousarray(res[k]).tobytes(), crc)
    # per-kernel CUDA-event timing (library profiler), taken RIGHT AFTER the timed region while the GPU is still at its
    # sustained (power-capped) clocks: 2 steps to settle, then `prof_steps` measured steps.  Events between the kernels
    # serialise them (no programmatic-launch overlap), so these are per-kernel durations, not a second step time.
    prof_steps = max(4, min(10, args.steps))
    _lib.profile(True)
    for _ in range(2):
        pipeline.process_level(img_d, msk_d, LEVEL, packed, stride=None, row_range=rows, chunk=args.chunk)
    torch.cuda.synchronize()
    _lib.profile_report()
    for _ in range(prof_steps):
        pipeline.process_level(img_d, msk_d, LEVEL, packed, stride=None, row_range=rows, chunk=args.chunk)
    torch.cuda.synchronize()
    prof = _lib.profile_report()
    _lib.profile(False)
    for v in prof.values():                              # normalise to the "per 2 steps" convention used below
        v["ms"] *= 2.0 / prof_steps
        v["work"] *= 2.0 / prof_steps
        v["launches"] = int(round(v["launches"] * 2.0 / prof_steps))
    ms_e2e, total_surv_e, n_e2e_rows = timed(step_e2e, args.steps, 1)
    # round 1's methodology, for comparison only: a 2-step profiled pass after the (PCIe-bound, cooler) e2e leg, i.e. at boost clocks
    _lib.profile(True)
    for _ in range(2):
        pipeline.process_level(img_d, msk_d, LEVEL, packed, stride=None, row_range=rows, chunk=args.chunk)
    torch.cuda.synchronize()
    prof_short = _lib.profile_report()
    _lib.profile(False)
    conv_ms_short = sum(v["ms"] for k, v in prof_short.items() if k.startswith("conv")) / 2
    ys = res["coords"][:, 1]
    n_surv = pb if pb is not None else int(((ys >= i0 * STRIDE) & (ys < i1 * STRIDE)).sum())   # this rank's own survivors

    peaks, peak_src = measured_peaks()
    traffic = ncu_traffic()
    conv = {k: v for k, v in prof.items() if k.startswith("conv")}
    conv_ms = sum(v["ms"] for v in conv.values())
    conv_flops = sum(v["work"] for v in conv.values())
    conv_tf = conv_flops / (conv_ms * 1e-3) / 1e12 if conv_ms else 0.0
    conv_tf_short = conv_flops / 2 / (conv_ms_short * 1e-3) / 1e12 if conv_ms_short else 0.0
    # stage 1 is paired with the (burst, best-of-10) HBM copy figure, so it is taken from the short pass at boost clocks -- round 1's
    # method; its duration at the step's sustained clocks is reported beside it
    s1 = {k: v for k, v in prof_short.items() if not k.startswith(("conv", "maxpool", "avgpool", "pack", "exchange"))}
    s1_ms = sum(v["ms"] for v in s1.values()) / 2
    s1_ms_sustained = sum(v["ms"] for k, v in prof.items() if not k.startswith(("conv", "maxpool", "avgpool", "pack", "exchange"))) / 2
    s1_bytes = img_d.numel() + msk_d.numel() + n_surv * ALGO_OUT_BYTES          # SURVEY.md section 8(d)
    s1_written = n_surv * (S2D_BYTES + 9)                                        # what the kernels really write
    s1_gbs = s1_bytes / (s1_ms * 1e-3) / 1e9 if s1_ms else 0.0
    kernels = {k: {"launches_per_step": v["launches"] // 2, "ms_per_step": round(v["ms"] / 2, 4),
                   "ms_per_step_boost": round(prof_short[k]["ms"] / 2, 4) if k in prof_short else None,
                   **({"tflops": round(v["work"] / (v["ms"] * 1e-3) / 1e12, 1)} if k.startswith("conv") and v["ms"] else {})}
               for k, v in prof.items()}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    cpu, parity = None, None
    if world == 1 and not args.no_cpu:
        port_rec, port = cpu_port_sample(args.cpu_candidates)
        parity = parity_block(res, port)
        if reference_available():
            torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
            step = reference_as_written_step(png=True)
            cpu = reference_record(step, int(torch.get_num_threads()))
            # the reference's own decisions on its sub-lattice vs the GPU arm's survivors at the same grid points
            stride = STRIDE * REF_STRIDE_MULT
            ours = {f"tumor_900_x{x}_y{y}_{'tumor' if l else 'normal'}.png" for (x, y), l in zip(res["coords"].tolist(), res["labels"].tolist())
                    if x % stride == 0 and y % stride == 0}
            parity["reference_as_written"] = {"n_candidates": step["candidates"], "n_survivors": step["survivors"],
                                              "file_names_equal": bool(ours == set(step["names"]))}
            parity["pass"] = bool(parity["pass"] and ours == set(step["names"]))
            cpu["port"] = port_rec
        else:
            cpu = port_rec
    out = {
        "metric": "patches/sec (tile+mask+ResNet18 features)",
        "value": round(total_surv / (ms_step * 1e-3), 1),
        "unit": "patches/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms_step, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8 (tiling/mask/resample, bit-exact) + bf16 tensor-core convs with fp32 accumulate",
        "data": "synthetic (counter-hash slide, seeded random-init ResNet18)",
        "config": {"workload": "configs[1]: level-0 16384x16384 RGB per GPU, P=1792 patches on the 224-px CLI grid, "
                               "tissue mean>240 rejection + lesion-mask labels + Pillow-exact resize + ResNet18 features/logits",
                   "level": LEVEL, "patch": PATCH, "stride": STRIDE, "width": WIDTH, "rows_per_gpu": ROWS_PER_GPU,
                   "candidates_per_step": n_cand * world if world == 1 else None, "survivors_per_step": total_surv,
                   "candidates_per_s": round(n_cand * world / (ms_step * 1e-3), 1),
                   "sharding": f"tile-row ranges over {world} rank(s) of one {ROWS_PER_GPU * world}-row slide (content periodic in y, period "
                               f"{ROWS_PER_GPU}); exchange step = device-side pack (count in the header) + ONE fixed-size NCCL all-gather + "
                               "index/scatter kernels into canonical (x, y) order (csrc/exchange.cu); no host-side count exchange",
                   "cache": "inputs (0.8 GB image + 0.27 GB mask per GPU) exceed the 126 MB L2; no flush needed",
                   "resnet_chunk": args.chunk, "e2e_upload_groups": args.groups, "host_threads_per_rank": host_threads, "cpus_near_gpu": near_cpus},
        "e2e": {"value": round(total_surv_e / (ms_e2e * 1e-3), 1), "unit": "patches/s",
                "h2d_bytes_per_step": int(pipe.last_h2d_bytes),
                "h2d_note": "the level image rows, once; the lesion mask never crosses PCIe: the annotation polygons "
                            f"({int(polys.xy.nbytes)} bytes of vertices, resident) are rasterised on the GPU every step (hipac_polygon_fill)",
                "d2h_bytes_per_step": int(n_e2e_rows * (512 * 4 + 2 * 4 + 8 + 1) + 8),
                "d2h_note": "coords + labels + features + logits of every row this rank returns to its host (N > 1: the gathered set)",
                "ms_per_step": round(ms_e2e, 3)},
        "gpu_launches": launches,
        "clocks": clk.summary(),
        "patch_set_crc32": f"{crc:08x}", "patch_set_in_canonical_order": canonical,
        "lesion_mask_device_equals_pillow": mask_equal,
        "roofline": {"bound": "tensor", "kernel": f"conv stack: k_conv1_pool + k_conv3x3_rows2 + k_conv3x3s2_rows2 + k_conv_umma2 ({sum(v['launches'] for v in conv.values()) // 2} launches = 20 conv layers per step)",
                     "achieved": round(conv_tf, 1),
                     "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                     "frac": round(conv_tf / peaks["bf16_tflops_sustained"], 4),
                     "peak_note": "kernels timed inside a long step (sustained, power-capped clocks) against the SUSTAINED cuBLAS bf16 figure, as "
                                  "the profiling recipe pairs them; the burst pairing -- the same kernels timed in a short 2-step pass at boost "
                                  "clocks (round 1's method) against the burst figure -- is given in `burst_pairing`",
                     "burst_pairing": {"achieved": round(conv_tf_short, 1), "peak": peaks["bf16_tflops"],
                                       "frac": round(conv_tf_short / peaks["bf16_tflops"], 4), "conv_ms_per_step": round(conv_ms_short, 3)},
                     "traffic": traffic.get("conv_dram_bytes_per_step"), "traffic_unit": "DRAM bytes per step over the conv launches",
                     "traffic_source": f"committed ncu capture {traffic.get('file')} ({traffic.get('source')}), not measured in this run",
                     "algorithmic_flops_per_step": conv_flops / 2, "peak_source": peak_src,
                     "conv_ms_per_step": round(conv_ms / 2, 3),
                     "timing_note": f"per-kernel CUDA events over {prof_steps} steps taken right after the timed region, at its sustained "
                                    "(power-capped) clocks"},
        "roofline_stage1": {"bound": "hbm", "kernel": "stage-1 tile scan (all kernels)",
                            "achieved": round(s1_gbs, 1) if s1_ms else None,
                            "peak": peaks["hbm_gbs"], "unit": "GB/s",
                            "frac": round(s1_gbs / peaks["hbm_gbs"], 4) if s1_ms else None,
                            "frac_of_nominal_8TBs": round(s1_gbs / 8000.0, 4) if s1_ms else None,
                            "ms_per_step": round(s1_ms, 3), "ms_per_step_at_sustained_clocks": round(s1_ms_sustained, 3),
                            "timing_note": "kernels timed in a short 2-step pass at boost clocks against the burst (best-of-10) HBM copy figure; inside "
                                           "the power-capped step the same kernels take ms_per_step_at_sustained_clocks",
                            "algorithmic_bytes": int(s1_bytes),
                            "algorithmic_bytes_note": "3HW image + HW mask + survivors x (224*224*3*2 + 9) (SURVEY.md 8d)",
                            "written_bytes": int(s1_written),
                            "written_note": "the batch is stored in conv1's S2D16 operand layout (16 of 12 channels, 115 of 112 columns): "
                                            f"{round(s1_written / max(n_surv * ALGO_OUT_BYTES, 1), 3)}x the algorithmic output bytes",
                            "traffic": traffic.get("stage1_dram_bytes_per_step"),
                            "traffic_source": f"committed ncu capture {traffic.get('file')} ({traffic.get('source')}), not measured in this run"},
        "kernels": kernels,
    }
    if parity:
        out["parity"] = parity
    if cpu:
        out["cpu_baseline"] = cpu
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def cpu_sample_regions(budget_candidates: int):
    """Every-k-th candidate of the N=1 workload with its source pixels pre-generated (so synthetic-data
    generation is NOT timed as reference work; the reference would get them from read_region)."""
    from concurrent.futures import ThreadPoolExecutor
    from ss25_hierarchical_multiscale_image_classification_b200.synthetic import make_level
    H = ROWS_PER_GPU
    pm = period_mask()
    nx, ny = (WIDTH + STRIDE - 1) // STRIDE, (H + STRIDE - 1) // STRIDE
    k = max(1, (nx * ny) // budget_candidates)
    cands = [(ix * STRIDE, iy * STRIDE) for ix in range(nx) for iy in range(ny)]
    sample = cands[k // 2::k][:budget_candidates]

    def gen(xy):
        x, y = xy
        w, h = min(PATCH, WIDTH - x), min(PATCH, H - y)
        return xy, (make_level(SEED, LEVEL, WIDTH, H, y, y + h, x, x + w), np.ascontiguousarray(pm[y:y + h, x:x + w]))

    with ThreadPoolExecutor(min(16, os.cpu_count() or 8)) as ex:
        cache = dict(ex.map(gen, sample))
    return sample, cache, k


def cpu_port_sample(budget_candidates: int, regions=None):
    """The CPU PORT of the reference path (oracle/cpu_pipeline.py style) on an every-k-th-candidate sample of the N=1
    workload: timing record + everything the parity block needs (decisions, labels, fp32 features and logits)."""
    import torch
    from oracle import cpu_pipeline, hipac_oracle as orc

    sample, cache, k = regions or cpu_sample_regions(budget_candidates)
    net = orc.make_resnet18(seed=0, classifier=True)

    from PIL import Image
    t0 = time.perf_counter()
    patches, kept, labels, decisions = [], [], [], {}
    for (x, y) in sample:                                      # the reference's per-candidate body (src/main.py:688-727)
        rgb, m = cache[(x, y)]
        region = Image.fromarray(np.dstack([rgb, np.full(rgb.shape[:2], 255, np.uint8)]), "RGBA").convert("RGB")
        if region.size != (PATCH, PATCH):
            padded = Image.new("RGB", (PATCH, PATCH), (255, 255, 255))
            padded.paste(region, (0, 0))
            region = padded
        mask_patch = Image.fromarray(m, "L").crop((0, 0, PATCH, PATCH))
        label = 1 if np.any(np.array(mask_patch) > 0) else 0
        keep = not (np.mean(np.array(region)) > 240)
        decisions[(x, y)] = (keep, label)
        if not keep:
            continue
        patches.append(region)
        kept.append((x, y))
        labels.append(label)
    t1 = time.perf_counter()
    feats = cpu_pipeline.stage2_reference_loop(patches, net, batch=64)
    t2 = time.perf_counter()
    with torch.no_grad():
        logits = net.fc(torch.from_numpy(feats)).numpy() if len(feats) else np.zeros((0, 2), np.float32)
    total = t2 - t0
    rec = {"value": round(len(patches) / total, 2), "unit": "patches/s", "cores": int(torch.get_num_threads()),
           "kind": "port",
           "sample": f"every {k}-th candidate of the N=1 workload: {len(sample)} candidates -> {len(patches)} survivors; "
                     f"stage 1 (single thread, as the reference; no PNG write) {t1 - t0:.2f} s, stage 2 (Resize+ToTensor+"
                     f"Normalize per patch, fp32 ResNet18 on {torch.get_num_threads()} threads, batch 64) {t2 - t1:.2f} s",
           "candidates_per_s": round(len(sample) / total, 2), "host_cpus": os.cpu_count(),
           "feature_checksum": float(np.abs(feats).sum())}
    return rec, {"decisions": decisions, "kept": kept, "labels": labels, "features": feats, "logits": logits}


def parity_block(gpu, port):
    """GPU arm vs the CPU oracle port on the sampled candidates of the FULL-SIZE workload: keep/reject decisions, labels
    (bit-exact bar), features (cosine >= 0.9995, max|d|/max|ref| <= 1e-2) and classifier argmax (>= 99.9 %)."""
    gx = {(int(x), int(y)): i for i, (x, y) in enumerate(gpu["coords"].tolist())}
    dec = port["decisions"]
    coords_equal = all(((xy in gx) == keep) for xy, (keep, _) in dec.items())
    labels_equal = all(int(gpu["labels"][gx[xy]]) == lab for xy, (keep, lab) in dec.items() if keep and xy in gx)
    idx = [gx[xy] for xy in port["kept"] if xy in gx]
    ok = len(idx) == len(port["kept"]) and len(idx) > 0
    out = {"against": "oracle port (fp32 torch, same seeded weights) on the cpu_baseline sample of the full-size workload",
           "n_candidates": len(dec), "n": len(idx), "coords_equal": bool(coords_equal), "labels_equal": bool(labels_equal)}
    if ok:
        g, r = gpu["features"][idx].astype(np.float64), port["features"].astype(np.float64)
        cos = (g * r).sum(1) / (np.linalg.norm(g, axis=1) * np.linalg.norm(r, axis=1))
        maxrel = np.abs(g - r).max(1) / np.abs(r).max(1)
        gl, rl = gpu["logits"][idx], port["logits"]
        out.update({"min_cos": round(float(cos.min()), 7), "max_rel": float(f"{maxrel.max():.3e}"),
                    "argmax_agree": round(float((gl.argmax(1) == rl.argmax(1)).mean()), 6),
                    "min_logit_margin_fp32": round(float(np.abs(rl[:, 0] - rl[:, 1]).min()), 5),
                    "max_logit_diff_error": float(f"{np.abs((gl[:, 1] - gl[:, 0]) - (rl[:, 1] - rl[:, 0])).max():.3e}")})
        out["pass"] = bool(coords_equal and labels_equal and cos.min() >= 0.9995 and maxrel.max() <= 1e-2 and out["argmax_agree"] >= 0.999)
    else:
        out["pass"] = False
    return out


# ---- the reference AS WRITTEN (oracle/ref_harness.py drives the unmodified src/main.py from baseline/_ref) -------------
_ref_slide = None


def reference_slide():
    """The N=1 bench slide as an OpenSlide duck type for the reference's own code (level 0 only) + its lesion mask."""
    global _ref_slide
    if _ref_slide is None:
        from ss25_hierarchical_multiscale_image_classification_b200.synthetic import SyntheticSlide
        img, msk, _ = build_slab(1, 0, pinned=False)          # msk = the annotation polygons rasterised by Pillow (period_mask)
        _ref_slide = (SyntheticSlide(levels=[img.numpy()], name="tumor_900"), msk.numpy())
        from oracle import ref_harness as rh
        rh.load_reference_main()                            # importing the reference's module is not a timed step either
    return _ref_slide


def reference_available():
    from oracle import ref_harness as rh
    return rh.reference_available()


def reference_as_written_step(png: bool = True):
    """One bounded step of the reference as written: ``extract_patches(level=0, stride=224*REF_STRIDE_MULT)`` -- the
    reference's own stride argument, i.e. every REF_STRIDE_MULT-th column and row of the workload's 224-px candidate
    grid over the WHOLE 16384^2 slide (16 full-size 1792^2 candidates) -- then ``extract_features(level=0)`` reading the
    PNGs back through ``PatchDataset`` + ``DataLoader(batch_size=512, num_workers=8)`` (src/main.py:805-894).
    ``png=False``: ``Image.save`` captured in memory (pure-compute stage 1) and the feature loop replayed in process."""
    import torch
    from oracle import ref_harness as rh
    slide, mask = reference_slide()
    stride = STRIDE * REF_STRIDE_MULT
    n_cand = len(range(0, WIDTH, stride)) * len(range(0, ROWS_PER_GPU, stride))
    if png:
        r = rh.run_reference_as_written(slide, LEVEL, stride=stride, mask_arr=mask)
        surv, s1, s2, names = int(r["n_png"]), r["stage1_s"], r["stage2_s"], r["paths"]
        checksum = float(np.abs(r["features"]).sum())
    else:
        t0 = time.perf_counter()
        saved = rh.run_reference_extract_patches(slide, LEVEL, stride=stride, mask_arr=mask)
        t1 = time.perf_counter()
        torch.manual_seed(0)
        feats = rh.run_reference_features([r[4] for r in saved], None, batch=512)
        t2 = time.perf_counter()
        surv, s1, s2, names, checksum = len(saved), t1 - t0, t2 - t1, [r[0] for r in saved], float(np.abs(feats).sum())
    return {"candidates": n_cand, "survivors": surv, "stage1_s": s1, "stage2_s": s2, "names": names, "feature_checksum": checksum}


def reference_record(step, cores):
    tot = step["stage1_s"] + step["stage2_s"]
    return {"value": round(step["survivors"] / tot, 3), "unit": "patches/s", "cores": cores, "kind": "reference",
            "sample": f"the unmodified reference (baseline/_ref/src/main.py) on the N=1 slide with its own stride argument = "
                      f"{STRIDE * REF_STRIDE_MULT} (every {REF_STRIDE_MULT}-th column and row of the 224-px grid): {step['candidates']} "
                      f"candidates -> {step['survivors']} survivors; extract_patches incl. PNG write {step['stage1_s']:.2f} s (single "
                      f"thread, as written), extract_features incl. PNG decode + Resize via DataLoader(num_workers=8) {step['stage2_s']:.2f} s",
            "candidates_per_s": round(step["candidates"] / tot, 3), "host_cpus": os.cpu_count(),
            "feature_checksum": step["feature_checksum"]}


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path on the box's host cores, each step a bounded
    sample (see reference_as_written_step).  Falls back to the oracle port only if baseline/_ref is absent."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    # torchrun exports OMP_NUM_THREADS=1: the reference arm gets every host core this process may use
    cores = max(1, len(os.sched_getaffinity(0)))
    torch.set_num_threads(cores)
    as_written = reference_available()
    vals, secs, last, extra = [], [], None, {}
    regions = None if as_written else cpu_sample_regions(args.cpu_candidates)
    if as_written:
        reference_slide()                                   # synthetic-data generation is not reference work
    for s in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        if as_written:
            rec = reference_record(reference_as_written_step(png=True), cores)
        else:
            rec, _ = cpu_port_sample(args.cpu_candidates, regions)
        if s >= args.warmup:
            vals.append(rec)
            secs.append(time.perf_counter() - t0)
        last = rec
    if as_written:
        nopng = reference_as_written_step(png=False)
        extra = {"no_png_value": round(nopng["survivors"] / (nopng["stage1_s"] + nopng["stage2_s"]), 3),
                 "no_png_note": f"same sample with Image.save captured in memory and the feature loop replayed in process (no "
                                f"DataLoader workers): stage 1 {nopng['stage1_s']:.2f} s, stage 2 {nopng['stage2_s']:.2f} s"}
    tot_surv = sum(float(v["value"]) for v in vals) / len(vals)
    out = {"impl": "reference", "metric": "patches/sec (tile+mask+ResNet18 features)", "value": round(tot_surv, 3),
           "unit": "patches/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": round(1e3 * sum(secs) / len(secs), 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "u8 + fp32 (CPU)", "data": "synthetic (same slide as the GPU arm; random-init ResNet18 as the reference builds it)",
           "config": {"workload": "configs[1] (bounded sample per step: the reference's extract_patches + extract_features as written, "
                                  f"stride argument {STRIDE * REF_STRIDE_MULT})" if as_written else
                                  "configs[1] (bounded every-k-th-candidate sample per step), CPU port of the reference path",
                      "level": LEVEL, "patch": PATCH, "stride": STRIDE, "width": WIDTH, "rows_per_gpu": ROWS_PER_GPU},
           "cpu_baseline": {**last, "value": round(tot_surv, 3), **extra},
           "e2e": {"value": round(tot_surv, 3), "unit": "patches/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


# ---- BASELINE configs[0]: the whole config on both arms ------------------------------------------------------------------
def run_config0(args):
    """`--config 0`: BASELINE.json configs[0] (SURVEY 8d "C1"): a 4096 x 4096 level-3 image (level 3 of a 32768^2 synthetic
    slide), P = S = 224 -> 19 x 19 = 361 candidates, tissue filter + lesion labels + ResNet18 512-d features.  Small enough
    for the unmodified reference to run the WHOLE config on the host (extract_patches with real PNG writes, then
    extract_features through PatchDataset + DataLoader, src/main.py:609-732, 805-894), so the two arms are on the same
    config, and EVERY survivor is compared: file names (coords + labels) and the 512-d features, computed by our kernels
    from the very weights the reference's random-init ResNet18FeatureExtractor drew (captured by the harness)."""
    import torch
    import __graft_entry__ as ge
    from oracle import ref_harness as rh
    from ss25_hierarchical_multiscale_image_classification_b200 import features, pipeline
    from ss25_hierarchical_multiscale_image_classification_b200.models.resnet import _sequential_to_tv
    from ss25_hierarchical_multiscale_image_classification_b200.synthetic import SyntheticSlide

    ge.build()
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    L, size0 = 3, 32768
    host_threads = max(1, min(16, len(os.sched_getaffinity(0))))
    torch.set_num_threads(host_threads)
    slide = SyntheticSlide(size0, size0, seed=SEED, name="tumor_900")
    img_np, msk_np = slide.level_array(L), slide.lesion_mask(L)
    rh.load_reference_main()
    ref = rh.run_reference_as_written(slide, L, stride=None, mask_arr=msk_np, capture_weights=True)
    ref_s = ref["stage1_s"] + ref["stage2_s"]
    packed = features.pack_resnet18(_sequential_to_tv(ref["weights"]), dev)

    img_h, msk_h = torch.from_numpy(img_np).pin_memory(), torch.from_numpy(msk_np).pin_memory()
    img_d, msk_d = img_h.to(dev), msk_h.to(dev)
    pipe = pipeline.HostPipeline(int(img_h.shape[0]), int(img_h.shape[1]), dev, with_mask=True, num_classes=0)

    def timed(fn):
        for _ in range(max(3, args.warmup)):
            r = fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            r = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps, r

    with ClockSampler(0) as clk:
        ms_res, r = timed(lambda: pipeline.process_level(img_d, msk_d, L, packed))
        ms_e2e, rh_ = timed(lambda: pipeline.process_level_host(img_h, msk_h, L, packed, pipe, groups=2))
    coords, labels, feats = r.coords.cpu().numpy(), r.labels.cpu().numpy(), r.features.float().cpu().numpy()
    ours = {f"{slide.name}_x{int(x)}_y{int(y)}_{'tumor' if int(l) else 'normal'}.png": i for i, ((x, y), l) in enumerate(zip(coords, labels))}
    names_equal = sorted(ours) == sorted(ref["paths"])
    par = {"against": "the unmodified reference on the WHOLE config (every candidate, every survivor), same random-init weights",
           "n_candidates": int(r.candidates), "n_survivors_reference": int(ref["n_png"]), "n_survivors_ours": int(len(coords)),
           "file_names_equal": bool(names_equal)}
    if names_equal and len(coords):
        idx = [ours[p] for p in ref["paths"]]
        g, f = feats[idx].astype(np.float64), ref["features"].astype(np.float64)
        cos = (g * f).sum(1) / (np.linalg.norm(g, axis=1) * np.linalg.norm(f, axis=1))
        maxrel = np.abs(g - f).max(1) / np.abs(f).max(1)
        par.update({"min_cos": round(float(cos.min()), 7), "max_rel": float(f"{maxrel.max():.3e}"),
                    "labels_equal_reference_npy": bool(np.array_equal(labels[idx].astype(np.int64), ref["labels"].astype(np.int64)))})
        par["pass"] = bool(cos.min() >= 0.9995 and maxrel.max() <= 1e-2 and par["labels_equal_reference_npy"])
    else:
        par["pass"] = False
    n = len(coords)
    print(json.dumps({
        "metric": "patches/sec (tile+mask+ResNet18 features)", "value": round(n / (ms_res * 1e-3), 1), "unit": "patches/s", "n_gpus": 1,
        "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": round(ms_res, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8 (tiling/mask, bit-exact) + bf16 tensor-core convs with fp32 accumulate",
        "data": "synthetic (counter-hash slide, the reference's own random-init ResNet18FeatureExtractor weights)",
        "config": {"workload": "configs[0]: 4096x4096 RGB level-3 image, P=S=224 tiling + tissue filter + lesion labels + ResNet18 512-d features; "
                               "the reference batches 512 (src/main.py:46), BASELINE.json says 64: with 116 survivors both are one batch",
                   "level": L, "patch": 224, "stride": 224, "width": int(img_h.shape[1]), "height": int(img_h.shape[0]),
                   "candidates_per_step": int(r.candidates), "survivors_per_step": n,
                   "cache": "the 48 MiB image fits the 126 MB L2: the resident number is an L2-warm number (this config is the reference's CPU timing row, not the roofline workload)"},
        "e2e": {"value": round(n / (ms_e2e * 1e-3), 1), "unit": "patches/s", "ms_per_step": round(ms_e2e, 4),
                "h2d_bytes_per_step": int(img_h.numel() + msk_h.numel()), "d2h_bytes_per_step": int(n * (512 * 4 + 8 + 1))},
        "clocks": clk.summary(), "same_config": True,
        "cpu_baseline": {"value": round(ref["n_png"] / ref_s, 3), "unit": "patches/s", "cores": host_threads, "kind": "reference",
                         "sample": f"the whole config: 361 candidates -> {ref['n_png']} survivors; extract_patches incl. PNG write "
                                   f"{ref['stage1_s']:.2f} s (single thread, as written), extract_features incl. PNG decode via "
                                   f"DataLoader(batch_size=512, num_workers=8) {ref['stage2_s']:.2f} s",
                         "candidates_per_s": round(r.candidates / ref_s, 2), "host_cpus": os.cpu_count()},
        "parity": par}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--chunk", type=int, default=8192, help="patches per ResNet18 chunk")
    ap.add_argument("--cpu-candidates", type=int, default=96, help="candidates in the bounded CPU-baseline sample")
    ap.add_argument("--groups", type=int, default=12, help="row groups of the pipelined host->device upload (e2e leg)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--config", type=int, default=1, choices=[0, 1],
                    help="1 (default): BASELINE configs[1], the bench workload; 0: configs[0] on both arms, whole config")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the patch set of the last timed step (coords, labels, features, logits) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.config != 1 or args.impl != "ours"):
        ap.error("--dump-outputs applies to the default workload of --impl ours")
    if args.config == 0:
        run_config0(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
