"""One level image -> survivors' coordinates, labels, 512-d features and logits, without the PNG round trip.

This is the device-resident composition of the reference's two stages -- ``extract_patches``
(``src/main.py:609-732``) feeding ``extract_features`` (``src/main.py:805-894``) through PNG files -- as
one pass: ``hipac_tile_scan`` writes the normalised bf16 batch that ``hipac_resnet18_forward`` consumes.

``process_level``       inputs already in HBM.
``process_level_host``  inputs in (pinned) host memory: the upload is cut into row groups and overlapped
                        with the tile scan + ResNet18 of the previous group on a second stream, and the
                        results come back into host buffers.  The lesion mask is uploaded sparsely: the host
                        finds its non-zero row blocks (one vectorised max per block, while the image DMA is in
                        flight) and only those travel; the rest of the device mask stays zero.
"""
from __future__ import annotations

from dataclasses import dataclass

import torch

from . import features as _features
from . import _lib
from .preprocessing.tensor_api import (alloc_level_image, extract_patches_enqueue, extract_patches_tensor, grid_shape,
                                       patch_and_stride, upload_level_rows)


@dataclass
class LevelResult:
    coords: torch.Tensor        # int32 [N,2] (x, y) level pixels, reference emission order within each row group
    labels: torch.Tensor        # uint8 [N]
    features: torch.Tensor      # float32 [N,512]
    logits: torch.Tensor | None  # float32 [N,k]
    candidates: int

    def __len__(self):
        return int(self.coords.shape[0])


@dataclass
class PendingLevel:
    """One enqueued tile-scan + ResNet18 pass (a SEGMENT of the exchange step): capacity-sized device tensors plus the
    device-side survivor counter; nothing has been waited for."""
    pend: object                # PendingPatchBatch
    features: torch.Tensor      # float32 [capacity, 512]
    logits: torch.Tensor | None

    @property
    def count(self):
        return self.pend.count

    @property
    def capacity(self):
        return self.pend.capacity


def process_level_enqueue(level_img, lesion_mask, level, packed, stride=None, row_range=None, chunk: int = 8192,
                          mode: str = "auto", tissue=None, tissue_scale: int = 1, min_tissue=0.5, roi=None,
                          roi_y_origin: int = 0, tta: bool = False, stain=None) -> PendingLevel:
    """Enqueue tile scan + ResNet18 of candidate grid rows ``row_range`` without any host wait (the network kernels read
    the survivor count from device memory).  Feed the result to ``sharding.SurvivorExchange.pack``.  ``tissue`` /
    ``tissue_scale`` / ``min_tissue``: the tissue-mask filter, ``roi`` / ``roi_y_origin``: the coarse-level ROI of
    ``extract_patches_enqueue``.  ``tta``: the D4 test-time augmentation of ``features.classify_tensor``.  ``stain``: the
    ``StainNormalizer`` applied to every survivor before the network (see ``extract_patches_enqueue``)."""
    pend = extract_patches_enqueue(level_img, lesion_mask, level, stride=stride, row_range=row_range, layout="s2d16", mode=mode,
                                   tissue=tissue, tissue_scale=tissue_scale, min_tissue=min_tissue, roi=roi, roi_y_origin=roi_y_origin,
                                   stain=stain)
    if packed.num_classes > 0:
        feats, logits = _features.classify_tensor(pend.batch, packed, chunk, count=pend.count, tta=tta)
    else:
        feats, logits = _features.extract_features_tensor(pend.batch, packed, chunk, count=pend.count, tta=tta), None
    return PendingLevel(pend, feats, logits)


def _process_rows(level_img, lesion_mask, level, packed, stride, rows, chunk, mode, tissue=None, tissue_scale=1, min_tissue=0.5,
                  roi=None, roi_y_origin=0, tta=False, stain=None):
    """Tile scan + ResNet18 of one candidate-row group, enqueued back to back: the network kernels take the survivor
    count from device memory (``hipac_resnet18_forward_dcount``), so the host only learns it afterwards, to slice the
    capacity-sized outputs -- while the GPU is already running the network."""
    if _lib.profiling():
        # the per-kernel profiler attributes flops by the host-side patch count: use the host-count path
        pb = extract_patches_tensor(level_img, lesion_mask, level, stride=stride, row_range=rows, layout="s2d16", mode=mode,
                                    tissue=tissue, tissue_scale=tissue_scale, min_tissue=min_tissue, roi=roi, roi_y_origin=roi_y_origin,
                                    stain=stain)
        if packed.num_classes > 0:
            feats, logits = _features.classify_tensor(pb.batch, packed, chunk, tta=tta)
        else:
            feats, logits = _features.extract_features_tensor(pb.batch, packed, chunk, tta=tta), None
        return LevelResult(pb.coords, pb.labels, feats, logits, pb.candidates)
    pend = extract_patches_enqueue(level_img, lesion_mask, level, stride=stride, row_range=rows, layout="s2d16", mode=mode,
                                   tissue=tissue, tissue_scale=tissue_scale, min_tissue=min_tissue, roi=roi, roi_y_origin=roi_y_origin,
                                   stain=stain)
    if packed.num_classes > 0:
        feats, logits = _features.classify_tensor(pend.batch, packed, chunk, count=pend.count, tta=tta)
    else:
        feats, logits = _features.extract_features_tensor(pend.batch, packed, chunk, count=pend.count, tta=tta), None
    pb = pend.resolve()
    n = len(pb)
    return LevelResult(pb.coords, pb.labels, feats[:n], logits[:n] if logits is not None else None, pb.candidates)


def process_level(level_img: torch.Tensor, lesion_mask, level: int, packed: _features.PackedResNet18, stride=None,
                  row_range=None, chunk: int = 8192, mode: str = "auto", max_candidates: int = 16384, tissue=None,
                  tissue_scale: int = 1, min_tissue=0.5, roi=None, roi_y_origin: int = 0, tta: bool = False,
                  stain=None) -> LevelResult:
    """Tile + tissue/lesion mask + ResNet18 features of a level image resident on the GPU.

    ``tissue`` / ``tissue_scale`` / ``min_tissue``: keep the candidates a tissue mask covers (e.g. ``segment_tissue`` of a
    coarser level, see ``extract_patches_enqueue``) instead of applying the ``mean > 240`` rule.

    ``roi`` / ``roi_y_origin``: keep only the candidates inside a coarser level's ``cascade.RoiGrid`` (see
    ``extract_patches_enqueue`` and ``cascade.process_cascade``).

    ``tta``: rotation/flip test-time augmentation in stage 2 (``features.classify_tensor(..., tta=True)``): features and
    logits of every survivor are those of its eight D4 views averaged; coordinates, labels and candidates do not change.

    ``stain``: a ``preprocessing.StainNormalizer`` (Macenko, e.g. from ``estimate_stain`` of the slide's thumbnail): every
    survivor is normalised before ToTensor/Normalize; coordinates, labels and candidates do not change.

    The batch buffer is sized for the worst case (every candidate survives), so levels with more than
    ``max_candidates`` candidates are processed in groups of whole candidate-grid rows (a 100k x 100k level at
    224-px tiles has 200k candidates = 82 GB of batch at once); the result is returned in canonical ``(x, y)``
    order either way."""
    H, W = int(level_img.shape[0]), int(level_img.shape[1])
    P, S = patch_and_stride(level, stride)
    nx, ny_all = grid_shape(W, H, S)
    i0, i1 = (0, ny_all) if row_range is None else (int(row_range[0]), int(row_range[1]))
    rows_per_group = max(1, max_candidates // max(nx, 1))
    tis = dict(tissue=tissue, tissue_scale=tissue_scale, min_tissue=min_tissue, tta=tta, stain=stain)
    if roi is not None:
        tis.update(roi=roi, roi_y_origin=roi_y_origin)
    if i1 - i0 <= rows_per_group:
        return _process_rows(level_img, lesion_mask, level, packed, stride, (i0, i1), chunk, mode, **tis)
    parts = [_process_rows(level_img, lesion_mask, level, packed, stride, (a, min(a + rows_per_group, i1)), chunk, mode, **tis)
             for a in range(i0, i1, rows_per_group)]
    coords = torch.cat([r.coords for r in parts])
    key = coords[:, 0].to(torch.int64) * (1 << 32) + coords[:, 1].to(torch.int64)
    perm = torch.argsort(key, stable=True)
    logits = torch.cat([r.logits for r in parts])[perm] if parts[0].logits is not None else None
    return LevelResult(coords[perm], torch.cat([r.labels for r in parts])[perm], torch.cat([r.features for r in parts])[perm],
                       logits, sum(r.candidates for r in parts))


def exchange_for_level(device, width: int, rows_per_rank: int, stride: int, num_classes: int, max_candidates: int = 16384,
                       with_features: bool = True, group=None):
    """A ``sharding.SurvivorExchange`` sized for ``process_level_exchanged``: every rank tiles at most ``rows_per_rank``
    candidate grid rows of a ``width``-pixel level, in row groups of at most ``max_candidates`` candidates (the batch
    buffer is sized for the worst case: every candidate survives)."""
    from . import sharding
    nx = (width + stride - 1) // stride
    rows_per_group = max(1, min(rows_per_rank, max_candidates // max(nx, 1)))
    n_groups = max(1, (rows_per_rank + rows_per_group - 1) // rows_per_group)
    return sharding.SurvivorExchange(device, nx * rows_per_group, num_classes, nx, stride, segs_per_rank=n_groups, group=group,
                                     with_features=with_features)


def process_level_exchanged(level_img, lesion_mask, level: int, packed: _features.PackedResNet18, exchange, stride=None,
                            row_range=None, y_offset: int = 0, chunk: int = 8192, mode: str = "auto", tissue=None,
                            tissue_scale: int = 1, min_tissue=0.5, roi=None, tta: bool = False, stain=None) -> int:
    """``process_level`` whose result goes straight into the exchange step: the rank's grid rows are cut into the exchange's
    row groups, each group is enqueued (tile scan + ResNet18, survivor count on the device) and packed as one segment, then
    ``exchange.merge()`` is enqueued.  No host wait anywhere; call ``exchange.result()`` for the merged, canonically
    ordered, (with several ranks) all-gathered survivors.  Returns the number of candidates of this rank.

    ``tissue`` is the tissue mask of THIS rank's ``level_img``: a rank whose image starts at level row ``y_offset`` passes
    the rows ``tissue_all[y_offset // tissue_scale:]`` of the whole-slide mask (``y_offset`` a multiple of the scale).
    Every rank segments the same thumbnail with integer arithmetic and one fixed fp64 sequence, so all ranks hold the
    same mask and an N-rank result equals a single-rank one.

    ``roi``: a ``cascade.RoiGrid`` of a coarser level over the WHOLE slide (every rank builds the same one from the
    exchanged coarse result); the rank's slab is placed in it by ``y_offset``.  ``tta``, ``stain``: as in ``process_level``
    (every rank estimates the same stain from the same thumbnail, bit for bit)."""
    H, W = int(level_img.shape[0]), int(level_img.shape[1])
    P, S = patch_and_stride(level, stride)
    nx, ny_all = grid_shape(W, H, S)
    i0, i1 = (0, ny_all) if row_range is None else (int(row_range[0]), int(row_range[1]))
    rows_per_group = max(1, exchange.cap // max(nx, 1))
    if (i1 - i0 + rows_per_group - 1) // rows_per_group > exchange.spr:
        raise ValueError(f"{i1 - i0} grid rows need more than the exchange's {exchange.spr} segments of {rows_per_group} rows")
    g = 0
    for a in range(i0, i1, rows_per_group):
        seg = process_level_enqueue(level_img, lesion_mask, level, packed, stride=stride, row_range=(a, min(a + rows_per_group, i1)),
                                    chunk=chunk, mode=mode, tissue=tissue, tissue_scale=tissue_scale, min_tissue=min_tissue,
                                    roi=roi, roi_y_origin=y_offset, tta=tta, stain=stain)
        exchange.pack(g, seg.pend.coords, seg.pend.labels, seg.features, seg.logits, seg.count, y_offset=y_offset)
        g += 1
    for e in range(g, exchange.spr):
        exchange.pack_empty(e)
    exchange.merge()
    return nx * (i1 - i0)


class HostPipeline:
    """Reusable device/host staging buffers + copy stream for ``process_level_host``."""

    MASK_BLOCK_ROWS = 32     # granularity of the sparse lesion-mask upload: blocks of whole rows, so that every copy is
                             # one contiguous pinned range (a column-narrowed rectangle would save another ~35 MB here,
                             # but PyTorch stages non-contiguous host views through a synchronous temporary: measured slower)

    def __init__(self, height: int, width: int, device, with_mask: bool = True, capacity: int | None = None,
                 num_classes: int = 2, sparse_mask: bool = True):
        self.device = torch.device(device)
        # device staging with 16-byte row pitch (the streaming pass's precondition, whatever the width)
        self.img = alloc_level_image(height, width, self.device)
        # the device mask is kept all-zero outside the rectangles uploaded by the current step
        self.mask = alloc_level_image(height, width, self.device, channels=1) if with_mask else None
        if self.mask is not None:
            self.mask.zero_()
        self.copy_stream = torch.cuda.Stream(self.device)
        self.capacity = capacity
        self.num_classes = num_classes
        self.sparse_mask = sparse_mask
        self._dirty: list[tuple[int, int, int, int]] = []   # mask rectangles (r0, r1, c0, c1) holding data of the previous step
        self.last_h2d_bytes = 0
        self._host = None

    def begin_step(self):
        """Re-zero the mask rectangles the previous step uploaded (copy stream) and reset the byte counter."""
        for r0, r1, c0, c1 in self._dirty:
            self.mask[r0:r1, c0:c1].zero_()
        self._dirty = []
        self.last_h2d_bytes = 0

    def _upload_rect(self, mask_host, r0, r1, c0, c1):
        if self.mask.is_cuda and c0 == 0 and c1 == int(self.mask.shape[1]):
            upload_level_rows(self.mask, mask_host[r0:r1], r0)          # whole rows: one 2-D DMA on the current stream
        else:
            self.mask[r0:r1, c0:c1].copy_(mask_host[r0:r1, c0:c1], non_blocking=True)
        self._dirty.append((r0, r1, c0, c1))
        self.last_h2d_bytes += (r1 - r0) * (c1 - c0)

    def upload_mask_rows(self, mask_host: torch.Tensor, r0: int, r1: int):
        """Queue the upload of mask rows [r0, r1) on the current (copy) stream.  Sparse mode: one max per block of
        MASK_BLOCK_ROWS rows on the host (contiguous, memory-bandwidth bound) decides which blocks are non-zero; every
        run of non-zero blocks is one copy, the rest is already zero on the device."""
        if r1 <= r0:
            return
        W = int(mask_host.shape[1])
        R = self.MASK_BLOCK_ROWS
        if not self.sparse_mask or not mask_host.is_contiguous():
            self._upload_rect(mask_host, r0, r1, 0, W)
            return
        nfull = (r1 - r0) // R
        rowflag = []
        if nfull:
            rowflag = mask_host[r0:r0 + nfull * R].view(nfull, R * W).amax(dim=1).ne(0).tolist()
        if r0 + nfull * R < r1:
            rowflag.append(bool(mask_host[r0 + nfull * R:r1].amax().item() != 0))
        b, nb = 0, len(rowflag)
        while b < nb:
            if not rowflag[b]:
                b += 1
                continue
            e = b
            while e < nb and rowflag[e]:
                e += 1
            self._upload_rect(mask_host, r0 + b * R, min(r0 + e * R, r1), 0, W)
            b = e

    def host_buffers(self, cap: int):
        if self._host is None or self._host[0].shape[0] < cap:
            self._host = (torch.empty((cap, 2), dtype=torch.int32).pin_memory(),
                          torch.empty((cap,), dtype=torch.uint8).pin_memory(),
                          torch.empty((cap, 512), dtype=torch.float32).pin_memory(),
                          torch.empty((cap, max(self.num_classes, 1)), dtype=torch.float32).pin_memory())
        return self._host


def upload_group_bounds(i0: int, i1: int, groups: int):
    """Candidate-row boundaries of the upload groups.  Tapered: the network of the LAST group cannot start before the
    whole image has landed, so the last group is the exposed tail of the pipeline and gets the smallest share (the
    taper is mild, largest / smallest = 2.5, so the first group does not delay the start of compute much)."""
    groups = max(1, min(groups, i1 - i0))
    w = [1.0 + 1.5 * (groups - 1 - g) / max(groups - 1, 1) for g in range(groups)]
    acc, tot, bounds = 0.0, sum(w), [i0]
    for g in range(groups):
        acc += w[g]
        bounds.append(max(bounds[-1], min(i1, i0 + int(round((i1 - i0) * acc / tot)))))
    bounds[-1] = i1
    return bounds


def process_level_host(level_img_host: torch.Tensor, mask_host, level: int, packed: _features.PackedResNet18,
                       pipe: HostPipeline, stride=None, row_range=None, groups: int = 4, chunk: int = 8192,
                       exchange=None, y_offset: int = 0, polygon_window=None) -> LevelResult:
    """Same as ``process_level`` for HOST inputs; returns HOST tensors (pinned views, valid until the next call).

    ``mask_host`` is the rasterised lesion mask (uint8 ``[H, W]`` host tensor, uploaded sparsely) OR a
    ``preprocessing.lesion_mask.PolygonSet``: the annotation polygons themselves, in which case the mask is rasterised on
    the GPU into the staging buffer (``polygon_window = (level_height, y_begin)`` places this slab inside the level the
    vertices refer to; default: the slab is the whole level) and no mask byte crosses PCIe.

    The candidate grid rows are cut into ``groups`` contiguous groups.  All uploads are queued in row order
    on the copy stream; group ``g`` is scanned as soon as the rows it touches (its own + the
    ``patch - stride`` halo) have landed, while the rest of the image is still in flight.

    ``exchange``: a ``sharding.SurvivorExchange`` with ``segs_per_rank >= groups``.  Every group then becomes one segment
    of the exchange step (packed on the device, no per-group host wait), the merged -- with several ranks: all-gathered --
    canonically ordered result is what comes back to the host, with ``y_offset`` added to this rank's y coordinates."""
    H, W = int(level_img_host.shape[0]), int(level_img_host.shape[1])
    P, S = patch_and_stride(level, stride)
    nx, ny_all = grid_shape(W, H, S)
    i0, i1 = (0, ny_all) if row_range is None else row_range
    bounds = upload_group_bounds(i0, i1, groups)
    groups = len(bounds) - 1
    dev = pipe.device
    main = torch.cuda.current_stream(dev)
    events, done_rows = [], i0 * S
    polys = mask_host if (mask_host is not None and not torch.is_tensor(mask_host)) else None
    if polys is not None:
        from .preprocessing.lesion_mask import rasterize_polygons
        if pipe.mask is None:
            raise ValueError("the pipeline was built without a mask buffer")
        level_h, y_begin = polygon_window if polygon_window is not None else (H, 0)
        # the previous step's kernels (same stream) are done with the buffer; the fill clears the slab's rows first
        rasterize_polygons(polys, W, int(level_h), y_begin=int(y_begin), n_rows=H, out=pipe.mask, check=False)
        pipe._dirty = []
        mask_host = None
    with torch.cuda.stream(pipe.copy_stream):
        pipe.copy_stream.wait_stream(main)          # previous step's kernels are done with the staging buffers
        if pipe.mask is not None and polys is None:
            pipe.begin_step()
        elif polys is not None:
            pipe.last_h2d_bytes = 0
        for g in range(groups):
            need = min(H, (bounds[g + 1] - 1) * S + P + 8) if bounds[g + 1] > bounds[g] else done_rows
            if need > done_rows:
                pipe.last_h2d_bytes += upload_level_rows(pipe.img, level_img_host[done_rows:need], done_rows)
                if pipe.mask is not None and mask_host is not None:
                    pipe.upload_mask_rows(mask_host, done_rows, need)   # host scan overlaps the image DMA just queued
                done_rows = need
            ev = torch.cuda.Event()
            ev.record(pipe.copy_stream)
            events.append(ev)
    mask_dev = pipe.mask if (pipe.mask is not None and (mask_host is not None or polys is not None)) else None
    if exchange is not None:
        if exchange.spr < groups:
            raise ValueError(f"exchange has {exchange.spr} segments per rank, {groups} row groups need one each")
        n_cand = 0
        for g in range(exchange.spr):
            if g >= groups or bounds[g + 1] <= bounds[g]:
                exchange.pack_empty(g)
                continue
            main.wait_event(events[g])
            seg = process_level_enqueue(pipe.img, mask_dev, level, packed, stride=stride, row_range=(bounds[g], bounds[g + 1]), chunk=chunk)
            exchange.pack(g, seg.pend.coords, seg.pend.labels, seg.features, seg.logits, seg.count, y_offset=y_offset)
            n_cand += nx * (bounds[g + 1] - bounds[g])
        exchange.merge()
        res = exchange.result()
        n = int(res["coords"].shape[0])
        h_coords, h_labels, h_feats, h_logits = pipe.host_buffers(max(n, 1))
        h_coords[:n].copy_(res["coords"], non_blocking=True)
        h_labels[:n].copy_(res["labels"], non_blocking=True)
        h_feats[:n].copy_(res["features"], non_blocking=True)
        if "logits" in res:
            h_logits[:n].copy_(res["logits"], non_blocking=True)
        main.synchronize()
        return LevelResult(h_coords[:n], h_labels[:n], h_feats[:n], h_logits[:n] if packed.num_classes > 0 else None, n_cand)
    cap = nx * (i1 - i0)
    h_coords, h_labels, h_feats, h_logits = pipe.host_buffers(cap)
    n_total, n_cand = 0, 0
    for g in range(groups):
        if bounds[g + 1] <= bounds[g]:
            continue
        main.wait_event(events[g])
        r = process_level(pipe.img, mask_dev, level, packed, stride=stride, row_range=(bounds[g], bounds[g + 1]), chunk=chunk)
        n = len(r)
        h_coords[n_total:n_total + n].copy_(r.coords, non_blocking=True)
        h_labels[n_total:n_total + n].copy_(r.labels, non_blocking=True)
        h_feats[n_total:n_total + n].copy_(r.features, non_blocking=True)
        if r.logits is not None:
            h_logits[n_total:n_total + n].copy_(r.logits, non_blocking=True)
        n_total += n
        n_cand += r.candidates
    main.synchronize()
    return LevelResult(h_coords[:n_total], h_labels[:n_total], h_feats[:n_total],
                       h_logits[:n_total] if packed.num_classes > 0 else None, n_cand)
