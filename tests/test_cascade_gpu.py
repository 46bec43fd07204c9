"""Coarse-to-fine cascade on the GPU, bit for bit: the ROI grid kernels against oracle/cascade.py, ROI-filtered scans against
the unfiltered scan restricted by the oracle, process_cascade against the full process_level restricted, and emulated
multi-rank runs against the single-rank cascade."""
import math
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import cascade as oc
from oracle import hipac_oracle as orc

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PATCH = {0: 1792, 1: 896, 2: 448, 3: 224}


@pytest.fixture(scope="module")
def slide():
    from ss25_hierarchical_multiscale_image_classification_b200.synthetic import SyntheticSlide
    s = SyntheticSlide(7168, 5888, seed=17)            # level 3: 896 x 736
    return s, {L: (s.level_array(L), s.lesion_mask(L)) for L in range(4)}


@pytest.fixture(scope="module")
def packed():
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    return features.pack_resnet18(orc.make_resnet18(seed=0, classifier=True).state_dict(), "cuda")


def _grid_dims(w, h, s):
    return -(-w // s), -(-h // s)


def _random_roi(rng, level, w, h, stride, frac, dilate):
    """An oracle ROI over the candidate grid of a (w x h) level image from random scores, and the same grid as an RoiGrid."""
    from ss25_hierarchical_multiscale_image_classification_b200.cascade import RoiGrid
    nx, ny = _grid_dims(w, h, stride)
    cc = np.array([(i * stride, j * stride) for i in range(nx) for j in range(ny)], np.int32)
    scores = rng.standard_normal(len(cc)).astype(np.float32)
    thr = np.quantile(scores, 1 - frac)
    grid = oc.roi_grid(cc, scores, thr, stride, nx, ny, dilate)
    roi = oc.Roi(grid, level, stride, PATCH[level])
    return roi, RoiGrid(torch.from_numpy(grid).cuda(), level, stride, PATCH[level], nx, ny)


def _scan(img, mask, level, stride=None, **kw):
    from ss25_hierarchical_multiscale_image_classification_b200.preprocessing import extract_patches_tensor
    return extract_patches_tensor(img, mask, level, stride=stride, want_u8=True, **kw)


def _assert_restricted(got, ref, keep, what):
    idx = torch.from_numpy(np.nonzero(keep)[0]).cuda()
    assert torch.equal(got.coords, ref.coords[idx]), what
    assert torch.equal(got.labels, ref.labels[idx]), what
    assert torch.equal(got.images_u8, ref.images_u8[idx]), what
    assert torch.equal(got.batch.view(torch.int16), ref.batch[idx].view(torch.int16)), what
    assert got.candidates == ref.candidates, what


# ---------------------------------------------------------------------------------------------------------------------
# 1. hipac_roi_grid
# ---------------------------------------------------------------------------------------------------------------------
def test_roi_grid_kernels_equal_oracle():
    from ss25_hierarchical_multiscale_image_classification_b200.cascade import roi_grid
    rng = np.random.default_rng(5)
    for (w, h, s) in ((896, 736, 224), (2048, 2048, 224), (3001, 517, 448), (224, 224, 224)):
        nx, ny = _grid_dims(w, h, s)
        cand = np.array([(i * s, j * s) for i in range(nx) for j in range(ny)], np.int32)
        sel = cand[rng.random(len(cand)) < 0.6]
        n = len(sel)
        scores = rng.standard_normal(n).astype(np.float32)
        d_c = torch.from_numpy(sel).cuda().reshape(-1, 2)
        d_s = torch.from_numpy(scores).cuda()
        level = 3 if s == 224 else 2
        for thr in (0.3, -0.5, math.inf, -math.inf):
            for dilate in (0, 1, 2):
                for cnt in sorted({0, n // 2, n, n + 5}):
                    count = torch.tensor([cnt, 0], dtype=torch.int32, device="cuda")
                    r = roi_grid(d_c, d_s, level, w, h, stride=s, threshold=thr, dilate=dilate, count=count)
                    k = min(cnt, n)
                    want = oc.roi_grid(sel[:k], scores[:k], thr, s, nx, ny, dilate)
                    assert (r.nx, r.ny, r.stride, r.patch, r.level) == (nx, ny, s, PATCH[level], level)
                    assert np.array_equal(r.grid.cpu().numpy(), want), (w, h, thr, dilate, cnt)
        # count on the host side (None): every row
        r = roi_grid(d_c, d_s, 3, w, h, stride=s, threshold=0.0)
        assert np.array_equal(r.grid.cpu().numpy(), oc.roi_grid(sel, scores, 0.0, s, nx, ny))


# ---------------------------------------------------------------------------------------------------------------------
# 2. ROI-filtered scans = unfiltered scan restricted by the oracle
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lc,lf", [(3, 0), (3, 1), (2, 0)])
@pytest.mark.parametrize("stride_kind", ["cli", "nonoverlap"])
def test_filtered_scan_equals_restricted_scan(slide, lc, lf, stride_kind):
    from ss25_hierarchical_multiscale_image_classification_b200.preprocessing import segment_tissue
    s, lv = slide
    rng = np.random.default_rng(lc * 10 + lf)
    sc = 224 if stride_kind == "cli" else PATCH[lc]
    sf = None if stride_kind == "cli" else PATCH[lf]
    hc, wc = lv[lc][0].shape[:2]
    img, lmask = lv[lf]
    d_img, d_mask = torch.from_numpy(img).cuda(), torch.from_numpy(lmask).cuda()
    roi, g = _random_roi(rng, lc, wc, hc, sc, 0.15, 0)
    for mode in ("auto", "direct", "fused", "fused_legacy"):
        ref = _scan(d_img, d_mask, lf, sf, mode=mode)
        keep = oc.roi_mask(ref.coords.cpu().numpy(), lf, roi, stride=sf)
        got = _scan(d_img, d_mask, lf, sf, mode=mode, roi=g)
        _assert_restricted(got, ref, keep, (lc, lf, stride_kind, mode))
        assert 0 < len(got) < len(ref)
    # without a lesion mask
    ref = _scan(d_img, None, lf, sf)
    got = _scan(d_img, None, lf, sf, roi=g)
    _assert_restricted(got, ref, oc.roi_mask(ref.coords.cpu().numpy(), lf, roi, stride=sf), "no lesion mask")
    # combined with the tissue-mask filter (a mask of the level-3 thumbnail)
    tissue = segment_tissue(torch.from_numpy(lv[3][0]).cuda())[0]
    m = 1 << (3 - lf)
    for mode in ("auto", "direct"):
        ref = _scan(d_img, d_mask, lf, sf, mode=mode, tissue=tissue, tissue_scale=m)
        got = _scan(d_img, d_mask, lf, sf, mode=mode, tissue=tissue, tissue_scale=m, roi=g)
        _assert_restricted(got, ref, oc.roi_mask(ref.coords.cpu().numpy(), lf, roi, stride=sf), ("tissue", mode))


def test_row_ranges_and_slab_with_y_origin(slide):
    s, lv = slide
    rng = np.random.default_rng(77)
    lc, lf, S = 3, 0, 224
    hc, wc = lv[lc][0].shape[:2]
    img, lmask = lv[lf]
    d_img, d_mask = torch.from_numpy(img).cuda(), torch.from_numpy(lmask).cuda()
    roi, g = _random_roi(rng, lc, wc, hc, 224, 0.4, 0)
    full = _scan(d_img, d_mask, lf, roi=g)
    fc = full.coords.cpu().numpy()
    nx, ny = _grid_dims(img.shape[1], img.shape[0], S)
    for mode in ("auto", "direct"):
        for a, b in ((0, 5), (7, 19), (ny - 3, ny), (4, 4)):
            got = _scan(d_img, d_mask, lf, mode=mode, row_range=(a, b), roi=g)
            sel = (fc[:, 1] // S >= a) & (fc[:, 1] // S < b)
            idx = torch.from_numpy(np.nonzero(sel)[0]).cuda()
            assert torch.equal(got.coords, full.coords[idx]) and torch.equal(got.batch.view(torch.int16), full.batch[idx].view(torch.int16))
            assert torch.equal(got.labels, full.labels[idx]) and got.candidates == nx * (b - a)
        # a slab starting at grid row k holds the rows [k*S, H): its candidates, shifted by the origin, are the full ones
        for k in (3, 11):
            y0 = k * S
            got = _scan(d_img[y0:], d_mask[y0:], lf, mode=mode, roi=g, roi_y_origin=y0)
            sel = fc[:, 1] >= y0
            idx = torch.from_numpy(np.nonzero(sel)[0]).cuda()
            shift = torch.tensor([0, y0], dtype=torch.int32, device="cuda")
            assert torch.equal(got.coords + shift, full.coords[idx]), (mode, k)
            assert torch.equal(got.images_u8, full.images_u8[idx]) and torch.equal(got.labels, full.labels[idx])
            # without the origin the same slab is tested against the wrong cells
            wrong = _scan(d_img[y0:], d_mask[y0:], lf, mode=mode, roi=g)
            assert not torch.equal(wrong.coords, got.coords)


# ---------------------------------------------------------------------------------------------------------------------
# 3. empty and full ROI; launch count; argument errors
# ---------------------------------------------------------------------------------------------------------------------
def test_empty_and_full_roi(slide):
    from ss25_hierarchical_multiscale_image_classification_b200 import _lib
    from ss25_hierarchical_multiscale_image_classification_b200.cascade import RoiGrid
    s, lv = slide
    img, lmask = lv[1]
    d_img, d_mask = torch.from_numpy(img).cuda(), torch.from_numpy(lmask).cuda()
    hc, wc = lv[3][0].shape[:2]
    nx, ny = _grid_dims(wc, hc, 224)
    empty = RoiGrid(torch.zeros((ny, nx), dtype=torch.uint8, device="cuda"), 3, 224, 224, nx, ny)
    full_roi = RoiGrid(torch.ones((ny, nx), dtype=torch.uint8, device="cuda"), 3, 224, 224, nx, ny)
    l = _lib.lib()
    for mode in ("auto", "direct", "fused_legacy"):
        ref = _scan(d_img, d_mask, 1, mode=mode)
        e = _scan(d_img, d_mask, 1, mode=mode, roi=empty)
        assert len(e) == 0 and e.candidates == ref.candidates
        f = _scan(d_img, d_mask, 1, mode=mode, roi=full_roi)
        _assert_restricted(f, ref, np.ones(len(ref), bool), mode)
        torch.cuda.synchronize()
        l.hipac_launch_count(1)
        _scan(d_img, d_mask, 1, mode=mode)
        n_plain = l.hipac_launch_count(1)
        _scan(d_img, d_mask, 1, mode=mode, roi=full_roi)
        assert l.hipac_launch_count(1) == n_plain + 1          # the ROI adds exactly k_roi_flags


def test_python_argument_errors(slide):
    from ss25_hierarchical_multiscale_image_classification_b200.cascade import RoiGrid, process_cascade, roi_grid
    s, lv = slide
    d_img = torch.from_numpy(lv[2][0]).cuda()
    g = RoiGrid(torch.ones((4, 4), dtype=torch.uint8, device="cuda"), 3, 224, 224, 4, 4)
    with pytest.raises(ValueError, match="keep_all"):
        _scan(d_img, None, 2, roi=g, keep_all=True)
    for lvl in (2, 1):
        bad = RoiGrid(g.grid, lvl, 224, PATCH[lvl], 4, 4)
        with pytest.raises(ValueError, match="coarser"):
            _scan(d_img, None, 2, roi=bad)
    with pytest.raises(ValueError):
        _scan(d_img, None, 2, roi=RoiGrid(g.grid, 3, 224, 224, 5, 4))        # shape mismatch
    with pytest.raises(RuntimeError, match="roi_stride"):
        _scan(d_img, None, 2, roi=RoiGrid(g.grid, 3, 0, 224, 4, 4))
    c = torch.zeros((3, 2), dtype=torch.int32, device="cuda")
    with pytest.raises(ValueError):
        roi_grid(c, torch.zeros(3, device="cuda"), 3, 896, 736, dilate=-1)
    with pytest.raises(ValueError):
        process_cascade({}, None, order=(0, 3))


# ---------------------------------------------------------------------------------------------------------------------
# 4. process_cascade = full process_level restricted
# ---------------------------------------------------------------------------------------------------------------------
def _levels_on_device(lv, levels):
    return {L: (torch.from_numpy(lv[L][0]).cuda(), torch.from_numpy(lv[L][1]).cuda()) for L in levels}


def _oracle_roi_of(result, level, w, h, theta, dilate):
    from ss25_hierarchical_multiscale_image_classification_b200.cascade import tumor_margin
    nx, ny = _grid_dims(w, h, 224)
    grid = oc.roi_grid(result.coords.cpu().numpy(), tumor_margin(result.logits).cpu().numpy(), theta, 224, nx, ny, dilate)
    return oc.Roi(grid, level, 224, PATCH[level])


def _assert_level_restricted(got, full, keep, what):
    idx = torch.from_numpy(np.nonzero(keep)[0]).cuda()
    for k in ("coords", "labels", "features", "logits"):
        a, b = getattr(got, k), getattr(full, k)[idx]
        assert a.shape == b.shape and torch.equal(a.view(torch.int32) if a.dtype == torch.float32 else a,
                                                  b.view(torch.int32) if b.dtype == torch.float32 else b), (what, k)
    assert got.candidates == full.candidates, what


def _median_tau(result):
    return 1.0 / (1.0 + math.exp(-_median_margin(result)))


def _median_margin(result):
    from ss25_hierarchical_multiscale_image_classification_b200.cascade import tumor_margin
    return float(np.median(tumor_margin(result.logits).cpu().numpy()))


def _splitting_tau(coarse, fine, level, w, h, fine_level, dilate):
    """A tau whose ROI keeps some but not all of ``fine``'s candidates: the positives are the top k coarse margins, k halved
    from n/2 until the dilated ROI leaves part of the fine level out (a 4 x 4 coarse grid dilated by one cell covers it
    whole at the median)."""
    from ss25_hierarchical_multiscale_image_classification_b200.cascade import threshold_of, tumor_margin
    m = np.sort(tumor_margin(coarse.logits).cpu().numpy().astype(np.float64))[::-1]
    k = len(m) // 2
    while k >= 1:
        if m[k - 1] > m[k]:
            tau = 1.0 / (1.0 + math.exp(-0.5 * (m[k - 1] + m[k])))
            keep = oc.roi_mask(fine.coords.cpu().numpy(), fine_level, _oracle_roi_of(coarse, level, w, h, threshold_of(tau), dilate))
            if 0 < keep.sum() < len(keep):
                return tau
        k //= 2
    raise AssertionError("no threshold splits the fine level")


@pytest.mark.parametrize("order,dilate", [((3, 0), 0), ((3, 0), 1), ((3, 1, 0), 0)])
def test_process_cascade_equals_restricted_full_levels(slide, packed, order, dilate):
    from ss25_hierarchical_multiscale_image_classification_b200 import features, pipeline
    from ss25_hierarchical_multiscale_image_classification_b200.cascade import process_cascade, threshold_of
    s, lv = slide
    levels = _levels_on_device(lv, order)
    nets = {L: packed for L in order}
    full = {L: pipeline.process_level(*levels[L], L, packed) for L in order}
    h0, w0 = lv[order[0]][0].shape[:2]
    tau = _splitting_tau(full[order[0]], full[order[1]], order[0], w0, h0, order[1], dilate)
    theta = threshold_of(tau)
    for up, L, down in zip(order, order[1:-1], order[2:]):
        # a level-specific head: the same network with the tumour bias moved so that the one tau also splits the next level
        # (the threshold that splits it, taken over this level's candidates inside the ROI above, moves onto logit(tau))
        hu, wu = lv[up][0].shape[:2]
        keep = oc.roi_mask(full[L].coords.cpu().numpy(), L, _oracle_roi_of(full[up], up, wu, hu, theta, dilate))
        idx = torch.from_numpy(np.nonzero(keep)[0]).cuda()
        inside = SimpleNamespace(coords=full[L].coords[idx], logits=full[L].logits[idx])
        hl, wl = lv[L][0].shape[:2]
        tau_l = _splitting_tau(inside, full[down], L, wl, hl, down, dilate)
        sd = orc.make_resnet18(seed=0, classifier=True).state_dict()
        sd["fc.bias"] = sd["fc.bias"].clone()
        sd["fc.bias"][1] += math.log(tau / (1 - tau)) - math.log(tau_l / (1 - tau_l))
        nets[L] = features.pack_resnet18(sd, "cuda")
        full[L] = pipeline.process_level(*levels[L], L, nets[L])
    res = process_cascade(levels, nets, order=order, tau=tau, dilate=dilate)
    assert set(res) == set(order)
    _assert_level_restricted(res[order[0]], full[order[0]], np.ones(len(full[order[0]]), bool), "coarse")
    for prev, L in zip(order, order[1:]):
        h, w = lv[prev][0].shape[:2]
        roi = _oracle_roi_of(res[prev], prev, w, h, theta, dilate)
        keep = oc.roi_mask(full[L].coords.cpu().numpy(), L, roi)
        assert 0 < keep.sum() < len(keep), (order, L, keep.sum())
        _assert_level_restricted(res[L], full[L], keep, (order, L))


def test_lesion_guided_roi(slide, packed):
    """labels.float() >= 0.5: tile level 0 only around the coarse patches that carry a lesion label."""
    from ss25_hierarchical_multiscale_image_classification_b200 import pipeline
    from ss25_hierarchical_multiscale_image_classification_b200.cascade import roi_grid
    s, lv = slide
    levels = _levels_on_device(lv, (3, 0))
    coarse = pipeline.process_level(*levels[3], 3, packed)
    assert int(coarse.labels.sum()) > 0
    h, w = lv[3][0].shape[:2]
    g = roi_grid(coarse.coords, coarse.labels.float(), 3, w, h, threshold=0.5)
    fine = pipeline.process_level(*levels[0], 0, packed, roi=g)
    full = pipeline.process_level(*levels[0], 0, packed)
    nx, ny = _grid_dims(w, h, 224)
    roi = oc.Roi(oc.roi_grid(coarse.coords.cpu().numpy(), coarse.labels.cpu().numpy().astype(np.float32), 0.5, 224, nx, ny), 3, 224, 224)
    keep = oc.roi_mask(full.coords.cpu().numpy(), 0, roi)
    _assert_level_restricted(fine, full, keep, "lesion-guided")
    assert int(fine.labels.sum()) == int(full.labels.sum())      # every tumour-labelled fine patch lies under a labelled coarse one


# ---------------------------------------------------------------------------------------------------------------------
# 5. emulated ranks: row shards through SurvivorExchange = single-rank cascade
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, 4])
def test_emulated_ranks_equal_single_rank_cascade(slide, packed, world):
    from ss25_hierarchical_multiscale_image_classification_b200 import pipeline, sharding
    from ss25_hierarchical_multiscale_image_classification_b200.cascade import (process_cascade, roi_grid, threshold_of,
                                                                                tumor_margin)
    s, lv = slide
    levels = _levels_on_device(lv, (3, 0))
    tau = _median_tau(pipeline.process_level(*levels[3], 3, packed))
    single = process_cascade(levels, packed, order=(3, 0), tau=tau, dilate=1)
    # coarse level: every rank tiles its row shard, the exchange delivers the whole-slide result to every rank
    img3, m3 = levels[3]
    h3, w3 = int(img3.shape[0]), int(img3.shape[1])
    nx3, ny3 = _grid_dims(w3, h3, 224)
    shards = [sharding.shard_rows(ny3, world, r) for r in range(world)]
    xc = sharding.SurvivorExchange("cuda", nx3 * max(b - a for a, b in shards), 2, nx3, 224, segs_per_rank=world)
    for r, (i0, i1) in enumerate(shards):
        y0, y1 = sharding.slab_rows(i0, i1, 224, 224, h3)
        seg = pipeline.process_level_enqueue(img3[y0:y1], m3[y0:y1], 3, packed, row_range=(0, i1 - i0))
        xc.pack(r, seg.pend.coords, seg.pend.labels, seg.features, seg.logits, seg.count, y_offset=y0)
    xc.merge()
    coarse = xc.result()
    for k in ("coords", "labels", "features", "logits"):
        assert torch.equal(coarse[k], getattr(single[3], k)), k
    g = roi_grid(coarse["coords"], tumor_margin(coarse["logits"]), 3, w3, h3, threshold=threshold_of(tau), dilate=1)
    # fine level: each rank holds the slab of its grid rows and places it in the ROI by its y offset
    img0, m0 = levels[0]
    h0, w0 = int(img0.shape[0]), int(img0.shape[1])
    _, ny0 = _grid_dims(w0, h0, 224)
    parts = []
    for r in range(world):
        i0, i1 = sharding.shard_rows(ny0, world, r)
        y0, y1 = sharding.slab_rows(i0, i1, 224, 1792, h0)
        x = pipeline.exchange_for_level("cuda", w0, i1 - i0, 224, 2, max_candidates=4 * ((w0 + 223) // 224))
        n_cand = pipeline.process_level_exchanged(img0[y0:y1], m0[y0:y1], 0, packed, x, row_range=(0, i1 - i0), y_offset=y0, roi=g)
        assert n_cand == ((w0 + 223) // 224) * (i1 - i0)
        parts.append({k: v.clone() for k, v in x.result().items()})
    merged = {k: torch.cat([p[k] for p in parts]) for k in parts[0]}
    perm = sharding.canonical_order(merged["coords"])
    fine = single[0]
    assert 0 < len(fine) < fine.candidates
    for k in ("coords", "labels", "features", "logits"):
        assert torch.equal(merged[k][perm], getattr(fine, k)), k


# ---------------------------------------------------------------------------------------------------------------------
# 6. the new kernels under the bounds-checking library
# ---------------------------------------------------------------------------------------------------------------------
DBG_SCRIPT = r"""
import numpy as np, torch, sys
sys.path.insert(0, %r)
from oracle import cascade as oc
from ss25_hierarchical_multiscale_image_classification_b200 import _lib
from ss25_hierarchical_multiscale_image_classification_b200.cascade import RoiGrid, roi_grid
from ss25_hierarchical_multiscale_image_classification_b200.preprocessing import extract_patches_tensor
assert _lib.lib()._name.endswith("libhipac_b200_dbg.so"), _lib.lib()._name
rng = np.random.default_rng(8)
# ROI grid: dilation at every border, count above the capacity
w3, h3 = 1117, 903
nx, ny = (w3 + 223) // 224, (h3 + 223) // 224
cc = np.array([(i * 224, j * 224) for i in range(nx) for j in range(ny)], np.int32)
sc = rng.standard_normal(len(cc)).astype(np.float32)
for dilate in (0, 2, 7):
    g = roi_grid(torch.from_numpy(cc).cuda(), torch.from_numpy(sc).cuda(), 3, w3, h3, threshold=0.8, dilate=dilate,
                 count=torch.tensor([len(cc) + 9, 0], dtype=torch.int32, device="cuda"))
    assert np.array_equal(g.grid.cpu().numpy(), oc.roi_grid(cc, sc, 0.8, 224, nx, ny, dilate))
roi = oc.Roi(oc.roi_grid(cc, sc, 0.5, 224, nx, ny, 0), 3, 224, 224)
g = RoiGrid(torch.from_numpy(roi.grid).cuda(), 3, 224, 224, nx, ny)
# fine level 1 (P = 896): footprints past the right and bottom edges of the coarse grid, row ranges, a slab origin
img = rng.integers(0, 200, (h3 * 4 + 5, w3 * 4 + 3, 3), dtype=np.uint8)
d = torch.from_numpy(img).cuda()
for mode in ("direct", "auto", "fused_legacy"):
    for rr, y0 in ((None, 0), ((3, 9), 0), (None, 224 * 6)):
        pb = extract_patches_tensor(d[y0:], None, 1, mode=mode, row_range=rr, roi=g, roi_y_origin=y0)
        ref = extract_patches_tensor(d[y0:], None, 1, mode=mode, row_range=rr, layout=None)
        keep = oc.roi_mask(ref.coords.cpu().numpy(), 1, roi, y_origin=y0)
        torch.cuda.synchronize()
        assert np.array_equal(pb.coords.cpu().numpy(), ref.coords.cpu().numpy()[keep]), (mode, rr, y0)
print("BOUNDS_OK")
""" % ROOT


def test_debug_bounds_cascade_kernels():
    from ss25_hierarchical_multiscale_image_classification_b200 import _lib
    _lib.build(debug_bounds=True)
    env = dict(os.environ, HIPAC_DEBUG_BOUNDS="1")
    r = subprocess.run([sys.executable, "-c", DBG_SCRIPT], capture_output=True, text=True, env=env, timeout=900)
    assert r.returncode == 0 and "BOUNDS_OK" in r.stdout, (r.stdout[-2000:], r.stderr[-4000:])
