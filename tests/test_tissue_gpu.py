"""Tissue segmentation and the tissue-mask patch filter on the GPU, bit for bit against oracle/tissue.py."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import hipac_oracle as orc
from oracle import tissue as tis

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _seg(img_np, k, threshold=None, pitched=False):
    from ss25_hierarchical_multiscale_image_classification_b200.preprocessing import segment_tissue
    if pitched:   # 16-byte row pitch with garbage in the padding: the kernels must never read it
        h, w = img_np.shape[:2]
        wp = (3 * w + 15) // 16 * 16
        buf = torch.full((h, wp), 201, dtype=torch.uint8, device="cuda")
        buf[:, :3 * w] = torch.from_numpy(img_np.reshape(h, 3 * w)).cuda()
        img = buf.as_strided((h, w, 3), (wp, 3, 1))
    else:
        img = torch.from_numpy(img_np).cuda()
    mask, t, blur = segment_tissue(img, k, threshold, with_blur=True)
    return mask.cpu().numpy(), int(t.item()), blur.cpu().numpy()


def _check_seg(img_np, k, threshold=None, pitched=False):
    mask, t, blur = _seg(img_np, k, threshold, pitched)
    want_mask, want_t, want_blur = tis.segment(img_np, k, threshold)
    assert np.array_equal(blur, want_blur), (img_np.shape, k)
    assert t == want_t, (img_np.shape, k, t, want_t)
    assert np.array_equal(mask, want_mask), (img_np.shape, k)
    return t


@pytest.mark.parametrize("k", [1, 3, 5, 7])
def test_segmentation_random_images(k):
    rng = np.random.default_rng(k)
    shapes = [(1, 1), (1, 37), (29, 1), (k, k + 2), (63, 65), (130, 257), (301, 199), (8, 64), (9, 66)]
    for i, (h, w) in enumerate(shapes):
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        _check_seg(img, k, pitched=bool(i % 2))
        for thr in (0, 8, 254, 255):
            _check_seg(img, k, thr, pitched=not i % 2)


def test_segmentation_synthetic_thumbnails_and_constant_image():
    from ss25_hierarchical_multiscale_image_classification_b200 import synthetic
    for lvl, (w, h) in ((3, (2048, 2048)), (2, (1500, 1300)), (3, (1001, 777))):
        img = synthetic.make_level(1234, lvl, w, h)
        t = _check_seg(img, 7, pitched=w % 2 == 1)
        assert 5 < t < 250
    assert _check_seg(np.full((100, 133, 3), (120, 40, 200), np.uint8), 7) == 0     # constant: Otsu gives 0


def test_segmentation_16384_square():
    rng = np.random.default_rng(9)
    img = rng.integers(0, 256, (16384, 16384, 3), dtype=np.uint8)
    img[::7] //= 3
    _check_seg(img, 3)


def _level_cases():
    from ss25_hierarchical_multiscale_image_classification_b200.synthetic import SyntheticSlide
    slide = SyntheticSlide(7168, 5888, seed=17)            # level 3: 896 x 736
    thumb = slide.level_array(3)
    return slide, thumb


def _run(img, mask, level, mode, tissue, m, min_tissue=0.5, row_range=None, keep_all=False, layout="s2d16"):
    from ss25_hierarchical_multiscale_image_classification_b200.preprocessing import extract_patches_tensor
    return extract_patches_tensor(img, mask, level, layout=layout, want_u8=True, mode=mode, row_range=row_range,
                                  tissue=tissue, tissue_scale=m, min_tissue=min_tissue, keep_all=keep_all)


@pytest.fixture(scope="module")
def slide_and_masks():
    from ss25_hierarchical_multiscale_image_classification_b200.preprocessing import segment_tissue
    slide, thumb = _level_cases()
    d_thumb_mask, _ = segment_tissue(torch.from_numpy(thumb).cuda())
    want_thumb_mask, _, _ = tis.segment(thumb, 7)
    assert np.array_equal(d_thumb_mask.cpu().numpy(), want_thumb_mask)
    return slide, d_thumb_mask


@pytest.mark.parametrize("level,m", [(0, 1), (0, 8), (1, 1), (1, 4), (2, 1), (2, 2), (3, 1)])
def test_filter_vs_oracle_every_mode(slide_and_masks, level, m):
    from ss25_hierarchical_multiscale_image_classification_b200.preprocessing import segment_tissue
    slide, d_thumb_mask = slide_and_masks
    img, lmask = slide.level_array(level), slide.lesion_mask(level)
    d_img, d_lmask = torch.from_numpy(img).cuda(), torch.from_numpy(lmask).cuda()
    tissue = d_thumb_mask if m == 2 ** (3 - level) else segment_tissue(d_img, 5)[0]
    tissue_np = tissue.cpu().numpy()
    for min_tissue in (0.5, 0.05, 1):
        want = tis.extract_patches_tissue_oracle(img, lmask, level, tissue_np, m, min_tissue=min_tissue, want_images=False)
        results = []
        for mode in ("direct", "auto", "fused_legacy"):
            pb = _run(d_img, d_lmask, level, mode, tissue, m, min_tissue)
            assert np.array_equal(pb.coords.cpu().numpy(), want["coords"]), (level, m, mode, min_tissue)
            assert np.array_equal(pb.labels.cpu().numpy(), want["labels"]), (level, m, mode, min_tissue)
            assert pb.candidates == want["candidates"]
            results.append(pb)
        for pb in results[1:]:
            assert torch.equal(pb.images_u8, results[0].images_u8) and torch.equal(pb.batch, results[0].batch)
        if min_tissue == 0.5 and level > 0:
            assert 0 < len(want["coords"]) < want["candidates"]


@pytest.mark.parametrize("level,m", [(2, 2), (1, 4), (3, 1)])
def test_survivor_rows_equal_keep_all_rows_and_min_tissue_zero_is_keep_all(slide_and_masks, level, m):
    from ss25_hierarchical_multiscale_image_classification_b200.preprocessing import segment_tissue
    slide, d_thumb_mask = slide_and_masks
    img, lmask = slide.level_array(level), slide.lesion_mask(level)
    d_img, d_lmask = torch.from_numpy(img).cuda(), torch.from_numpy(lmask).cuda()
    tissue = d_thumb_mask if m > 1 else segment_tissue(d_img, 7)[0]
    S = 224
    ny = (img.shape[0] + S - 1) // S
    for layout in ("s2d16", "nhwc3"):
        ref = _run(d_img, d_lmask, level, "auto", None, 1, keep_all=True, layout=layout)
        pb = _run(d_img, d_lmask, level, "auto", tissue, m, layout=layout)
        c = pb.coords.cpu().numpy()
        idx = torch.from_numpy((c[:, 0] // S) * ny + c[:, 1] // S).cuda().long()
        assert torch.equal(pb.batch, ref.batch[idx]) and torch.equal(pb.images_u8, ref.images_u8[idx])
        assert torch.equal(pb.labels, ref.labels[idx])
        zero = _run(d_img, d_lmask, level, "auto", tissue, m, min_tissue=0, layout=layout)
        for a, b in ((zero.coords, ref.coords), (zero.labels, ref.labels), (zero.batch, ref.batch), (zero.images_u8, ref.images_u8)):
            assert torch.equal(a, b)


@pytest.mark.parametrize("mode", ["direct", "auto"])
def test_row_range_runs_merge_to_one_run(slide_and_masks, mode):
    slide, d_thumb_mask = slide_and_masks
    level, m = 1, 4
    d_img = torch.from_numpy(slide.level_array(level)).cuda()
    whole = _run(d_img, None, level, mode, d_thumb_mask, m)
    ny = (d_img.shape[0] + 223) // 224
    parts = [_run(d_img, None, level, mode, d_thumb_mask, m, row_range=(a, min(a + 5, ny))) for a in range(0, ny, 5)]
    coords = torch.cat([p.coords for p in parts])
    key = coords[:, 0].long() * (1 << 32) + coords[:, 1].long()
    perm = torch.argsort(key, stable=True)
    assert torch.equal(coords[perm], whole.coords)
    assert torch.equal(torch.cat([p.batch for p in parts])[perm], whole.batch)
    assert sum(p.candidates for p in parts) == whole.candidates


def test_pipeline_and_exchanged_path(slide_and_masks):
    from ss25_hierarchical_multiscale_image_classification_b200 import features, pipeline
    slide, d_thumb_mask = slide_and_masks
    level, m = 1, 4
    img, lmask = slide.level_array(level), slide.lesion_mask(level)
    d_img, d_lmask = torch.from_numpy(img).cuda(), torch.from_numpy(lmask).cuda()
    net = orc.make_resnet18(seed=0, classifier=True)
    packed = features.pack_resnet18(net.state_dict(), "cuda")
    got = pipeline.process_level(d_img, d_lmask, level, packed, tissue=d_thumb_mask, tissue_scale=m)
    full = pipeline.process_level(d_img, d_lmask, level, packed, tissue=d_thumb_mask, tissue_scale=m, min_tissue=0)
    ny = (img.shape[0] + 223) // 224
    assert full.coords.shape[0] == full.candidates
    c = got.coords.cpu().numpy()
    idx = torch.from_numpy((c[:, 0] // 224) * ny + c[:, 1] // 224).cuda().long()
    assert 0 < len(got) < len(full)
    for a, b in ((got.labels, full.labels), (got.features, full.features), (got.logits, full.logits)):
        assert torch.equal(a, b[idx])
    # grouped process_level and the exchange with emulated segments (row groups) equal the single pass
    grouped = pipeline.process_level(d_img, d_lmask, level, packed, tissue=d_thumb_mask, tissue_scale=m, max_candidates=3 * 28)
    nx = (img.shape[1] + 223) // 224
    x = pipeline.exchange_for_level("cuda", img.shape[1], ny, 224, 2, max_candidates=nx * 4)
    n_cand = pipeline.process_level_exchanged(d_img, d_lmask, level, packed, x, tissue=d_thumb_mask, tissue_scale=m)
    out = x.result()
    assert n_cand == got.candidates
    for k, want in (("coords", got.coords), ("labels", got.labels), ("features", got.features), ("logits", got.logits)):
        assert torch.equal(out[k], want), k
        assert torch.equal(getattr(grouped, k), want), k
    # a rank holding only the slab of its grid rows passes the matching mask rows (its origin is a multiple of m)
    r0 = (ny // 2) * 224
    slab = pipeline.process_level(d_img[r0:], d_lmask[r0:], level, packed, tissue=d_thumb_mask[r0 // m:], tissue_scale=m)
    sel = got.coords[:, 1] >= r0
    assert torch.equal(slab.coords + torch.tensor([0, r0], dtype=torch.int32, device="cuda"), got.coords[sel])
    assert torch.equal(slab.features, got.features[sel])


def test_argument_errors():
    from ss25_hierarchical_multiscale_image_classification_b200.preprocessing import extract_patches_tensor, segment_tissue
    img = torch.zeros((500, 500, 3), dtype=torch.uint8, device="cuda")
    t = torch.zeros((100, 100), dtype=torch.uint8, device="cuda")
    with pytest.raises(ValueError):
        segment_tissue(img, 9)
    with pytest.raises(ValueError):
        segment_tissue(img, 7, 256)
    for bad in (3, 64, 128):
        with pytest.raises(ValueError):
            extract_patches_tensor(img, None, 2, tissue=t, tissue_scale=bad)
    with pytest.raises(ValueError):
        extract_patches_tensor(img, None, 2, tissue=t, tissue_scale=2, min_tissue=1.5)
    with pytest.raises(ValueError):
        extract_patches_tensor(img, None, 2, stride=100, tissue=t, tissue_scale=8)    # stride not a multiple of m


DBG_SCRIPT = r"""
import numpy as np, torch, sys
sys.path.insert(0, %r)
from oracle import tissue as tis
from ss25_hierarchical_multiscale_image_classification_b200 import _lib
from ss25_hierarchical_multiscale_image_classification_b200.preprocessing import extract_patches_tensor, segment_tissue
assert _lib.lib()._name.endswith("libhipac_b200_dbg.so"), _lib.lib()._name
rng = np.random.default_rng(4)
img = rng.integers(0, 256, (1117, 903, 3), dtype=np.uint8)
img[300:800, 200:700] //= 4
mask, t, blur = segment_tissue(torch.from_numpy(img).cuda(), 7, with_blur=True)
wm, wt, wb = tis.segment(img, 7)
assert np.array_equal(blur.cpu().numpy(), wb) and int(t.item()) == wt and np.array_equal(mask.cpu().numpy(), wm)
level_img = rng.integers(0, 256, (2233, 1805, 3), dtype=np.uint8)
tissue = (rng.random((131, 97)) < 0.5).astype(np.uint8)          # smaller than the grid's footprint
for mode in ("direct", "auto", "fused_legacy"):
    for rr in (None, (3, 7)):
        pb = extract_patches_tensor(torch.from_numpy(level_img).cuda(), None, 2, mode=mode, row_range=rr, want_u8=True,
                                    tissue=torch.from_numpy(tissue).cuda(), tissue_scale=4, min_tissue=0.25)
        want = tis.extract_patches_tissue_oracle(level_img, None, 2, tissue, 4, min_tissue=0.25, want_images=False, row_range=rr)
        torch.cuda.synchronize()
        assert np.array_equal(pb.coords.cpu().numpy(), want["coords"]), (mode, rr)
print("BOUNDS_OK")
""" % ROOT


def test_debug_bounds_edge_geometry():
    from ss25_hierarchical_multiscale_image_classification_b200 import _lib
    _lib.build(debug_bounds=True)
    env = dict(os.environ, HIPAC_DEBUG_BOUNDS="1")
    r = subprocess.run([sys.executable, "-c", DBG_SCRIPT], capture_output=True, text=True, env=env, timeout=900)
    assert r.returncode == 0 and "BOUNDS_OK" in r.stdout, (r.stdout[-2000:], r.stderr[-4000:])
