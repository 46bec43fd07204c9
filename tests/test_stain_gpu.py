"""Macenko stain normalisation on the GPU: the parameter block and the apply kernel bit for bit against oracle/stain.py's
fast form (all 2^24 colours), the estimate against the literal torchstain restatement, stage 1 / the pipeline / the
exchange / the cascade with a normaliser against the plain runs normalised afterwards, the launch counts, and the new
kernels under the bounds-checking build."""
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import hipac_oracle as orc
from oracle import stain as ost

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "ss25_hierarchical_multiscale_image_classification_b200"


def _mods():
    import importlib
    return importlib.import_module(PKG + ".preprocessing.stain"), importlib.import_module(PKG + "._lib")


def _lut_bits():
    return orc.to_bf16_bits(orc.normalize_lut())      # uint16 [256, 3]


def _want_batch(u8: np.ndarray, layout: str) -> np.ndarray:
    """int16 bits of stage 1's ToTensor/Normalize of uint8 [n, 224, 224, 3] patches in `layout`."""
    lut = _lut_bits()
    x = np.stack([lut[:, c][u8[..., c]] for c in range(3)], axis=-1)
    if layout == "nhwc3":
        return x.view(np.int16)
    n = u8.shape[0]
    y = np.zeros((n, 112, 115, 16), np.uint16)
    y[:, :, 2:114, :12] = x.reshape(n, 112, 2, 112, 2, 3).transpose(0, 1, 3, 2, 4, 5).reshape(n, 112, 112, 12)
    return y.view(np.int16)


def _params_of(norm):
    p = norm.params.cpu().numpy()
    return bool(p[0]), p[2:11].reshape(3, 3), p[11:]


# ---------------------------------------------------------------------------------------------------------------------
# 1. the parameter block
# ---------------------------------------------------------------------------------------------------------------------
def test_od_table_within_one_ulp():
    stain, _ = _mods()
    src = stain.Stain.reference("cuda")
    for io in (1, 128, 240, 255):
        norm = stain.StainNormalizer(src, io=io)
        valid, _, od = _params_of(norm)
        want = -np.log((np.arange(256) + 1.0) / io)
        assert valid and float(norm.params[1]) == io
        assert np.all(np.abs(od - want) <= np.spacing(np.abs(want))), io
        assert np.all(np.diff(od) < 0)


def test_normalizer_matrix_equals_the_fixed_sequence():
    stain, _ = _mods()
    rng = np.random.default_rng(1)
    est = ost.estimate_literal(ost.he_image(7, 300, 300, ost.HE_TRUE))
    sources = [(ost.HE_REF, ost.MAXC_REF), (est[0], est[1])]
    sources += [(rng.uniform(0.05, 1.0, (3, 2)), rng.uniform(0.3, 3.0, 2)) for _ in range(20)]
    for k, (he, max_c) in enumerate(sources):
        src = stain.Stain.from_matrix(he, max_c, "cuda")
        for target in (None, stain.Stain.from_matrix(*sources[(k + 1) % len(sources)], "cuda")):
            norm = stain.StainNormalizer(src, target)
            valid, M, _ = _params_of(norm)
            t = sources[(k + 1) % len(sources)] if target is not None else (ost.HE_REF, ost.MAXC_REF)
            want = ost.normalizer_matrix(np.asarray(he), np.asarray(max_c), np.asarray(t[0]), np.asarray(t[1]))
            assert valid and np.array_equal(M.view(np.int64), want.view(np.int64)), k


def test_normalizer_invalid_inputs():
    stain, _ = _mods()
    ref = stain.Stain.reference("cuda")
    bad = stain.Stain.from_matrix(ost.HE_REF, ost.MAXC_REF, "cuda")
    bad.block[8] = 0
    singular = stain.Stain.from_matrix([[0.5, 0.5], [0.6, 0.6], [0.2, 0.2]], [1.0, 1.0], "cuda")
    for src, tgt in ((bad, None), (ref, bad), (singular, None)):
        assert not _params_of(stain.StainNormalizer(src, tgt))[0]


# ---------------------------------------------------------------------------------------------------------------------
# 2. the apply kernel, every colour
# ---------------------------------------------------------------------------------------------------------------------
N_ALL = 335   # 335 patches of 224^2 hold all 2^24 colours


@pytest.fixture(scope="module")
def all_colour_patches():
    c = np.zeros((N_ALL * 224 * 224, 3), np.uint8)
    c[:1 << 24] = ost.all_colours()
    return c.reshape(N_ALL, 224, 224, 3)


@pytest.fixture(scope="module")
def normaliser():
    stain, _ = _mods()
    he, max_c, _ = ost.estimate_literal(ost.he_image(11, 400, 400, ost.HE_TRUE_B))
    return stain.StainNormalizer(stain.Stain.from_matrix(he, max_c, "cuda"))


def test_apply_every_colour(all_colour_patches, normaliser):
    x = torch.from_numpy(all_colour_patches).cuda()
    _, M, od = _params_of(normaliser)
    want = ost.apply(all_colour_patches, M, od)
    got = normaliser.apply(x, None).cpu().numpy()
    assert np.array_equal(got, want)
    assert (want == 0).any() or (want == 255).any()
    for layout in ("nhwc3", "s2d16"):
        shape = (N_ALL, 224, 224, 3) if layout == "nhwc3" else (N_ALL, 112, 115, 16)
        out = torch.full(shape, -7.0, dtype=torch.bfloat16, device="cuda")        # garbage in the S2D16 padding
        u8 = torch.full_like(x, 3)
        batch = normaliser.apply(x, layout, out_u8=u8, out=out)
        assert batch.data_ptr() == out.data_ptr()
        assert np.array_equal(u8.cpu().numpy(), want), layout
        assert np.array_equal(batch.view(torch.int16).cpu().numpy(), _want_batch(want, layout)), layout
    # exact in place
    y = x.clone()
    normaliser.apply(y, None, out_u8=y)
    assert np.array_equal(y.cpu().numpy(), want)


@pytest.mark.parametrize("layout", ["nhwc3", "s2d16", None])
def test_apply_device_count_and_pass_through(normaliser, layout):
    stain, _ = _mods()
    rng = np.random.default_rng(5)
    n, base = 9, 4
    x_np = rng.integers(0, 256, (n, 224, 224, 3), dtype=np.uint8)
    x = torch.from_numpy(x_np).cuda()
    _, M, od = _params_of(normaliser)
    want_u8 = ost.apply(x_np, M, od)
    shape = (n, 224, 224, 3) if layout == "nhwc3" else (n, 112, 115, 16)
    for count in (0, base, base + 5, base + n, base + n + 7):
        cnt = torch.tensor([count, 0], dtype=torch.int32, device="cuda")
        u8 = torch.full_like(x, 0xA5)
        out = torch.full(shape, 0x7F81, dtype=torch.int16, device="cuda").view(torch.bfloat16) if layout else None
        normaliser.apply(x, layout, count=cnt, base=base, out_u8=u8, out=out)
        k = max(0, min(n, count - base))
        got = u8.cpu().numpy()
        assert np.array_equal(got[:k], want_u8[:k]) and np.all(got[k:] == 0xA5), count
        if layout:
            bits = out.view(torch.int16).cpu().numpy()
            assert np.array_equal(bits[:k], _want_batch(want_u8[:k], layout)) and np.all(bits[k:] == 0x7F81), count
    # valid = 0: the bytes pass through, the batch is plain stage 1's
    off = stain.StainNormalizer(stain.Stain.from_matrix(ost.HE_REF, ost.MAXC_REF * 0, "cuda"))
    assert not _params_of(off)[0]
    got = off.apply(x, layout)
    if layout is None:
        assert np.array_equal(got.cpu().numpy(), x_np)
    else:
        assert np.array_equal(got.view(torch.int16).cpu().numpy(), _want_batch(x_np, layout))


# ---------------------------------------------------------------------------------------------------------------------
# 3. the estimate
# ---------------------------------------------------------------------------------------------------------------------
def _estimate_raw(img_t, garbage: bool):
    """hipac_stain_estimate with an explicit workspace (optionally garbage-filled)."""
    stain, _lib = _mods()
    l = _lib.lib()
    H, W = int(img_t.shape[0]), int(img_t.shape[1])
    ws_bytes = l.hipac_stain_workspace_bytes(H, W)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device="cuda")
    if garbage:
        ws.random_(0, 256)
    block = torch.full((16,), float("nan"), dtype=torch.float64, device="cuda")
    _lib.check(l.hipac_stain_estimate(img_t.data_ptr(), H, W, int(img_t.stride(0)), 240, 1.0, 0.15, block.data_ptr(),
                                      ws.data_ptr(), ws_bytes, torch.cuda.current_stream().cuda_stream), "estimate")
    torch.cuda.synchronize()
    return block.cpu().numpy()


def _pitched(img_np):
    h, w = img_np.shape[:2]
    wp = (3 * w + 31) // 32 * 32 + 16
    buf = torch.full((h, wp), 77, dtype=torch.uint8, device="cuda")
    buf[:, :3 * w] = torch.from_numpy(img_np.reshape(h, 3 * w)).cuda()
    return buf.as_strided((h, w, 3), (wp, 3, 1))


def test_estimate_against_literal():
    worst_he, worst_c = 0.0, 0.0
    cases = [(ost.he_image(21, 7, 13, ost.HE_TRUE, background=0.1), False),
             (ost.he_image(22, 1000, 777, ost.HE_TRUE_B), True),
             (ost.he_image(23, 2048, 2048, ost.HE_TRUE), False),
             (ost.he_image(24, 333, 517, ost.HE_TRUE_B, background=0.8), True)]
    for img, pitched in cases:
        lit = ost.estimate_literal(img)
        assert lit is not None
        t = _pitched(img) if pitched else torch.from_numpy(img).cuda()
        a, b = _estimate_raw(t, False), _estimate_raw(t, True)
        assert np.array_equal(a.view(np.int64), b.view(np.int64)), img.shape      # same bits over a garbage workspace
        he, max_c = a[:6].reshape(3, 2), a[6:8]
        assert a[8] == 1.0 and a[9] == lit[2], (img.shape, a[9], lit[2])
        dhe, dc = np.abs(he - lit[0]).max(), (np.abs(max_c - lit[1]) / lit[1]).max()
        worst_he, worst_c = max(worst_he, dhe), max(worst_c, dc)
        assert dhe <= 1e-9 and dc <= 1e-9, (img.shape, dhe, dc)
        assert np.all(a[10:] == 0)
    print(f"largest |dHE| {worst_he:.3e}, largest |dmaxC| / maxC {worst_c:.3e}")


def test_estimate_invalid_images():
    white = np.full((40, 50, 3), 255, np.uint8)
    one = white.copy()
    one[7, 9] = (30, 60, 90)
    for img, n_hat in ((white, 0), (one, 1), (np.full((1, 1, 3), 20, np.uint8), 1)):
        assert ost.estimate_literal(img) is None
        for t in (torch.from_numpy(img).cuda(), _pitched(img)):
            blk = _estimate_raw(t, True)
            assert blk[8] == 0.0 and blk[9] == n_hat, (img.shape, blk)


def test_estimate_python_api():
    stain, _ = _mods()
    img = ost.he_image(31, 300, 200, ost.HE_TRUE)
    s = stain.estimate_stain(torch.from_numpy(img).cuda())
    lit = ost.estimate_literal(img)
    assert s.valid() and int(s.n_hat) == lit[2]
    assert np.abs(s.he.cpu().numpy() - lit[0]).max() <= 1e-9
    with pytest.raises(ValueError):
        stain.estimate_stain(torch.zeros((4, 4), dtype=torch.uint8, device="cuda"))


# ---------------------------------------------------------------------------------------------------------------------
# 4. stage 1 with a normaliser
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def slide():
    from ss25_hierarchical_multiscale_image_classification_b200.synthetic import SyntheticSlide
    s = SyntheticSlide(7168, 5888, seed=17)            # level 3: 896 x 736
    return {L: (torch.from_numpy(s.level_array(L)).cuda(), torch.from_numpy(s.lesion_mask(L)).cuda()) for L in range(4)}


@pytest.fixture(scope="module")
def slide_norm(slide):
    stain, _ = _mods()
    s = stain.estimate_stain(slide[3][0])
    assert s.valid()
    return stain.StainNormalizer(s)


def _roi_of_level3(slide):
    from ss25_hierarchical_multiscale_image_classification_b200.cascade import roi_grid
    from ss25_hierarchical_multiscale_image_classification_b200.preprocessing import extract_patches_tensor
    img3 = slide[3][0]
    pb = extract_patches_tensor(img3, None, 3)
    scores = torch.from_numpy(np.random.default_rng(3).random(len(pb)).astype(np.float32)).cuda()
    return roi_grid(pb.coords, scores, 3, int(img3.shape[1]), int(img3.shape[0]), threshold=0.5)


@pytest.mark.parametrize("level", [0, 1, 2, 3])
def test_stage1_with_normaliser_equals_plain_then_apply(slide, slide_norm, level):
    from ss25_hierarchical_multiscale_image_classification_b200.preprocessing import extract_patches_tensor, segment_tissue
    img, mask = slide[level]
    tissue = segment_tissue(slide[3][0])[0]
    roi = _roi_of_level3(slide) if level < 3 else None
    ny = (int(img.shape[0]) + 223) // 224
    variants = [dict(), dict(tissue=tissue, tissue_scale=1 << (3 - level))]
    if roi is not None:
        variants += [dict(roi=roi), dict(roi=roi, tissue=tissue, tissue_scale=1 << (3 - level))]
    for mode in ("fused", "fused_legacy", "direct"):
        for kw in variants:
            for rr, layout in ((None, "s2d16"), ((1, max(2, ny - 1)), "nhwc3")):
                plain = extract_patches_tensor(img, mask, level, mode=mode, row_range=rr, layout=layout, want_u8=True, **kw)
                got = extract_patches_tensor(img, mask, level, mode=mode, row_range=rr, layout=layout, want_u8=True,
                                             stain=slide_norm, **kw)
                what = (level, mode, tuple(kw), rr)
                assert torch.equal(got.coords, plain.coords) and torch.equal(got.labels, plain.labels), what
                assert got.candidates == plain.candidates, what
                want_u8 = slide_norm.apply(plain.images_u8, None)
                assert torch.equal(got.images_u8, want_u8), what
                want_batch = slide_norm.apply(plain.images_u8, layout)
                assert torch.equal(got.batch.view(torch.int16), want_batch.view(torch.int16)), what
                assert np.array_equal(want_batch.view(torch.int16).cpu().numpy(), _want_batch(want_u8.cpu().numpy(), layout))
                if len(plain) and kw == {}:
                    assert not torch.equal(got.images_u8, plain.images_u8)
            only = extract_patches_tensor(img, mask, level, mode=mode, stain=slide_norm, **kw)          # batch only
            ref = extract_patches_tensor(img, mask, level, mode=mode, want_u8=True, stain=slide_norm, **kw)
            assert only.images_u8 is None and torch.equal(only.batch.view(torch.int16), ref.batch.view(torch.int16))


# ---------------------------------------------------------------------------------------------------------------------
# 5. pipeline, exchange, cascade
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def packed2():
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    return features.pack_resnet18(orc.make_resnet18(seed=0, classifier=True).state_dict(), "cuda")


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _assert_equal_results(got, want, what):
    for k in ("coords", "labels", "features", "logits"):
        a, b = getattr(got, k), getattr(want, k)
        assert a.shape == b.shape and torch.equal(_bits(a), _bits(b)), (what, k)


@pytest.mark.parametrize("tta", [False, True])
def test_process_level_with_normaliser_equals_classify_tensor(slide, slide_norm, packed2, tta):
    from ss25_hierarchical_multiscale_image_classification_b200 import features, pipeline
    from ss25_hierarchical_multiscale_image_classification_b200.preprocessing import extract_patches_tensor
    img, mask = slide[0]
    nx = (int(img.shape[1]) + 223) // 224
    got = pipeline.process_level(img, mask, 0, packed2, stain=slide_norm, tta=tta)
    plain = pipeline.process_level(img, mask, 0, packed2, tta=tta)
    assert torch.equal(got.coords, plain.coords) and got.candidates == plain.candidates and len(got) > 0
    pb = extract_patches_tensor(img, mask, 0, want_u8=True)
    f, lg = features.classify_tensor(slide_norm.apply(pb.images_u8, "s2d16"), packed2, tta=tta)
    _assert_equal_results(got, SimpleNamespace(coords=pb.coords, labels=pb.labels, features=f, logits=lg), "process_level")
    assert not torch.equal(got.features, plain.features)
    grouped = pipeline.process_level(img, mask, 0, packed2, stain=slide_norm, tta=tta, max_candidates=3 * nx)
    _assert_equal_results(grouped, got, "row groups")


@pytest.mark.parametrize("world", [2, 4])
def test_exchanged_with_normaliser_equals_single_rank(slide, packed2, world):
    """Every emulated rank estimates the stain from the same thumbnail itself; the merged result equals the single rank."""
    from ss25_hierarchical_multiscale_image_classification_b200 import pipeline, sharding
    stain, _ = _mods()
    img, mask = slide[0]
    h, w = int(img.shape[0]), int(img.shape[1])
    nx, ny = (w + 223) // 224, (h + 223) // 224
    single = pipeline.process_level(img, mask, 0, packed2, stain=stain.StainNormalizer(stain.estimate_stain(slide[3][0])))
    parts = []
    for r in range(world):
        norm = stain.StainNormalizer(stain.estimate_stain(slide[3][0].clone()))
        i0, i1 = sharding.shard_rows(ny, world, r)
        y0, y1 = sharding.slab_rows(i0, i1, 224, 1792, h)
        x = pipeline.exchange_for_level("cuda", w, i1 - i0, 224, 2, max_candidates=4 * nx)
        n_cand = pipeline.process_level_exchanged(img[y0:y1], mask[y0:y1], 0, packed2, x, row_range=(0, i1 - i0), y_offset=y0,
                                                  stain=norm)
        assert n_cand == nx * (i1 - i0)
        parts.append({k: v.clone() for k, v in x.result().items()})
    merged = {k: torch.cat([p[k] for p in parts]) for k in parts[0]}
    perm = sharding.canonical_order(merged["coords"])
    for k in ("coords", "labels", "features", "logits"):
        assert torch.equal(merged[k][perm], getattr(single, k)), (world, k)


def test_cascade_with_normaliser_equals_restricted_level(slide, slide_norm, packed2):
    from oracle import cascade as oc
    from ss25_hierarchical_multiscale_image_classification_b200 import pipeline
    from ss25_hierarchical_multiscale_image_classification_b200.cascade import process_cascade, threshold_of, tumor_margin
    coarse = pipeline.process_level(*slide[3], 3, packed2, stain=slide_norm)
    full = pipeline.process_level(*slide[0], 0, packed2, stain=slide_norm)
    h3, w3 = int(slide[3][0].shape[0]), int(slide[3][0].shape[1])
    nx, ny = (w3 + 223) // 224, (h3 + 223) // 224
    margins = tumor_margin(coarse.logits).cpu().numpy()
    m = np.sort(margins.astype(np.float64))[::-1]
    k = max(1, len(m) // 3)
    tau = float(1.0 / (1.0 + np.exp(-0.5 * (m[k - 1] + m[k])))) if m[k - 1] > m[k] else 0.5
    res = process_cascade({L: slide[L] for L in (3, 0)}, packed2, order=(3, 0), tau=tau, stain=slide_norm)
    _assert_equal_results(res[3], coarse, "coarse")
    grid = oc.roi_grid(coarse.coords.cpu().numpy(), margins, threshold_of(tau), 224, nx, ny, 0)
    keep = oc.roi_mask(full.coords.cpu().numpy(), 0, oc.Roi(grid, 3, 224, 224))
    idx = torch.from_numpy(np.nonzero(keep)[0]).cuda()
    assert 0 < len(idx) <= len(full)
    for key in ("coords", "labels", "features", "logits"):
        assert torch.equal(getattr(res[0], key), getattr(full, key)[idx]), key


# ---------------------------------------------------------------------------------------------------------------------
# 6. launches
# ---------------------------------------------------------------------------------------------------------------------
ESTIMATE_LAUNCHES = 4 + 16 + 2 + 16 + 1   # sums, cov, eig, phi; 8 x (hist, pick); he, conc; 8 x (hist, pick); finish


def test_launch_counts(slide, slide_norm, packed2):
    from ss25_hierarchical_multiscale_image_classification_b200 import _lib, pipeline
    stain, _ = _mods()
    l = _lib.lib()

    def launches(fn):
        torch.cuda.synchronize()
        l.hipac_launch_count(1)
        fn()
        return l.hipac_launch_count(1)

    for shape in ((1, 1), (7, 13), (736, 896)):
        img = torch.zeros(shape + (3,), dtype=torch.uint8, device="cuda")
        assert launches(lambda: stain.estimate_stain(img)) == ESTIMATE_LAUNCHES
    assert launches(lambda: stain.StainNormalizer(stain.Stain.reference("cuda"))) == 1
    img, mask = slide[0]
    nx = (int(img.shape[1]) + 223) // 224
    ny = (int(img.shape[0]) + 223) // 224
    for mc, groups in ((16384, 1), (3 * nx, (ny + 2) // 3)):
        plain = launches(lambda: pipeline.process_level(img, mask, 0, packed2, max_candidates=mc))
        again = launches(lambda: pipeline.process_level(img, mask, 0, packed2, max_candidates=mc, stain=None))
        with_stain = launches(lambda: pipeline.process_level(img, mask, 0, packed2, max_candidates=mc, stain=slide_norm))
        assert again == plain and with_stain == plain + groups, (mc, plain, with_stain)


# ---------------------------------------------------------------------------------------------------------------------
# 7. bounds-checking build
# ---------------------------------------------------------------------------------------------------------------------
DBG_SCRIPT = r"""
import numpy as np, torch, sys
sys.path.insert(0, %r)
from oracle import stain as ost
from ss25_hierarchical_multiscale_image_classification_b200 import _lib
from ss25_hierarchical_multiscale_image_classification_b200.preprocessing import StainNormalizer, estimate_stain
assert _lib.lib()._name.endswith("libhipac_b200_dbg.so"), _lib.lib()._name
for (h, w) in ((1, 1), (7, 13), (97, 61)):
    img = ost.he_image(h * w, h, w, ost.HE_TRUE)
    wp = (3 * w + 15) // 16 * 16
    buf = torch.full((h, wp), 9, dtype=torch.uint8, device="cuda")
    buf[:, :3 * w] = torch.from_numpy(img.reshape(h, 3 * w)).cuda()
    s = estimate_stain(buf.as_strided((h, w, 3), (wp, 3, 1)))
    torch.cuda.synchronize()
    lit = ost.estimate_literal(img)
    assert s.valid() == (lit is not None), (h, w)
    norm = StainNormalizer(s)
x = torch.from_numpy(np.random.default_rng(0).integers(0, 256, (3, 224, 224, 3), dtype=np.uint8)).cuda()
for layout in ("s2d16", "nhwc3", None):
    for count in (None, torch.tensor([5], dtype=torch.int32, device="cuda")):
        norm.apply(x, layout, count=count, base=2, out_u8=torch.empty_like(x))
torch.cuda.synchronize()
print("BOUNDS_OK")
""" % ROOT


def test_debug_bounds_edge_geometry():
    from ss25_hierarchical_multiscale_image_classification_b200 import _lib
    _lib.build(debug_bounds=True)
    env = dict(os.environ, HIPAC_DEBUG_BOUNDS="1")
    r = subprocess.run([sys.executable, "-c", DBG_SCRIPT], capture_output=True, text=True, env=env, timeout=900)
    assert r.returncode == 0 and "BOUNDS_OK" in r.stdout, (r.stdout[-2000:], r.stderr[-4000:])
