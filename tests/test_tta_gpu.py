"""Rotation/flip test-time augmentation on the GPU: the D4 view kernel against the torch definition, the TTA forward against
the mean of the view forwards (bit for bit) and its invariance under the group, device-count mode, the launch count, and
the pipeline / exchange / cascade entry points with tta=True against classify_tensor(..., tta=True)."""
import numpy as np
import pytest

from oracle import cascade as oc
from oracle import hipac_oracle as orc

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

SENTINEL = 0x7F81                  # a bf16 NaN bit pattern: no kernel writes it, so an untouched row still holds it


def view_torch(x, v):
    """View v = 4 f + k of an NHWC batch under D4: the definition the library implements."""
    f, k = divmod(v, 4)
    return torch.rot90(torch.flip(x, dims=[2]) if f else x, k, dims=(1, 2))


def _s2d16(x):
    """bf16 NHWC3 [n,224,224,3] -> the S2D16 layout [n,112,115,16] (see HIPAC_LAYOUT_S2D16_BF16)."""
    n = x.shape[0]
    y = torch.zeros((n, 112, 115, 16), dtype=torch.bfloat16, device=x.device)
    y[:, :, 2:114, :12] = x.reshape(n, 112, 2, 112, 2, 3).permute(0, 1, 3, 2, 4, 5).reshape(n, 112, 112, 12)
    return y


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


def _normalised_batch(n, seed):
    """bf16 NHWC3 patches as the tile scan writes them: ToTensor + Normalize of random uint8 pixels."""
    rng = np.random.default_rng(seed)
    u8 = torch.from_numpy(rng.integers(0, 256, size=(n, 224, 224, 3), dtype=np.uint8)).cuda().long()
    lut = torch.from_numpy(orc.normalize_lut()).cuda()
    return torch.stack([lut[:, c][u8[..., c]] for c in range(3)], dim=-1).bfloat16()


def _packed_with_head(num_classes, seed=0):
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    sd = dict(orc.make_resnet18(seed=seed, classifier=True).state_dict())
    gen = torch.Generator().manual_seed(num_classes)
    sd["fc.weight"] = torch.randn((num_classes, 512), generator=gen) * 512 ** -0.5
    sd["fc.bias"] = torch.randn((num_classes,), generator=gen)
    return features.pack_resnet18(sd, "cuda"), sd


@pytest.fixture(scope="module")
def packed2():
    return _packed_with_head(2)[0]


# ---------------------------------------------------------------------------------------------------------------------
# 1. the view kernel
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", ["nhwc3", "s2d16"])
def test_view_kernel_equals_torch_definition(layout):
    """Every view of an odd batch in both input layouts equals the S2D16 form of the torch definition over the whole
    tensor, padding included; an S2D16 input with garbage in its padding columns and channels 12..15 is rewritten to
    zeros there.  Device-count mode writes exactly the rows below clamp(count - base, 0, n)."""
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    n = 7
    g = torch.Generator(device="cuda").manual_seed(11)
    x3 = torch.randn((n, 224, 224, 3), generator=g, device="cuda").bfloat16()
    if layout == "s2d16":
        xin = _s2d16(x3)
        junk = torch.randn(xin.shape, generator=g, device="cuda").bfloat16()
        xin[:, :, :2], xin[:, :, 114:], xin[..., 12:] = junk[:, :, :2], junk[:, :, 114:], junk[..., 12:]
    else:
        xin = x3
    base = 3
    for v in range(8):
        want = _bits(_s2d16(view_torch(x3, v)))
        got = features.d4_view(xin, v)
        torch.cuda.synchronize()
        assert torch.equal(_bits(got), want), (layout, v)
        for count, eff in ((base - 1, 0), (base + n // 2, n // 2), (base + n + 4, n)):
            out = torch.empty_like(got)
            out.view(torch.int16).fill_(SENTINEL)
            features.d4_view(xin, v, count=torch.tensor([count, 12345], dtype=torch.int32, device="cuda"), base=base, out=out)
            torch.cuda.synchronize()
            assert torch.equal(_bits(out)[:eff], want[:eff]), (layout, v, count)
            assert bool((_bits(out)[eff:] == SENTINEL).all()), (layout, v, count)


def test_views_form_the_group():
    """Applying the kernel to a view gives another view: for each u, w -> view_w(view_u(x)) is a permutation of the eight
    views (the composition table of D4), so the eight are the group and not eight arbitrary transforms."""
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    g = torch.Generator(device="cuda").manual_seed(12)
    x3 = torch.randn((2, 224, 224, 3), generator=g, device="cuda").bfloat16()
    views = [_bits(features.d4_view(x3, c)) for c in range(8)]
    assert all(not torch.equal(views[a], views[b]) for a in range(8) for b in range(a))
    for u in range(8):
        xu = features.d4_view(x3, u)
        hits = []
        for w in range(8):
            got = _bits(features.d4_view(xu, w))
            hits.append([c for c in range(8) if torch.equal(got, views[c])])
        assert all(len(h) == 1 for h in hits) and sorted(h[0] for h in hits) == list(range(8)), (u, hits)


# ---------------------------------------------------------------------------------------------------------------------
# 2. the TTA forward is the mean of the view forwards
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("num_classes", [1, 2, 9, 1000])
def test_tta_forward_is_the_mean_of_the_view_forwards(num_classes):
    """Three chunks with a partial last one: both input layouts give the same bits, the features are
    ((f_0 + f_1) + ... + f_7) * 0.125 in fp32 bit for bit with f_v the plain forward of view v, and the logits are the head
    applied to them within the fp32 bound of the fp64 product (the bound test_forward_is_the_chain_of_tested_kernels uses)."""
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    packed, sd = _packed_with_head(num_classes)
    n, chunk = 200, 96
    x3 = _normalised_batch(n, num_classes)
    xs = _s2d16(x3)
    f3, l3 = features.classify_tensor(x3, packed, chunk, tta=True)
    fs, ls = features.classify_tensor(xs, packed, chunk, tta=True)
    only_f = features.extract_features_tensor(xs, packed, chunk, tta=True)
    acc = None
    for v in range(8):
        fv = features.extract_features_tensor(_s2d16(view_torch(x3, v)), packed, chunk)
        acc = fv if acc is None else acc + fv
    mean = acc * torch.tensor(0.125, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    assert torch.equal(f3, fs) and torch.equal(l3, ls), "the NHWC3 and S2D16 inputs give different results"
    assert torch.equal(fs, mean), "the TTA features are not the fp32 mean of the eight view forwards"
    assert torch.equal(only_f, fs)
    w, b = sd["fc.weight"].double().cuda(), sd["fc.bias"].double().cuda()
    f = fs.double()
    bound = 32 * 2.0 ** -24 * (f.abs() @ w.abs().T + b.abs())
    assert bool(((ls.double() - (f @ w.T + b)).abs() <= bound).all())


# ---------------------------------------------------------------------------------------------------------------------
# 3. invariance
# ---------------------------------------------------------------------------------------------------------------------
def test_tta_features_are_invariant_under_d4(packed2):
    """tta(view_u(x)) = tta(x) for every u up to the reordering of the fp32 running sum: both sum the same eight view
    features, so they differ by at most 2 * 7 roundings of a partial sum, 14 * 2^-24 * 0.125 * sum_v |f_v|."""
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    n = 24
    x3 = _normalised_batch(n, 5)
    ref = features.extract_features_tensor(x3, packed2, tta=True)
    mag = sum(features.extract_features_tensor(_s2d16(view_torch(x3, v)), packed2).abs() for v in range(8))
    bound = 14 * 2.0 ** -24 * 0.125 * mag
    plain = features.extract_features_tensor(x3, packed2)
    for u in range(1, 8):
        got = features.extract_features_tensor(view_torch(x3, u).contiguous(), packed2, tta=True)
        torch.cuda.synchronize()
        assert bool(((got - ref).abs() <= bound).all()), u
    # the plain features are not invariant: the test would not notice a TTA that ignored the views
    moved = features.extract_features_tensor(view_torch(x3, 1).contiguous(), packed2)
    assert not bool(((moved - plain).abs() <= bound).all())


# ---------------------------------------------------------------------------------------------------------------------
# 4. device count
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", ["s2d16", "nhwc3"])
@pytest.mark.parametrize("cap,n,chunk", [(11, 6, 4096), (11, 6, 4), (11, 11, 4096), (11, 0, 4096), (300, 150, 128), (5, 9, 4096)])
def test_device_count_tta_equals_host_count(packed2, layout, cap, n, chunk):
    """hipac_resnet18_forward_d4 with the patch count in device memory gives the host-count bits on the first
    min(count, capacity) patches and leaves the other rows of features and logits untouched."""
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    g = torch.Generator(device="cuda").manual_seed(cap * 1000 + n)
    x = torch.randn((cap, 224, 224, 3), generator=g, device="cuda").bfloat16()
    if layout == "s2d16":
        x = _s2d16(x)
    m = min(n, cap)
    count = torch.tensor([n, 12345], dtype=torch.int32, device="cuda")
    f_ref, l_ref = features.classify_tensor(x[:m], packed2, chunk, tta=True) if m else (None, None)
    f, l = features._forward(x, packed2, True, chunk, count=count, tta=True)
    f2 = torch.full((cap, 512), 7.0, device="cuda")
    l2 = torch.full((cap, 2), 7.0, device="cuda")
    lib = features._lib.lib()
    ws_bytes = lib.hipac_resnet18_workspace_bytes(cap, chunk)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device="cuda")
    rc = lib.hipac_resnet18_forward_d4(packed2.blob.data_ptr(), packed2.num_classes, x.data_ptr(), 2 if layout == "s2d16" else 1,
                                       cap, count.data_ptr(), f2.data_ptr(), l2.data_ptr(), ws.data_ptr(), ws_bytes, chunk,
                                       torch.cuda.current_stream().cuda_stream)
    assert rc == 0, lib.hipac_last_error()
    torch.cuda.synchronize()
    assert bool((f2[m:] == 7.0).all()) and bool((l2[m:] == 7.0).all())
    if m:
        assert torch.equal(f[:m], f_ref) and torch.equal(l[:m], l_ref)
        assert torch.equal(f2[:m], f_ref) and torch.equal(l2[:m], l_ref)


# ---------------------------------------------------------------------------------------------------------------------
# 5. launches
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,chunk,chunks", [(20, 4096, 1), (20, 8, 3)])
def test_launch_count(packed2, n, chunk, chunks):
    """Per chunk: the plain forward issues 18 launches (stem, 16 convs, pool) plus the repack for NHWC3 input, the TTA
    forward eight times that, plus the view kernels of views 1..7 for S2D16 input."""
    from ss25_hierarchical_multiscale_image_classification_b200 import _lib, features
    l = _lib.lib()
    x3 = _normalised_batch(n, 1)
    xs = _s2d16(x3)

    def launches(x, tta):
        torch.cuda.synchronize()
        l.hipac_launch_count(1)
        features.classify_tensor(x, packed2, chunk, tta=tta)
        return l.hipac_launch_count(1)

    plain_s, plain_3 = launches(xs, False), launches(x3, False)
    assert plain_s == 18 * chunks and plain_3 == 19 * chunks
    assert launches(xs, True) == 8 * plain_s + 7 * chunks
    assert launches(x3, True) == 8 * plain_3


# ---------------------------------------------------------------------------------------------------------------------
# 6. pipeline, exchange, cascade
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def slide():
    """The cascade tests' seeded slide (level 3: 896 x 736)."""
    from ss25_hierarchical_multiscale_image_classification_b200.synthetic import SyntheticSlide
    s = SyntheticSlide(7168, 5888, seed=17)
    return {L: (torch.from_numpy(s.level_array(L)).cuda(), torch.from_numpy(s.lesion_mask(L)).cuda()) for L in (0, 3)}


def _assert_equal_results(got, want, what):
    for k in ("coords", "labels", "features", "logits"):
        a, b = getattr(got, k), getattr(want, k)
        assert a.shape == b.shape and torch.equal(_bits(a) if a.is_floating_point() else a,
                                                  _bits(b) if b.is_floating_point() else b), (what, k)


def test_process_level_tta_equals_classify_tensor(slide, packed2):
    """process_level(tta=True) keeps the plain run's coordinates, labels and candidate count, and its features and logits are
    classify_tensor(batch, tta=True) of the same survivors bit for bit: in one pass, with a tissue mask, and in row groups."""
    from types import SimpleNamespace

    from ss25_hierarchical_multiscale_image_classification_b200 import features, pipeline
    from ss25_hierarchical_multiscale_image_classification_b200.preprocessing import extract_patches_tensor, segment_tissue
    img, mask = slide[0]
    tissue = segment_tissue(slide[3][0])[0]
    nx = (int(img.shape[1]) + 223) // 224
    for kw in ({}, dict(tissue=tissue, tissue_scale=8)):
        plain = pipeline.process_level(img, mask, 0, packed2, **kw)
        tta = pipeline.process_level(img, mask, 0, packed2, tta=True, **kw)
        assert len(tta) > 0 and torch.equal(tta.coords, plain.coords) and torch.equal(tta.labels, plain.labels)
        assert tta.candidates == plain.candidates
        pb = extract_patches_tensor(img, mask, 0, **kw)
        f, lg = features.classify_tensor(pb.batch, packed2, tta=True)
        want = SimpleNamespace(coords=pb.coords, labels=pb.labels, features=f, logits=lg)
        _assert_equal_results(tta, want, ("process_level", tuple(kw)))
        assert not torch.equal(tta.features, plain.features)
        grouped = pipeline.process_level(img, mask, 0, packed2, tta=True, max_candidates=3 * nx, **kw)
        _assert_equal_results(grouped, tta, ("row groups", tuple(kw)))


@pytest.mark.parametrize("world", [2, 4])
def test_exchanged_tta_equals_single_rank(slide, packed2, world):
    """process_level_exchanged(tta=True) on `world` emulated row shards, merged, equals the single-rank TTA run."""
    from ss25_hierarchical_multiscale_image_classification_b200 import pipeline, sharding
    img, mask = slide[0]
    h, w = int(img.shape[0]), int(img.shape[1])
    nx, ny = (w + 223) // 224, (h + 223) // 224
    single = pipeline.process_level(img, mask, 0, packed2, tta=True)
    parts = []
    for r in range(world):
        i0, i1 = sharding.shard_rows(ny, world, r)
        y0, y1 = sharding.slab_rows(i0, i1, 224, 1792, h)
        x = pipeline.exchange_for_level("cuda", w, i1 - i0, 224, 2, max_candidates=4 * nx)
        n_cand = pipeline.process_level_exchanged(img[y0:y1], mask[y0:y1], 0, packed2, x, row_range=(0, i1 - i0), y_offset=y0,
                                                  tta=True)
        assert n_cand == nx * (i1 - i0)
        parts.append({k: v.clone() for k, v in x.result().items()})
    merged = {k: torch.cat([p[k] for p in parts]) for k in parts[0]}
    perm = sharding.canonical_order(merged["coords"])
    for k in ("coords", "labels", "features", "logits"):
        assert torch.equal(merged[k][perm], getattr(single, k)), (world, k)


def test_cascade_tta_equals_restricted_full_tta_level(slide, packed2):
    """process_cascade(order=(3, 0), tta=True) = the full TTA process_level of level 0 restricted to the ROI that the oracle
    builds from the level-3 TTA margins, with a tau that keeps some but not all level-0 survivors."""
    import math

    from ss25_hierarchical_multiscale_image_classification_b200 import pipeline
    from ss25_hierarchical_multiscale_image_classification_b200.cascade import process_cascade, threshold_of, tumor_margin
    coarse = pipeline.process_level(*slide[3], 3, packed2, tta=True)
    full = pipeline.process_level(*slide[0], 0, packed2, tta=True)
    h3, w3 = int(slide[3][0].shape[0]), int(slide[3][0].shape[1])
    nx, ny = (w3 + 223) // 224, (h3 + 223) // 224
    margins = tumor_margin(coarse.logits).cpu().numpy()

    def keep_of(theta):
        grid = oc.roi_grid(coarse.coords.cpu().numpy(), margins, theta, 224, nx, ny, 0)
        return oc.roi_mask(full.coords.cpu().numpy(), 0, oc.Roi(grid, 3, 224, 224))

    m = np.sort(margins.astype(np.float64))[::-1]
    tau = None
    for k in range(len(m) // 2, 0, -1):           # top-k margins positive, from half of the coarse survivors down
        if m[k - 1] > m[k]:
            t = 1.0 / (1.0 + math.exp(-0.5 * (m[k - 1] + m[k])))
            if 0 < keep_of(threshold_of(t)).sum() < len(full):
                tau = t
                break
    assert tau is not None, "no threshold splits level 0"
    res = process_cascade({L: slide[L] for L in (3, 0)}, packed2, order=(3, 0), tau=tau, tta=True)
    _assert_equal_results(res[3], coarse, "coarse")
    keep = keep_of(threshold_of(tau))
    idx = torch.from_numpy(np.nonzero(keep)[0]).cuda()
    for k in ("coords", "labels", "features", "logits"):
        assert torch.equal(getattr(res[0], k), getattr(full, k)[idx]), k
    assert res[0].candidates == full.candidates
