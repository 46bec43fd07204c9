"""Stage-2 parity on the GPU: the tcgen05 ResNet18 kernels (through the C ABI) vs fp64 references and the fp32 oracle.

Per-kernel tests feed the SAME bf16-rounded operands to the kernel and to an fp64 reference and bound every output
element by the bf16 output rounding plus fp32 accumulation (see REL_OUT / REL_ACC).  They run each kernel in both tile
orders, on batches where every CTA pair loops over several work items, and in device-count mode, as the forward does.  A
chained test checks that the forward is exactly those kernels in sequence.  End-to-end tests compare against the fp32
oracle / the golden vectors frozen from the reference with the tolerances BASELINE.json's north_star states: cosine >=
0.9995, max|d|/max|ref| <= 1e-2, argmax agreement >= 99.9 %."""
import itertools

import numpy as np
import pytest

from conftest import load_golden
from oracle import hipac_oracle as orc

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

SPECS = [(3, 64, 7, 2, 3, 224)] + [(64, 64, 3, 1, 1, 56)] * 4 + \
        [(64, 128, 3, 2, 1, 56), (128, 128, 3, 1, 1, 28), (64, 128, 1, 2, 0, 56), (128, 128, 3, 1, 1, 28), (128, 128, 3, 1, 1, 28)] + \
        [(128, 256, 3, 2, 1, 28), (256, 256, 3, 1, 1, 14), (128, 256, 1, 2, 0, 28), (256, 256, 3, 1, 1, 14), (256, 256, 3, 1, 1, 14)] + \
        [(256, 512, 3, 2, 1, 14), (512, 512, 3, 1, 1, 7), (256, 512, 1, 2, 0, 14), (512, 512, 3, 1, 1, 7), (512, 512, 3, 1, 1, 7)]


@pytest.fixture(scope="module")
def net_and_packed():
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    net = orc.make_resnet18(seed=0, classifier=True)
    packed = features.pack_resnet18(net.state_dict(), "cuda")
    return net, packed


def _folded(net, layer):
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    conv, bn = features.conv_bn_names()[layer]
    sd = net.state_dict()
    scale = sd[f"{bn}.weight"] / torch.sqrt(sd[f"{bn}.running_var"] + 1e-5)
    w = (sd[f"{conv}.weight"] * scale[:, None, None, None]).bfloat16().float()
    b = sd[f"{bn}.bias"] - sd[f"{bn}.running_mean"] * scale
    return w.cuda(), b.cuda()


# ---------------------------------------------------------------------------------------------------------------------
# Per-kernel tests against fp64, at the batch sizes and with the launch state the forward uses
# ---------------------------------------------------------------------------------------------------------------------
# Every output element must satisfy |got - ref| <= 2^-8 |ref| + 2^-11 A, where ref and A = conv(|x|, |w|) + |b| (+ |res|)
# are computed in fp64 from the same bf16 activations, bf16 folded weights and fp32 bias the kernel reads.  2^-8 |ref| is the
# single bf16 rounding of the output (half an ulp of an 8-bit significand).  2^-11 A covers the fp32 accumulation of
# K <= 4864 products: its worst case is K 2^-24 A ~ 2^-11.75 A, its typical size sqrt(K) 2^-24 A ~ 2^-18 A.  A dropped
# 64-channel K-block of a 4608-term sum is ~2^-8 A on random data, which the bound does not admit.  ReLU and max are
# 1-Lipschitz, so the bound carries through them (for the stem: the max of the pre-pool bounds over each pool window).
# The per-kernel tests are named `..._vs_torch_fp32` after the kernel's fp32 accumulation that this bound models; their
# reference is torch in fp64.
REL_OUT, REL_ACC = 2.0 ** -8, 2.0 ** -11
SENTINEL = 0x7F81                  # a bf16 NaN bit pattern: no kernel writes it, so an untouched row still holds it
CONV_LAYERS = [l for l in range(20) if l not in (0, 7)]   # 0 and 7 exist only fused: the stem and projection tests
RES_LAYERS = (2, 4, 6, 9, 11, 14, 16, 19)
# one layer per kernel and epilogue the forward runs: layer1 without / with residual (64-channel row kernel, two epilogue
# warpgroups, TMA epilogue), layer2.0.conv1 (stride-2 row kernel), layer2 without residual (per-thread epilogue) and with
# residual (staged TMA epilogue), layer3 / layer4 3x3 at stride 2 and at stride 1 without / with residual (im2col)
MANY_ITEM_LAYERS = (1, 2, 5, 8, 9, 10, 13, 14, 15, 18, 19)


def _pairs():
    """CTA pairs of a launch with more work items than that: launch_pairs puts at most one pair on every two SMs."""
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count // 2


def _kernel(cout, hout):
    """Work geometry of the kernel that computes a conv with `cout` channels at `hout` x `hout`: ("rows", tiles per patch, 1)
    for the row kernels, ("im2col", output pixels per patch, weight tiles) for the im2col kernel."""
    if cout == 64:
        return ("rows", 28, 1)                                  # 2-row tiles of 56 rows
    if cout == 128:
        return ("rows", 7, 1)                                   # 4-row tiles of 28 rows
    return ("im2col", hout * hout, cout // 256)


STEM_KERNEL = ("rows", 7, 1)                                    # blocks of 8 pooled rows of 56


def _schedule(kernel, n):
    """(tiles, work items) of one launch on n patches, counted as the kernels count them: an item is the pair of tiles one
    CTA pair computes, a phantom second tile when the count is odd; im2col tiles are 128 output pixels x 256 channels."""
    kind, per_patch, n_tiles = kernel
    tiles = n * per_patch if kind == "rows" else -(-n * per_patch // 128)
    return tiles, (tiles + 1) // 2 * n_tiles


def _many_items_n(kernel, min_items):
    """The smallest batch on which every CTA pair walks at least `min_items` items: 4 reach both TMEM accumulator parities,
    8 give each of the two epilogue warpgroups of the 64-channel kernel both staging buffers in both parities.  The item
    count is not a multiple of the pair count (the pairs end on different iterations) and, where the geometry allows, the
    tile count is odd (a phantom tile); for im2col the last 128-pixel tile is only partly inside the batch."""
    pairs = _pairs()
    kind, per_patch, _ = kernel
    odd_possible = kind == "im2col" or per_patch % 2 == 1
    n = 1
    while True:
        tiles, items = _schedule(kernel, n)
        if items >= min_items * pairs and items % pairs != 0 and (tiles % 2 == 1 or not odd_possible) and \
                (kind == "rows" or n * per_patch % 128 != 0):
            break
        n += 1
    tiles, items = _schedule(kernel, n)
    assert items // pairs >= min_items and items % pairs != 0, (kernel, n, pairs)
    assert tiles % 2 == 1 or not odd_possible, (kernel, n)
    return n


def _ref64(terms, biases, res, relu):
    """fp64 reference (NCHW) of sum(conv(x, w)) + sum(b) (+ res) (+ ReLU) over terms (x NHWC bf16, w, stride, pad) and the
    per-element error bound 2^-8 |ref| + 2^-11 A."""
    ref = acc = 0.0
    for x, w, stride, pad in terms:
        xd, wd = x.permute(0, 3, 1, 2).double(), w.double()
        ref = ref + torch.nn.functional.conv2d(xd, wd, stride=stride, padding=pad)
        acc = acc + torch.nn.functional.conv2d(xd.abs(), wd.abs(), stride=stride, padding=pad)
        del xd
    for b in biases:
        ref = ref + b.double()[:, None, None]
        acc = acc + b.double().abs()[:, None, None]
    if res is not None:
        rd = res.permute(0, 3, 1, 2).double()
        ref, acc = ref + rd, acc + rd.abs()
    if relu:
        ref = torch.relu(ref)
    return ref, REL_OUT * ref.abs() + REL_ACC * acc


def _assert_within(got, ref, bound, what):
    err = (got.permute(0, 3, 1, 2).double() - ref).abs()
    ratio = float((err / bound.clamp_min(1e-300)).max())
    print(f"{what}: max |got - ref| / bound = {ratio:.4f}")
    bad = (err > bound).nonzero()
    assert bad.numel() == 0, f"{what}: {bad.shape[0]} elements outside the bound, first (n, c, y, x) = {bad[0].tolist()}, " \
                             f"max ratio {ratio:.3f}"


def _run_both_orders(run):
    """The kernel walking its tiles ascending and descending: both outputs are returned after checking they are bitwise
    equal (no tile's arithmetic depends on the walk order)."""
    fwd, rev = run(reverse=False), run(reverse=True)
    torch.cuda.synchronize()
    assert torch.equal(fwd.view(torch.int16), rev.view(torch.int16)), "the output depends on the tile order"
    return fwd


def _check_device_count(run, host_out, kernel, n):
    """Device-count mode with a nonzero chunk base: for effective patch counts clamp(count - base, 0, n) of 0, one with an
    odd tile count (if the geometry has one), n, and count > base + n, in both tile orders, the first rows equal the
    host-count output bit for bit and every other row still holds the sentinel the output was filled with."""
    base = 5
    e_odd = next((e for e in range(n // 2, n) if _schedule(kernel, e)[0] % 2 == 1), n // 2)
    want = host_out.view(torch.int16)
    for count, eff in ((base - 2, 0), (base + e_odd, e_odd), (base + n, n), (base + n + 1, n)):
        d_count = torch.tensor([count, 12345], dtype=torch.int32, device="cuda")
        for reverse in (False, True):
            out = torch.empty_like(host_out)
            out.view(torch.int16).fill_(SENTINEL)
            run(reverse=reverse, count=d_count, base=base, out=out)
            torch.cuda.synchronize()
            got = out.view(torch.int16)
            assert torch.equal(got[:eff], want[:eff]), f"count {count}, base {base}, reverse {reverse}: rows differ"
            assert bool((got[eff:] == SENTINEL).all()), f"count {count}, base {base}, reverse {reverse}: rows >= {eff} written"


def _s2d16(x):
    """bf16 NHWC3 [n,224,224,3] -> the S2D16 layout [n,112,115,16] (see HIPAC_LAYOUT_S2D16_BF16)."""
    n = x.shape[0]
    y = torch.zeros((n, 112, 115, 16), dtype=torch.bfloat16, device=x.device)
    y[:, :, 2:114, :12] = x.reshape(n, 112, 2, 112, 2, 3).permute(0, 1, 3, 2, 4, 5).reshape(n, 112, 112, 12)
    return y


@pytest.mark.parametrize("layer,n", [(l, n) for l in CONV_LAYERS for n in (1, 3)] + [(l, "many") for l in MANY_ITEM_LAYERS])
def test_conv_layer_vs_torch_fp32(net_and_packed, layer, n):
    """One conv(+folded BN)(+residual)(+ReLU) layer in both tile orders vs fp64.  n = "many": the batch on which every CTA
    pair loops over several items (_many_items_n), also run in device-count mode."""
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    net, packed = net_and_packed
    cin, cout, k, stride, pad, hin = SPECS[layer]
    hout = (hin + 2 * pad - k) // stride + 1
    kernel = _kernel(cout, hout)
    many = n == "many"
    if many:
        n = _many_items_n(kernel, 8 if cout == 64 else 4)
    g = torch.Generator(device="cuda").manual_seed(100 + layer)
    x = torch.randn((n, hin, hin, cin), generator=g, device="cuda").bfloat16()
    res = torch.randn((n, hout, hout, cout), generator=g, device="cuda").bfloat16() if layer in RES_LAYERS else None
    relu = layer not in (12, 17)
    w, b = _folded(net, layer)
    ref, bound = _ref64([(x, w, stride, pad)], [b], res, relu)

    def run(**kw):
        return features.conv_layer(packed, layer, x, res, relu, **kw)

    out = _run_both_orders(run)
    _assert_within(out, ref, bound, f"layer {layer}, n = {n}")
    if many:
        _check_device_count(run, out, kernel, n)


@pytest.mark.parametrize("layer,fused_hook", [(0, "hipac_resnet18_stem"), (7, "hipac_resnet18_conv_ds_fused")])
def test_conv_layer_refuses_fused_only_layers(net_and_packed, layer, fused_hook):
    """conv1 exists only fused with the max pool, layer2.0's projection shortcut only fused into layer2.0.conv2: the per-layer
    hook refuses both and names the fused hook that computes them."""
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    _, packed = net_and_packed
    cin, _, _, _, _, hin = SPECS[layer]
    x = torch.zeros((1, hin, hin, cin), dtype=torch.bfloat16, device="cuda")
    with pytest.raises(RuntimeError, match=fused_hook):
        features.conv_layer(packed, layer, x, None, layer == 0)


def _metrics(got, ref):
    cos = (got * ref).sum(1) / (np.linalg.norm(got, axis=1) * np.linalg.norm(ref, axis=1))
    maxrel = np.abs(got - ref).max(1) / np.abs(ref).max(1)
    return cos.min(), maxrel.max()


def _gpu_features(packed, images_u8, layout):
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    lut = torch.from_numpy(orc.normalize_lut()).cuda()
    u8 = torch.from_numpy(images_u8).cuda().long()
    x = torch.stack([lut[:, c][u8[..., c]] for c in range(3)], dim=-1).bfloat16()     # NHWC3 bf16
    if layout == "s2d16":
        x = _s2d16(x)
    f, lg = features.classify_tensor(x, packed, chunk=5)
    torch.cuda.synchronize()
    return f.cpu().numpy(), lg.cpu().numpy()


@pytest.mark.parametrize("layout", ["s2d16", "nhwc3"])
def test_features_vs_golden_reference(net_and_packed, layout):
    net, packed = net_and_packed
    g = load_golden("stage2_features.npz")
    feats, logits = _gpu_features(packed, g["images"], layout)
    cos, maxrel = _metrics(feats, g["features"])
    assert cos >= 0.9995 and maxrel <= 1e-2, (cos, maxrel)
    assert np.array_equal(logits.argmax(1), g["logits"].argmax(1))


def test_features_vs_fp32_oracle_random_patches(net_and_packed):
    net, packed = net_and_packed
    rng = np.random.default_rng(0)
    n = 23                                                    # not a multiple of the chunk (5)
    base = rng.integers(0, 256, size=(n, 28, 28, 3), dtype=np.uint8)
    imgs = np.repeat(np.repeat(base, 8, axis=1), 8, axis=2)  # blocky structure + noise
    imgs = np.clip(imgs.astype(np.int32) + rng.integers(-20, 21, size=imgs.shape), 0, 255).astype(np.uint8)
    ref_f, ref_l = orc.resnet18_features_fp32(net, imgs)
    feats, logits = _gpu_features(packed, imgs, "s2d16")
    cos, maxrel = _metrics(feats, ref_f)
    assert cos >= 0.9995 and maxrel <= 1e-2, (cos, maxrel)
    margin = np.abs(ref_l[:, 0] - ref_l[:, 1])
    agree = (logits.argmax(1) == ref_l.argmax(1)) | (margin < 1e-3 * np.abs(ref_l).max())
    assert agree.mean() >= 0.999


def test_headless_packed_weights_and_errors():
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    net = orc.make_resnet18(seed=1, classifier=False)
    sd = {k: v for k, v in net.state_dict().items() if not k.startswith("fc.")}
    packed = features.pack_resnet18(sd, "cuda")
    assert packed.num_classes == 0
    x = torch.zeros((2, 112, 115, 16), dtype=torch.bfloat16, device="cuda")
    f = features.extract_features_tensor(x, packed)
    assert f.shape == (2, 512) and torch.isfinite(f).all()
    with pytest.raises(ValueError):
        features.classify_tensor(x, packed)
    with pytest.raises(ValueError):
        features.extract_features_tensor(x.float(), packed)
    assert features.extract_features_tensor(x[:0], packed).shape == (0, 512)


@pytest.mark.parametrize("n", [1, 2, 23, "many"])
def test_fused_stem_vs_torch_fp32(net_and_packed, n):
    """conv1 + folded BN + ReLU + 3x3/s2 max pool in one kernel, in both block orders, vs fp64 on the same bf16 operands."""
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    net, packed = net_and_packed
    many = n == "many"
    if many:
        n = _many_items_n(STEM_KERNEL, 4)
    g = torch.Generator(device="cuda").manual_seed(n)
    x = torch.randn((n, 224, 224, 3), generator=g, device="cuda").bfloat16()
    w, b = _folded(net, 0)
    conv, bound = _ref64([(x, w, 2, 3)], [b], None, True)
    ref = torch.nn.functional.max_pool2d(conv, 3, 2, 1)
    bound = torch.nn.functional.max_pool2d(bound, 3, 2, 1)
    del conv
    xin = _s2d16(x)

    def run(**kw):
        return features.stem(packed, xin, **kw)

    out = _run_both_orders(run)
    _assert_within(out, ref, bound, f"stem, n = {n}")
    if many:
        _check_device_count(run, out, STEM_KERNEL, n)


@pytest.mark.parametrize("n", [1, 5, "many"])
@pytest.mark.parametrize("stage", [0, 1, 2])
def test_fused_projection_shortcut_vs_torch_fp32(net_and_packed, stage, n):
    """relu(conv3x3(x) + conv1x1_s2(block_in) + both folded BN biases) accumulated in one TMEM tile, in both tile orders,
    vs fp64."""
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    net, packed = net_and_packed
    lc, ld = 6 + 5 * stage, 7 + 5 * stage
    cin, cout, _, _, _, hin = SPECS[lc]
    dcin, _, _, _, _, dhin = SPECS[ld]
    kernel = _kernel(cout, hin)
    many = n == "many"
    if many:
        n = _many_items_n(kernel, 4)
    g = torch.Generator(device="cuda").manual_seed(50 + stage)
    x = torch.randn((n, hin, hin, cin), generator=g, device="cuda").bfloat16()
    xb = torch.randn((n, dhin, dhin, dcin), generator=g, device="cuda").bfloat16()
    w1, b1 = _folded(net, lc)
    w2, b2 = _folded(net, ld)
    ref, bound = _ref64([(x, w1, 1, 1), (xb, w2, 2, 0)], [b1, b2], None, True)

    def run(**kw):
        return features.conv_ds_fused(packed, stage, x, xb, **kw)

    out = _run_both_orders(run)
    _assert_within(out, ref, bound, f"projection stage {stage}, n = {n}")
    if many:
        _check_device_count(run, out, kernel, n)


def _chained_trunk(packed, x_s2d):
    """The trunk on one chunk as forward_impl runs it, through the per-kernel test hooks: same launches in the same order,
    the stem walking its tiles descending and every later launch flipping the order -> bf16 [n,7,7,512]."""
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    orders = itertools.cycle((True, False))

    def conv(layer, x, res):
        return features.conv_layer(packed, layer, x, res, True, reverse=next(orders))

    a = features.stem(packed, x_s2d, reverse=next(orders))
    b = conv(1, a, None)
    c = conv(2, b, a)
    b = conv(3, c, None)
    a = conv(4, b, c)
    for s in range(3):
        l0 = 5 + 5 * s
        b = conv(l0, a, None)
        c = features.conv_ds_fused(packed, s, b, a, reverse=next(orders))
        b = conv(l0 + 3, c, None)
        a = conv(l0 + 4, b, c)
    return a


@pytest.mark.parametrize("num_classes", [1, 2, 9, 1000])
def test_forward_is_the_chain_of_tested_kernels(num_classes):
    """classify_tensor on several chunks with a partial last one, in both input layouts, against the per-kernel hooks
    chained in the forward's order: the features are the fp32 7x7 mean of the chained layer4 output (bit for bit, and
    within the fp32 bound of the fp64 mean), the logits are features . W^T + b within the fp32 bound of the fp64 product."""
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    net = orc.make_resnet18(seed=0, classifier=True)
    sd = dict(net.state_dict())
    gen = torch.Generator().manual_seed(num_classes)
    sd["fc.weight"] = torch.randn((num_classes, 512), generator=gen) * 512 ** -0.5
    sd["fc.bias"] = torch.randn((num_classes,), generator=gen)
    packed = features.pack_resnet18(sd, "cuda")
    assert packed.num_classes == num_classes
    n, chunk = 200, 96                                          # chunks of 96, 96 and 8 patches
    rng = np.random.default_rng(num_classes)
    u8 = torch.from_numpy(rng.integers(0, 256, size=(n, 224, 224, 3), dtype=np.uint8)).cuda().long()
    lut = torch.from_numpy(orc.normalize_lut()).cuda()
    x3 = torch.stack([lut[:, c][u8[..., c]] for c in range(3)], dim=-1).bfloat16()
    xs = _s2d16(x3)
    f3, l3 = features.classify_tensor(x3, packed, chunk)
    fs, ls = features.classify_tensor(xs, packed, chunk)
    trunk = torch.cat([_chained_trunk(packed, xs[i:i + chunk]) for i in range(0, n, chunk)]).reshape(n, 49, 512)
    torch.cuda.synchronize()
    assert torch.equal(f3, fs) and torch.equal(l3, ls), "the NHWC3 and S2D16 inputs give different results"
    # k_avgpool_fc's arithmetic: an fp32 sum over the 49 pixels in order, times fp32(1/49)
    s = torch.zeros((n, 512), dtype=torch.float32, device="cuda")
    for px in range(49):
        s = s + trunk[:, px].float()
    assert torch.equal(fs, s * torch.tensor(1.0 / 49.0, dtype=torch.float32, device="cuda")), \
        "the forward's features are not the mean of the chained kernels' output"
    # 48 roundings of the running sum, the rounded 1/49 and the product: <= 50 * 2^-24 of the mean magnitude
    t = trunk.double()
    assert bool(((fs.double() - t.mean(1)).abs() <= 64 * 2.0 ** -24 * t.abs().mean(1)).all())
    # each lane sums 16 products, then 5 shuffle additions and the bias: <= 22 roundings of 2^-24 of the magnitudes' sum
    w, b = sd["fc.weight"].double().cuda(), sd["fc.bias"].double().cuda()
    f = fs.double()
    bound = 32 * 2.0 ** -24 * (f.abs() @ w.abs().T + b.abs())
    assert bool(((ls.double() - (f @ w.T + b)).abs() <= bound).all())




@pytest.mark.parametrize("cap,n,chunk", [(11, 6, 4096), (11, 6, 4), (11, 11, 4096), (11, 0, 4096), (300, 150, 128), (5, 9, 4096)])
def test_device_count_forward_equals_host_count(net_and_packed, cap, n, chunk):
    """hipac_resnet18_forward_dcount (patch count read from device memory, everything sized for a capacity) gives the
    same bits as the host-count call on the first min(count, capacity) patches and leaves the other rows untouched."""
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    net, packed = net_and_packed
    g = torch.Generator(device="cuda").manual_seed(cap * 1000 + n)
    x = torch.randn((cap, 112, 115, 16), generator=g, device="cuda").to(torch.bfloat16)
    x[:, :, :2] = 0
    x[:, :, 114] = 0
    x[..., 12:] = 0
    m = min(n, cap)
    count = torch.tensor([n, 12345], dtype=torch.int32, device="cuda")
    f_ref, l_ref = features.classify_tensor(x[:m], packed, chunk) if m else (None, None)
    f, l = features._forward(x, packed, True, chunk, count=count)
    torch.cuda.synchronize()
    if m:
        assert torch.equal(f[:m], f_ref) and torch.equal(l[:m], l_ref)
    # rows beyond the device count are never written
    f2 = torch.full((cap, 512), 7.0, device="cuda")
    lib = features._lib.lib()
    ws_bytes = lib.hipac_resnet18_workspace_bytes(cap, chunk)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device="cuda")
    rc = lib.hipac_resnet18_forward_dcount(packed.blob.data_ptr(), packed.num_classes, x.data_ptr(), 2, cap, count.data_ptr(),
                                           f2.data_ptr(), None, ws.data_ptr(), ws_bytes, chunk,
                                           torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    torch.cuda.synchronize()
    assert bool((f2[m:] == 7.0).all())
    if m:
        assert torch.equal(f2[:m], f_ref)
