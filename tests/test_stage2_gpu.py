"""Stage-2 parity on the GPU: the tcgen05 ResNet18 kernels (through the C ABI) vs plain PyTorch fp32.

Per-layer tests feed the SAME bf16-rounded operands to both sides, so only accumulation order and the
final bf16 rounding differ (tolerance: 1.5 bf16 ulp of the layer's dynamic range).  End-to-end tests
compare against the fp32 oracle / the golden vectors frozen from the reference with the tolerances
BASELINE.json's north_star states: cosine >= 0.9995, max|d|/max|ref| <= 1e-2, argmax agreement >= 99.9 %."""
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


@pytest.mark.parametrize("n", [1, 3])
@pytest.mark.parametrize("layer", [l for l in range(20) if l not in (0, 7)])   # 0 and 7 exist only fused: tests below
def test_conv_layer_vs_torch_fp32(net_and_packed, layer, n):
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    net, packed = net_and_packed
    cin, cout, k, stride, pad, hin = SPECS[layer]
    g = torch.Generator(device="cuda").manual_seed(100 + layer)
    x = torch.randn((n, hin, hin, cin), generator=g, device="cuda").bfloat16()
    w, b = _folded(net, layer)
    ref = torch.nn.functional.conv2d(x.float().permute(0, 3, 1, 2), w, b, stride=stride, padding=pad)
    hout = ref.shape[-1]
    use_res = layer in (2, 4, 6, 9, 11, 14, 16, 19)
    res = torch.randn((n, hout, hout, cout), generator=g, device="cuda").bfloat16() if use_res else None
    if res is not None:
        ref = ref + res.float().permute(0, 3, 1, 2)
    relu = layer not in (12, 17)
    if relu:
        ref = torch.relu(ref)
    out = features.conv_layer(packed, layer, x, res, relu)
    torch.cuda.synchronize()
    got = out.float().permute(0, 3, 1, 2)
    scale = float(ref.abs().max())
    err = float((got - ref).abs().max())
    assert err <= 1.5 * 2.0 ** -8 * scale + 1e-3, f"layer {layer}: max err {err} at scale {scale}"


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
        n = x.shape[0]
        y = torch.zeros((n, 112, 115, 16), dtype=torch.bfloat16, device="cuda")
        y[:, :, 2:114, :12] = x.reshape(n, 112, 2, 112, 2, 3).permute(0, 1, 3, 2, 4, 5).reshape(n, 112, 112, 12)
        x = y
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


@pytest.mark.parametrize("n", [1, 2, 23])
def test_fused_stem_vs_torch_fp32(net_and_packed, n):
    """conv1 + folded BN + ReLU + 3x3/s2 max pool in one kernel vs torch on the same bf16 operands."""
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    net, packed = net_and_packed
    g = torch.Generator(device="cuda").manual_seed(n)
    x = torch.randn((n, 224, 224, 3), generator=g, device="cuda").bfloat16()
    w, b = _folded(net, 0)
    conv = torch.relu(torch.nn.functional.conv2d(x.float().permute(0, 3, 1, 2), w, b, stride=2, padding=3))
    ref = torch.nn.functional.max_pool2d(conv.bfloat16().float(), 3, 2, 1)       # kernel rounds to bf16 before pooling
    xin = torch.zeros((n, 112, 115, 16), dtype=torch.bfloat16, device="cuda")
    xin[:, :, 2:114, :12] = x.reshape(n, 112, 2, 112, 2, 3).permute(0, 1, 3, 2, 4, 5).reshape(n, 112, 112, 12)
    out = features.stem(packed, xin)
    torch.cuda.synchronize()
    got = out.float().permute(0, 3, 1, 2)
    scale = float(ref.abs().max())
    err = float((got - ref).abs().max())
    assert err <= 1.5 * 2.0 ** -8 * scale + 1e-3, f"stem: max err {err} at scale {scale}"


@pytest.mark.parametrize("n", [1, 5])
@pytest.mark.parametrize("stage", [0, 1, 2])
def test_fused_projection_shortcut_vs_torch_fp32(net_and_packed, stage, n):
    """relu(conv3x3(x) + conv1x1_s2(block_in) + both folded BN biases) accumulated in one TMEM tile."""
    from ss25_hierarchical_multiscale_image_classification_b200 import features
    net, packed = net_and_packed
    lc, ld = 6 + 5 * stage, 7 + 5 * stage
    cin, cout, _, _, _, hin = SPECS[lc]
    dcin, _, _, _, _, dhin = SPECS[ld]
    g = torch.Generator(device="cuda").manual_seed(50 + stage)
    x = torch.randn((n, hin, hin, cin), generator=g, device="cuda").bfloat16()
    xb = torch.randn((n, dhin, dhin, dcin), generator=g, device="cuda").bfloat16()
    w1, b1 = _folded(net, lc)
    w2, b2 = _folded(net, ld)
    ref = torch.nn.functional.conv2d(x.float().permute(0, 3, 1, 2), w1, b1, stride=1, padding=1) + \
        torch.nn.functional.conv2d(xb.float().permute(0, 3, 1, 2), w2, b2, stride=2, padding=0)
    ref = torch.relu(ref)
    out = features.conv_ds_fused(packed, stage, x, xb)
    torch.cuda.synchronize()
    got = out.float().permute(0, 3, 1, 2)
    scale = float(ref.abs().max())
    err = float((got - ref).abs().max())
    assert err <= 1.5 * 2.0 ** -8 * scale + 1e-3, f"stage {stage}: max err {err} at scale {scale}"


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
