"""BASELINE configs[0] (4096 x 4096 level-3 image, 361 candidates) end to end on the GPU, every survivor compared with
tests/golden/config0.npz (file names = coords + labels, 512-d features).  The fixture is the CPU oracle's run of the
whole config (tests/golden/make_golden.py config0): its stage 1 is pinned to the unmodified reference by the stage-1
fixtures, and it keeps the 116 survivors the reference kept on this slide."""
import numpy as np
import pytest

from conftest import load_golden

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


def test_config0_whole_config_equals_golden():
    from oracle import hipac_oracle as orc
    from ss25_hierarchical_multiscale_image_classification_b200 import features, pipeline
    from ss25_hierarchical_multiscale_image_classification_b200.synthetic import SyntheticSlide
    g = load_golden("config0.npz")
    L = int(g["level"])
    net = orc.make_resnet18(seed=int(g["weight_seed"]), classifier=True)
    wsum = float(sum(v.double().abs().sum() for v in net.state_dict().values()))
    assert abs(wsum - float(g["weight_abs_sum"])) < 1e-6 * wsum, "seeded weights differ from the fixture's"
    slide = SyntheticSlide(int(g["size0"]), int(g["size0"]), seed=int(g["slide_seed"]))
    img_d = torch.from_numpy(slide.level_array(L)).cuda()
    msk_d = torch.from_numpy(slide.lesion_mask(L)).cuda()
    packed = features.pack_resnet18(net.state_dict(), "cuda")
    r = pipeline.process_level(img_d, msk_d, L, packed)
    torch.cuda.synchronize()
    coords, labels, feats = r.coords.cpu().numpy(), r.labels.cpu().numpy(), r.features.float().cpu().numpy()

    def names(cs, ls):
        return [orc.patch_name(slide.name, int(x), int(y), int(l)) for (x, y), l in zip(cs, ls)]

    ours = {n: i for i, n in enumerate(names(coords, labels))}
    want = names(g["coords"], g["labels"])
    assert r.candidates == int(g["candidates"]) == 361
    assert len(coords) == len(want) > 50
    assert sorted(ours) == sorted(want)                                          # coords + labels of every survivor
    idx = [ours[n] for n in want]
    f, ref = feats[idx].astype(np.float64), g["features"].astype(np.float64)
    cos = (f * ref).sum(1) / (np.linalg.norm(f, axis=1) * np.linalg.norm(ref, axis=1))
    maxrel = np.abs(f - ref).max(1) / np.abs(ref).max(1)
    assert cos.min() >= 0.9995 and maxrel.max() <= 1e-2, (cos.min(), maxrel.max())   # north_star's feature tolerance
