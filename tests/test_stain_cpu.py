"""Macenko stain normalisation without a GPU: the exact fast form the kernels compute (oracle.stain.normalizer_matrix /
apply) against the literal torchstain restatement over all 2^24 colours, the estimate's recovery of a known stain and its
independence of eigenvector signs, and every argument the four C entry points refuse before touching the device."""
import ctypes as C

import numpy as np
import pytest

from oracle import stain as st

CHUNK = 1 << 22


def _normalisers(img_seed):
    """The three normalisers of one image: to torchstain's reference, to a target estimated from another centre's image,
    and one with extreme maxC ratios (its outputs hit 0 and the 255 clip)."""
    he, max_c, _ = st.estimate_literal(st.he_image(img_seed, 256, 256, st.HE_TRUE))
    he_b, max_c_b, _ = st.estimate_literal(st.he_image(img_seed + 100, 256, 256, st.HE_TRUE_B))
    return [("reference", he, max_c, st.HE_REF, st.MAXC_REF),
            ("estimated target", he, max_c, he_b, max_c_b),
            ("extreme", he, max_c, st.HE_REF, st.MAXC_REF * np.array([8.0, 1.0 / 16]))]


@pytest.mark.parametrize("img_seed", [0, 1, 2])
def test_fast_form_equals_literal_on_every_colour(img_seed):
    od = st.od_table()
    for name, he, max_c, he_ref, max_c_ref in _normalisers(img_seed):
        M = st.normalizer_matrix(he, max_c, he_ref, max_c_ref)
        mismatches, seen = 0, np.zeros(256, bool)
        for lo in range(0, 1 << 24, CHUNK):
            c = st.all_colours(lo, lo + CHUNK)
            lit = st.normalize_literal(c, he, max_c, he_ref, max_c_ref)
            fast = st.apply(c, M, od)
            d = np.abs(lit.astype(np.int16) - fast)
            assert d.max() <= 1, (name, lo)
            mismatches += int(np.count_nonzero(d))
            seen[fast.reshape(-1)] = True
        print(f"image {img_seed} {name}: {mismatches} mismatching channel values of 3 x 2^24")
        assert mismatches == 0, (name, mismatches)
        if name == "extreme":
            assert seen[0] and seen[255]


@pytest.mark.parametrize("seed,he_true", [(3, st.HE_TRUE), (4, st.HE_TRUE_B)])
def test_estimate_recovers_the_generating_stain(seed, he_true):
    he, max_c, n_hat = st.estimate_literal(st.he_image(seed, 512, 512, he_true))
    want = he_true / np.linalg.norm(he_true, axis=0)
    cos = (he * want).sum(0) / np.linalg.norm(he, axis=0)
    assert cos.min() >= 0.99, cos
    assert n_hat > 512 * 512 // 2 and np.all(max_c > 0)


def test_estimate_does_not_depend_on_eigenvector_signs():
    img = st.he_image(5, 300, 200, st.HE_TRUE)
    he, max_c, _ = st.estimate_literal(img)
    for flip in ((True, False), (False, True), (True, True)):
        he2, max_c2, _ = st.estimate_literal(img, flip=flip)
        assert np.abs(he2 - he).max() <= 1e-12 and np.abs(max_c2 - max_c).max() <= 1e-12 * max_c.max(), flip


def test_invalid_estimates():
    assert st.estimate_literal(np.full((20, 30, 3), 255, np.uint8)) is None          # no stained pixel
    one = np.full((20, 30, 3), 255, np.uint8)
    one[3, 4] = (40, 20, 60)
    assert st.estimate_literal(one) is None                                         # n_hat = 1


# ---------------------------------------------------------------------------------------------------------------------
# refusals of the C entry points (validated before any CUDA call)
# ---------------------------------------------------------------------------------------------------------------------
FAKE = 1 << 30
U8_BYTES = 224 * 224 * 3
v = lambda p: C.c_void_p(p) if p else None     # noqa: E731


def _estimate(lib, rgb=FAKE, H=64, W=48, pitch=None, io=240, alpha=1.0, beta=0.15, out=2 * FAKE, ws=3 * FAKE, ws_bytes=None):
    pitch = 3 * W if pitch is None else pitch
    ws_bytes = lib.hipac_stain_workspace_bytes(max(H, 1), max(W, 1)) if ws_bytes is None else ws_bytes
    return lib.hipac_stain_estimate(v(rgb), H, W, pitch, io, alpha, beta, v(out), v(ws), ws_bytes, None)


@pytest.mark.parametrize("kw,msg", [
    (dict(rgb=0), b"null pointer"),
    (dict(out=0), b"null pointer"),
    (dict(ws=0), b"null pointer"),
    (dict(H=0), b"empty image"),
    (dict(W=-3), b"empty image"),
    (dict(H=1 << 16, W=1 << 15), b"2^31 pixels"),
    (dict(pitch=3 * 48 - 1), b"pitch smaller than a row"),
    (dict(io=0), b"Io must be in 1..255"),
    (dict(io=256), b"Io must be in 1..255"),
    (dict(alpha=0.0), b"alpha must be in (0, 50)"),
    (dict(alpha=50.0), b"alpha must be in (0, 50)"),
    (dict(alpha=float("nan")), b"alpha must be in (0, 50)"),
    (dict(beta=-0.01), b"beta must be finite"),
    (dict(beta=float("inf")), b"beta must be finite"),
    (dict(beta=float("nan")), b"beta must be finite"),
    (dict(ws=3 * FAKE + 128), b"256-byte aligned"),
    (dict(ws_bytes=1024), b"workspace too small"),
])
def test_estimate_refuses_bad_arguments(built_lib, kw, msg):
    assert _estimate(built_lib, **kw) == -1
    assert msg in built_lib.hipac_last_error()


def test_workspace_bytes(built_lib):
    lib = built_lib
    assert lib.hipac_stain_workspace_bytes(0, 5) == 0 and b"empty image" in lib.hipac_last_error()
    assert lib.hipac_stain_workspace_bytes(1 << 16, 1 << 15) == 0 and b"2^31" in lib.hipac_last_error()
    small, big = lib.hipac_stain_workspace_bytes(7, 13), lib.hipac_stain_workspace_bytes(2048, 2048)
    assert small >= 16 * 7 * 13 and 16 * 2048 * 2048 <= big <= 16 * 2048 * 2048 + (64 << 10) and big % 256 == 0


@pytest.mark.parametrize("kw,msg", [
    (dict(src=0), b"null pointer"),
    (dict(params=0), b"null pointer"),
    (dict(io=0), b"Io must be in 1..255"),
    (dict(io=300), b"Io must be in 1..255"),
])
def test_normalizer_refuses_bad_arguments(built_lib, kw, msg):
    a = dict(src=FAKE, target=0, io=240, params=2 * FAKE)
    a.update(kw)
    assert built_lib.hipac_stain_normalizer(v(a["src"]), v(a["target"]), a["io"], v(a["params"]), None) == -1
    assert msg in built_lib.hipac_last_error()


def _apply(lib, d_in=FAKE, n=4, count=None, base=0, params=2 * FAKE, out_u8=3 * FAKE, batch=4 * FAKE, layout=2):
    return lib.hipac_stain_apply(v(d_in), n, v(count), base, v(params), v(out_u8), v(batch), layout, None)


@pytest.mark.parametrize("kw,msg", [
    (dict(d_in=0), b"null pointer"),
    (dict(params=0), b"null pointer"),
    (dict(n=-1), b"negative n_patches"),
    (dict(base=-1), b"n_base must be non-negative"),
    (dict(layout=3), b"unknown batch layout"),
    (dict(layout=-1), b"unknown batch layout"),
    (dict(layout=0), b"d_batch needs a layout"),
    (dict(batch=0), b"d_batch needs a layout"),
    (dict(batch=0, layout=0, out_u8=0), b"no output"),
    (dict(d_in=FAKE + 8), b"16-byte aligned"),
    (dict(out_u8=3 * FAKE + 4), b"16-byte aligned"),
    (dict(batch=4 * FAKE + 2), b"16-byte aligned"),
    (dict(out_u8=FAKE + 16), b"d_out_u8 partially overlaps d_in"),
    (dict(out_u8=FAKE - 4 * U8_BYTES + 16), b"d_out_u8 partially overlaps d_in"),
    (dict(batch=FAKE + 4 * U8_BYTES - 16), b"d_batch overlaps d_in"),
    (dict(batch=FAKE - 4 * 412160 + 16), b"d_batch overlaps d_in"),
    (dict(batch=FAKE - 4 * 301056 + 16, layout=1), b"d_batch overlaps d_in"),
    (dict(batch=3 * FAKE + 4 * U8_BYTES - 16), b"d_batch overlaps d_out_u8"),
])
def test_apply_refuses_bad_arguments(built_lib, kw, msg):
    assert _apply(built_lib, **kw) == -1
    assert msg in built_lib.hipac_last_error()


def test_apply_accepts_exact_in_place_and_empty_batches(built_lib):
    """Exact in place is allowed for the uint8 output; an empty batch returns before any device call; a batch right
    after the input does not overlap it."""
    lib = built_lib
    assert _apply(lib, n=0, out_u8=FAKE) == 0
    assert _apply(lib, n=0, batch=FAKE + 4 * U8_BYTES, out_u8=0) == 0
    assert _apply(lib, n=0, layout=5) == -1 and b"layout" in lib.hipac_last_error()
