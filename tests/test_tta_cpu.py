"""D4 test-time augmentation without a GPU: both entry points refuse every bad argument before touching the device and
name it in hipac_last_error()."""
import ctypes as C

import pytest

NHWC3, S2D16 = 1, 2
S2D16_BYTES = 112 * 115 * 16 * 2
NHWC3_BYTES = 224 * 224 * 3 * 2


def _forward_d4(lib, packed=1 << 20, num_classes=2, batch=2 << 20, layout=S2D16, n=4, count=None, feats=3 << 20,
                logits=4 << 20, ws=None, ws_bytes=None, chunk=0):
    ws = (1 << 30) if ws is None else ws                            # never dereferenced: validation fails first
    ws_bytes = lib.hipac_resnet18_workspace_bytes(n, chunk) if ws_bytes is None else ws_bytes
    v = lambda p: C.c_void_p(p) if p else None                      # noqa: E731
    return lib.hipac_resnet18_forward_d4(v(packed), num_classes, v(batch), layout, n, v(count), v(feats), v(logits), v(ws),
                                         ws_bytes, chunk, None)


def _view(lib, d_in=1 << 30, layout=S2D16, n=4, view=3, d_out=2 << 30, count=None, base=0):
    v = lambda p: C.c_void_p(p) if p else None                      # noqa: E731
    return lib.hipac_batch_d4_view(v(d_in), layout, n, view, v(d_out), v(count), base, None)


@pytest.mark.parametrize("kw,msg", [
    (dict(packed=0), b"null pointer"),
    (dict(batch=0), b"null pointer"),
    (dict(feats=0), b"null pointer"),
    (dict(ws=0), b"null pointer"),
    (dict(layout=0), b"unknown batch layout"),
    (dict(layout=3), b"unknown batch layout"),
    (dict(n=-1), b"negative n_patches"),
    (dict(num_classes=0), b"no classifier head"),
    (dict(ws_bytes=1024), b"workspace too small"),
    (dict(ws=(1 << 30) + 64), b"256-byte aligned"),
])
def test_forward_d4_refuses_bad_arguments(built_lib, kw, msg):
    assert _forward_d4(built_lib, **kw) == -1
    assert msg in built_lib.hipac_last_error()


def test_forward_d4_takes_the_plain_forwards_workspace(built_lib):
    """Same validation as hipac_resnet18_forward, including the workspace size: the view goes into the S2D16 scratch
    buffer the plain forward already has."""
    lib = built_lib
    need = lib.hipac_resnet18_workspace_bytes(300, 128)
    fake = C.c_void_p(1 << 30)
    for fn, extra in ((lib.hipac_resnet18_forward, ()), (lib.hipac_resnet18_forward_d4, (None,))):
        args = (fake, 2, fake) + (S2D16, 300) + extra + (fake, fake, fake, need - 1, 128, None)
        assert fn(*args) == -1 and b"workspace too small" in lib.hipac_last_error()
    assert _forward_d4(lib, n=0, packed=0, batch=0) == 0            # nothing to do, like the plain forward


@pytest.mark.parametrize("kw,msg", [
    (dict(d_in=0), b"null pointer"),
    (dict(d_out=0), b"null pointer"),
    (dict(layout=0), b"unknown batch layout"),
    (dict(layout=7), b"unknown batch layout"),
    (dict(view=-1), b"view must be in 0..7"),
    (dict(view=8), b"view must be in 0..7"),
    (dict(n=-2), b"negative n_patches"),
    (dict(base=-1), b"n_base must be non-negative"),
    (dict(d_out=1 << 30), b"overlaps"),                                             # in place
    (dict(d_out=(1 << 30) + 4 * S2D16_BYTES - 32), b"overlaps"),                    # last pixel of the input
    (dict(d_out=(1 << 30) - 4 * S2D16_BYTES + 32), b"overlaps"),                    # output ends inside the input
    (dict(layout=NHWC3, d_out=(1 << 30) + 4 * NHWC3_BYTES - 2), b"overlaps"),       # NHWC3 input is larger
])
def test_batch_d4_view_refuses_bad_arguments(built_lib, kw, msg):
    assert _view(built_lib, **kw) == -1
    assert msg in built_lib.hipac_last_error()


def test_batch_d4_view_empty_batch_is_a_no_op(built_lib):
    """An empty batch returns before any device call (two empty ranges do not overlap); bad arguments still fail."""
    lib = built_lib
    assert _view(lib, n=0) == 0
    assert _view(lib, n=0, d_out=1 << 30) == 0
    assert _view(lib, n=0, view=9) == -1 and b"view" in lib.hipac_last_error()
