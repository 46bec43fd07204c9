"""ctypes binding of libhipac_b200.so (the C ABI in include/hipac_b200.h).

The shared library is built in-tree by ``build()`` (nvcc, sm_100a only) and loaded lazily.
There is no CPU or PyTorch fallback: if the library is missing, ``lib()`` raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(_HERE, "libhipac_b200.so")
# the same library with -DHIPAC_DEBUG_BOUNDS (device-side bounds assertions in the stage-1 kernels); loaded instead of
# LIB_PATH when HIPAC_DEBUG_BOUNDS=1 is in the environment (tests/test_debug_bounds_gpu.py runs it in a subprocess)
DBG_LIB_PATH = os.path.join(_HERE, "libhipac_b200_dbg.so")
SOURCES = ["capi.cu", "tile_scan.cu", "resnet18.cu", "exchange.cu", "polygon.cu", "mil.cu", "debug_umma.cu", "tissue.cu", "cascade.cu", "stain.cu"]
HEADER = os.path.join(os.path.dirname(_HERE), "include", "hipac_b200.h")

LAYOUT_NHWC3_BF16 = 1
LAYOUT_S2D16_BF16 = 2
SCAN_AUTO, SCAN_DIRECT, SCAN_FUSED = 0, 1, 2
SCAN_KEEP_ALL = 0x100
SCAN_NO_STREAM = 0x200
RESNET18_NUM_CONVS = 20
STAIN_BLOCK_DOUBLES = 16
STAIN_PARAMS_DOUBLES = 267

_lock = threading.Lock()
_lib = None


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _source_hash() -> str:
    """sha256 over the CUDA sources and the public header: what a built library is a function of."""
    import hashlib
    h = hashlib.sha256()
    for d in sorted(os.path.join(_CSRC, f) for f in os.listdir(_CSRC)) + [HEADER]:
        h.update(os.path.basename(d).encode())
        h.update(open(d, "rb").read())
    return h.hexdigest()


def _stale(path: str = LIB_PATH) -> bool:
    """A library is fresh iff the source hash recorded beside it equals the current one (file times do not survive the
    copy to the GPU box, so they are not consulted)."""
    try:
        return open(path + ".srchash").read().strip() != _source_hash() or not os.path.exists(path)
    except OSError:
        return True


def build(force: bool = False, verbose: bool = False, debug_bounds: bool = False) -> str:
    """Compile every CUDA source for sm_100a into ``libhipac_b200.so`` (in-tree); ``debug_bounds`` builds the
    ``-DHIPAC_DEBUG_BOUNDS`` variant ``libhipac_b200_dbg.so`` instead."""
    out_path = DBG_LIB_PATH if debug_bounds else LIB_PATH
    if not force and not _stale(out_path):
        return out_path
    # several ranks may call build() at once (torchrun): one compiles, the others wait and find a fresh library
    import fcntl
    with open(os.path.join(_HERE, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not _stale(out_path):
                return out_path
            return _build_locked(out_path, verbose, debug_bounds)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(out_path: str, verbose: bool, debug_bounds: bool) -> str:
    src_hash = _source_hash()
    objs = []
    build_dir = os.path.join(_HERE, "build", "dbg" if debug_bounds else "")
    os.makedirs(build_dir, exist_ok=True)
    flags = ["-std=c++17", "-O3", "-lineinfo", "-gencode", "arch=compute_100a,code=sm_100a",
             "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"] + (["-DHIPAC_DEBUG_BOUNDS"] if debug_bounds else [])
    procs = []
    for src in SOURCES:
        obj = os.path.join(build_dir, src.replace(".cu", ".o"))
        cmd = [_nvcc(), *flags, "-c", os.path.join(_CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd))
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, pr in procs:
        out, _ = pr.communicate()
        if verbose and out:
            print(out)
        if pr.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{out}")
    cmd = [_nvcc(), "-shared", "-o", out_path + ".tmp", *objs, "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    os.replace(out_path + ".tmp", out_path)
    with open(out_path + ".srchash", "w") as f:
        f.write(src_hash + "\n")
    return out_path


def _declare(l):
    vp, i32, i64, sz = C.c_void_p, C.c_int, C.c_int64, C.c_size_t
    l.hipac_last_error.restype = C.c_char_p
    l.hipac_last_error.argtypes = []
    l.hipac_abi_version.restype = i32
    l.hipac_abi_version.argtypes = []
    l.hipac_launch_count.restype = C.c_longlong
    l.hipac_launch_count.argtypes = [i32]
    l.hipac_tile_scan_workspace_bytes.restype = sz
    l.hipac_tile_scan_workspace_bytes.argtypes = [i32] * 7
    l.hipac_tile_scan.restype = i32
    l.hipac_tile_scan.argtypes = [vp, i32, i32, i64, vp, i64, i32, i32, i32, i32, vp, vp, vp, vp, i32, vp, i32,
                                  vp, sz, i32, vp]
    l.hipac_tile_scan_tissue_workspace_bytes.restype = sz
    l.hipac_tile_scan_tissue_workspace_bytes.argtypes = [i32] * 8
    l.hipac_tile_scan_tissue.restype = i32
    l.hipac_tile_scan_tissue.argtypes = [vp, i32, i32, i64, vp, i64, i32, i32, i32, i32, vp, vp, vp, vp, i32, vp, i32,
                                         vp, sz, i32, vp, i32, i32, i64, i32, i32, vp]
    l.hipac_tile_scan_roi_workspace_bytes.restype = sz
    l.hipac_tile_scan_roi_workspace_bytes.argtypes = [i32] * 8
    l.hipac_tile_scan_roi.restype = i32
    l.hipac_tile_scan_roi.argtypes = [vp, i32, i32, i64, vp, i64, i32, i32, i32, i32, vp, vp, vp, vp, i32, vp, i32,
                                      vp, sz, i32, vp, i32, i32, i64, i32, i32, vp, i32, i32, i32, i32, i32, i64, vp]
    l.hipac_roi_grid_bytes.restype = sz
    l.hipac_roi_grid_bytes.argtypes = [i32, i32]
    l.hipac_roi_grid.restype = i32
    l.hipac_roi_grid.argtypes = [vp, vp, vp, i32, C.c_float, i32, i32, i32, i32, vp, vp]
    l.hipac_tissue_workspace_bytes.restype = sz
    l.hipac_tissue_workspace_bytes.argtypes = [i32, i32]
    l.hipac_tissue_segment.restype = i32
    l.hipac_tissue_segment.argtypes = [vp, i32, i32, i64, i32, i32, vp, i64, vp, vp, i64, vp, sz, vp]
    l.hipac_stain_workspace_bytes.restype = sz
    l.hipac_stain_workspace_bytes.argtypes = [i32, i32]
    l.hipac_stain_estimate.restype = i32
    l.hipac_stain_estimate.argtypes = [vp, i32, i32, i64, i32, C.c_double, C.c_double, vp, vp, sz, vp]
    l.hipac_stain_normalizer.restype = i32
    l.hipac_stain_normalizer.argtypes = [vp, vp, i32, vp, vp]
    l.hipac_stain_apply.restype = i32
    l.hipac_stain_apply.argtypes = [vp, i32, vp, i32, vp, vp, vp, i32, vp]
    l.hipac_tile_scan_set_count_buffer.restype = i32
    l.hipac_tile_scan_set_count_buffer.argtypes = [vp]
    l.hipac_tile_scan_wait_count.restype = i32
    l.hipac_tile_scan_wait_count.argtypes = []
    l.hipac_upload_rows.restype = i32
    l.hipac_upload_rows.argtypes = [vp, i64, vp, i64, i64, i64, vp]
    l.hipac_pillow_coeffs.restype = i32
    l.hipac_pillow_coeffs.argtypes = [i32, vp, vp, vp]
    l.hipac_normalize_lut_bf16.restype = i32
    l.hipac_normalize_lut_bf16.argtypes = [vp]
    l.hipac_resnet18_packed_bytes.restype = sz
    l.hipac_resnet18_packed_bytes.argtypes = [i32]
    l.hipac_resnet18_pack.restype = i32
    l.hipac_resnet18_pack.argtypes = [C.POINTER(vp), i32, i32, C.c_float, vp, sz]
    l.hipac_resnet18_workspace_bytes.restype = sz
    l.hipac_resnet18_workspace_bytes.argtypes = [i32, i32]
    l.hipac_resnet18_forward.restype = i32
    l.hipac_resnet18_forward.argtypes = [vp, i32, vp, i32, i32, vp, vp, vp, sz, i32, vp]
    l.hipac_resnet18_forward_dcount.restype = i32
    l.hipac_resnet18_forward_dcount.argtypes = [vp, i32, vp, i32, i32, vp, vp, vp, vp, sz, i32, vp]
    l.hipac_resnet18_forward_d4.restype = i32
    l.hipac_resnet18_forward_d4.argtypes = [vp, i32, vp, i32, i32, vp, vp, vp, vp, sz, i32, vp]
    l.hipac_batch_d4_view.restype = i32
    l.hipac_batch_d4_view.argtypes = [vp, i32, i32, i32, vp, vp, i32, vp]
    l.hipac_resnet18_conv_ds_fused.restype = i32
    l.hipac_resnet18_conv_ds_fused.argtypes = [vp, i32, i32, vp, vp, vp, i32, vp, i32, vp, i32]
    l.hipac_resnet18_stem.restype = i32
    l.hipac_resnet18_stem.argtypes = [vp, i32, vp, vp, i32, vp, i32, vp, i32]
    l.hipac_exchange_row_bytes.restype = sz
    l.hipac_exchange_row_bytes.argtypes = [i32, i32]
    l.hipac_exchange_segment_bytes.restype = sz
    l.hipac_exchange_segment_bytes.argtypes = [i32, i32, i32]
    l.hipac_exchange_workspace_bytes.restype = sz
    l.hipac_exchange_workspace_bytes.argtypes = [i32, i32]
    l.hipac_exchange_pack.restype = i32
    l.hipac_exchange_pack.argtypes = [vp, vp, vp, vp, i32, i32, vp, i32, i32, vp, vp]
    l.hipac_exchange_merge.restype = i32
    l.hipac_exchange_merge.argtypes = [vp, i32, i32, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, i32, vp, sz, vp]
    l.hipac_polygon_workspace_bytes.restype = sz
    l.hipac_polygon_workspace_bytes.argtypes = [i32]
    l.hipac_polygon_fill.restype = i32
    l.hipac_polygon_fill.argtypes = [vp, vp, i32, vp, vp, i32, i32, i64, i32, i32, i32, vp, sz, vp]
    l.hipac_polygon_overflowed.restype = i32
    l.hipac_polygon_overflowed.argtypes = [vp, vp]
    l.hipac_mil_packed_floats.restype = sz
    l.hipac_mil_packed_floats.argtypes = [i32]
    l.hipac_mil_pack.restype = i32
    l.hipac_mil_pack.argtypes = [vp] * 8 + [i32, vp]
    l.hipac_mil_workspace_bytes.restype = sz
    l.hipac_mil_workspace_bytes.argtypes = [i32]
    l.hipac_mil_forward.restype = i32
    l.hipac_mil_forward.argtypes = [vp, i32, vp, vp, i32, i32, vp, vp, vp, vp, sz, vp]
    l.hipac_debug_umma_shift.restype = i32
    l.hipac_debug_umma_shift.argtypes = [vp, vp, vp, i32, i32, vp]
    l.hipac_profile_enable.restype = i32
    l.hipac_profile_enable.argtypes = [i32]
    l.hipac_profile_report.restype = C.c_longlong
    l.hipac_profile_report.argtypes = [C.c_char_p, sz]
    l.hipac_resnet18_conv_layer.restype = i32
    l.hipac_resnet18_conv_layer.argtypes = [vp, i32, i32, vp, vp, vp, i32, i32, vp, i32, vp, i32]


EXPORTS = [
    "hipac_last_error", "hipac_abi_version", "hipac_launch_count", "hipac_tile_scan_workspace_bytes",
    "hipac_tile_scan", "hipac_upload_rows", "hipac_tile_scan_set_count_buffer", "hipac_tile_scan_wait_count", "hipac_pillow_coeffs", "hipac_normalize_lut_bf16", "hipac_resnet18_packed_bytes",
    "hipac_resnet18_pack", "hipac_resnet18_workspace_bytes", "hipac_resnet18_forward", "hipac_resnet18_forward_dcount",
    "hipac_resnet18_conv_layer", "hipac_exchange_row_bytes", "hipac_exchange_segment_bytes", "hipac_exchange_workspace_bytes",
    "hipac_exchange_pack", "hipac_exchange_merge", "hipac_polygon_workspace_bytes", "hipac_polygon_fill", "hipac_polygon_overflowed", "hipac_mil_packed_floats", "hipac_mil_pack", "hipac_mil_workspace_bytes", "hipac_mil_forward",
    "hipac_profile_enable", "hipac_profile_report", "hipac_debug_umma_shift", "hipac_resnet18_stem", "hipac_resnet18_conv_ds_fused",
    "hipac_tile_scan_tissue_workspace_bytes", "hipac_tile_scan_tissue", "hipac_tissue_workspace_bytes", "hipac_tissue_segment",
    "hipac_roi_grid_bytes", "hipac_roi_grid", "hipac_tile_scan_roi_workspace_bytes", "hipac_tile_scan_roi",
    "hipac_resnet18_forward_d4", "hipac_batch_d4_view",
    "hipac_stain_workspace_bytes", "hipac_stain_estimate", "hipac_stain_normalizer", "hipac_stain_apply",
]


def lib():
    """The loaded shared library; raises if it has not been built (no fallback path exists)."""
    global _lib
    with _lock:
        if _lib is None:
            path = DBG_LIB_PATH if os.environ.get("HIPAC_DEBUG_BOUNDS") == "1" else LIB_PATH
            if not os.path.exists(path):
                raise RuntimeError(
                    f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                    "(the HiPAC B200 path has no CPU/PyTorch fallback)")
            if _stale(path):
                raise RuntimeError(f"{path} was built from different sources than csrc/ now holds: run "
                                   "`python -c 'import __graft_entry__ as g; g.build()'`")
            l = C.CDLL(path)
            _declare(l)
            _lib = l
    return _lib


def check(rc: int, what: str):
    if rc != 0:
        raise RuntimeError(f"{what} failed ({rc}): {lib().hipac_last_error().decode()}")


_profiling = threading.local()


def profile(enable: bool):
    """Switch the library's per-kernel CUDA-event profiler on or off (calling thread)."""
    lib().hipac_profile_enable(int(enable))
    _profiling.on = bool(enable)


def profiling() -> bool:
    return bool(getattr(_profiling, "on", False))


def profile_report() -> dict:
    """``{kernel: {"launches": n, "ms": total_ms, "work": bytes_or_flops}}`` since the last report."""
    l = lib()
    buf = C.create_string_buffer(1 << 16)
    l.hipac_profile_report(buf, len(buf))
    out = {}
    for line in buf.value.decode().splitlines():
        name, n, ms, work = line.split()
        out[name] = {"launches": int(n), "ms": float(ms), "work": float(work)}
    return out
