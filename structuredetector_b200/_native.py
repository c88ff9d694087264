"""ctypes binding of ``libsdnet_decode.so`` (C ABI declared in ``include/sdnet_decode.h``).

There is deliberately no fallback: if the shared library is missing or does not export
the expected ABI, importing the decode ops raises.  Build it with
``python structuredetector_b200/build.py`` (or ``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes
from pathlib import Path

import os as _os

# SDNET_DECODE_LIB: load another build of the same library (kernel experiments, tools/xbuild.sh)
LIB_PATH = Path(_os.environ.get("SDNET_DECODE_LIB") or Path(__file__).resolve().parent / "csrc" / "libsdnet_decode.so").resolve()
ABI_VERSION = 10
DEST_PEER_STORES, DEST_MULTICAST = 0, 1  # SdnetDecodeParams.dest_mode

FLAG_PRE_ACTIVATED = 1
FLAG_NO_GROUPING = 2
FLAG_EXACT_SELECT = 4
FLAG_WARP_KERNEL = 8
FLAG_WORKSPACE_CLEAN = 16
DTYPE_F32 = 0
DTYPE_F16 = 1
DTYPE_BF16 = 2
MAX_TOPK = 1024
MAX_CHANNELS = 255
MAX_DEST = 16
MAX_GT = 1024  # SDNET_MAX_GT
MAX_THRESHOLDS = 256  # SDNET_MAX_THRESHOLDS
MAX_GATES = 64  # SDNET_MAX_GATES
SWEEP_OBJECTS = 1  # SdnetSweepParams.flags

EXPORTS = (
    "sdnet_abi_version",
    "sdnet_error_string",
    "sdnet_decode_workspace_bytes",
    "sdnet_decode_launch",
    "sdnet_decode_launch_timed",
    "sdnet_decode_peaks_path",
    "sdnet_decode_schedule",
    "sdnet_match_launch",
    "sdnet_gather_wait_launch",
    "sdnet_match_objects_launch",
    "sdnet_sweep_launch",
    "sdnet_activate_launch",
    "sdnet_suppress_launch",
    "sdnet_suppress_into_launch",
    "sdnet_decode_host_launch",
)


class SdnetTensor4(ctypes.Structure):
    _fields_ = [
        ("data", ctypes.c_void_p),
        ("stride_b", ctypes.c_int64),
        ("stride_c", ctypes.c_int64),
        ("stride_h", ctypes.c_int64),
        ("stride_w", ctypes.c_int64),
    ]


class SdnetDecodeParams(ctypes.Structure):
    _fields_ = [
        ("struct_size", ctypes.c_uint32),
        ("dtype", ctypes.c_int32),
        ("B", ctypes.c_int32),
        ("M", ctypes.c_int32),
        ("N", ctypes.c_int32),
        ("H", ctypes.c_int32),
        ("W", ctypes.c_int32),
        ("K", ctypes.c_int32),
        ("P", ctypes.c_int32),
        ("radius", ctypes.c_int32),
        ("flags", ctypes.c_uint32),
        ("conf_f32", ctypes.c_float),
        ("dist_abs_f32", ctypes.c_float),
        ("anchor_hm", SdnetTensor4),
        ("part_hm", SdnetTensor4),
        ("offsets", SdnetTensor4),
        ("embeddings", SdnetTensor4),
        ("anchor_out", ctypes.c_void_p),
        ("part_out", ctypes.c_void_p),
        ("anchor_inds", ctypes.c_void_p),
        ("part_inds", ctypes.c_void_p),
        ("part_emb", ctypes.c_void_p),
        ("assign", ctypes.c_void_p),
        ("counts", ctypes.c_void_p),
        ("diag", ctypes.c_void_p),
        ("workspace", ctypes.c_void_p),
        ("workspace_bytes", ctypes.c_size_t),
        ("n_dest", ctypes.c_int32),
        ("dest_mode", ctypes.c_int32),
        ("dest_delta", ctypes.c_int64 * MAX_DEST),
        ("done_flag", ctypes.c_void_p),
        ("done_value", ctypes.c_uint32),
        ("reserved1", ctypes.c_uint32),
    ]


class SdnetSchedule(ctypes.Structure):
    _fields_ = [("struct_size", ctypes.c_uint32)] + [(name, ctypes.c_int32) for name in (
        "path", "units", "tier1_units", "chunk_units", "chunk_groups", "groups_per_column", "panels", "strips",
        "rows_per_strip", "ctas", "warps_per_cta", "ctas_per_sm", "sms", "list_capacity")]


class SdnetMatchParams(ctypes.Structure):
    _fields_ = [
        ("struct_size", ctypes.c_uint32),
        ("B", ctypes.c_int32), ("M", ctypes.c_int32), ("N", ctypes.c_int32), ("K", ctypes.c_int32), ("P", ctypes.c_int32),
        ("max_gt_anchors", ctypes.c_int32), ("max_gt_parts", ctypes.c_int32),
        ("conf", ctypes.c_double), ("sx", ctypes.c_double), ("sy", ctypes.c_double),
        ("anchor_out", ctypes.c_void_p), ("part_out", ctypes.c_void_p), ("image_scale", ctypes.c_void_p),
        ("gt_anchors", ctypes.c_void_p), ("n_gt_anchors", ctypes.c_void_p),
        ("gt_parts", ctypes.c_void_p), ("n_gt_parts", ctypes.c_void_p),
        ("anchor_stats", ctypes.c_void_p), ("part_stats", ctypes.c_void_p),
        ("anchor_acc", ctypes.c_void_p), ("part_acc", ctypes.c_void_p),
    ]


class SdnetObjectMatchParams(ctypes.Structure):
    _fields_ = [
        ("struct_size", ctypes.c_uint32),
        ("B", ctypes.c_int32), ("M", ctypes.c_int32), ("N", ctypes.c_int32), ("K", ctypes.c_int32), ("P", ctypes.c_int32),
        ("max_gt_objects", ctypes.c_int32), ("max_gt_parts", ctypes.c_int32),
        ("conf", ctypes.c_double), ("sx", ctypes.c_double), ("sy", ctypes.c_double), ("csi_threshold", ctypes.c_double),
        ("anchor_out", ctypes.c_void_p), ("part_out", ctypes.c_void_p), ("assign", ctypes.c_void_p),
        ("image_scale", ctypes.c_void_p),
        ("gt_objects", ctypes.c_void_p), ("n_gt_objects", ctypes.c_void_p),
        ("gt_parts", ctypes.c_void_p), ("gt_part_owner", ctypes.c_void_p), ("n_gt_parts", ctypes.c_void_p),
        ("cls_group", ctypes.c_void_p),
        ("csi_stats", ctypes.c_void_p), ("csi_acc", ctypes.c_void_p),
        ("classif_stats", ctypes.c_void_p), ("classif_acc", ctypes.c_void_p), ("pred_parts", ctypes.c_void_p),
    ]


class SdnetSweepParams(ctypes.Structure):
    _fields_ = [
        ("struct_size", ctypes.c_uint32),
        ("B", ctypes.c_int32), ("M", ctypes.c_int32), ("N", ctypes.c_int32), ("K", ctypes.c_int32), ("P", ctypes.c_int32),
        ("T", ctypes.c_int32), ("max_gt_objects", ctypes.c_int32), ("max_gt_parts", ctypes.c_int32),
        ("flags", ctypes.c_uint32), ("dist_abs_f32", ctypes.c_float),
        ("sx", ctypes.c_double), ("sy", ctypes.c_double), ("csi_threshold", ctypes.c_double),
        ("conf", ctypes.c_void_p), ("conf_group", ctypes.c_void_p),
        ("anchor_out", ctypes.c_void_p), ("part_out", ctypes.c_void_p), ("image_scale", ctypes.c_void_p),
        ("gt_objects", ctypes.c_void_p), ("n_gt_objects", ctypes.c_void_p),
        ("gt_parts", ctypes.c_void_p), ("gt_part_owner", ctypes.c_void_p), ("n_gt_parts", ctypes.c_void_p),
        ("cls_group", ctypes.c_void_p),
        ("anchor_stats", ctypes.c_void_p), ("part_stats", ctypes.c_void_p),
        ("anchor_acc", ctypes.c_void_p), ("part_acc", ctypes.c_void_p),
        ("csi_stats", ctypes.c_void_p), ("csi_acc", ctypes.c_void_p),
        ("classif_stats", ctypes.c_void_p), ("classif_acc", ctypes.c_void_p), ("pred_parts", ctypes.c_void_p),
        ("assign_out", ctypes.c_void_p),
        ("G", ctypes.c_int32), ("dist_abs_grid", ctypes.c_void_p),
    ]


class NativeLibraryError(RuntimeError):
    pass


_lib = None


def load() -> ctypes.CDLL:
    """Load the decode library once; raise ``NativeLibraryError`` if it cannot be used."""
    global _lib
    if _lib is None:
        _lib = load_from(LIB_PATH)
    return _lib


def load_from(path) -> ctypes.CDLL:
    """dlopen one build of the library and declare its entry points (``load()`` for the product build;
    kernel experiments load several builds side by side, tools/sweep.py)."""
    path = Path(path)
    if not path.exists():
        raise NativeLibraryError(
            f"{path} is missing: build the CUDA extension first "
            "(python structuredetector_b200/build.py). There is no CPU fallback."
        )
    lib = ctypes.CDLL(str(path))
    missing = [name for name in EXPORTS if not hasattr(lib, name)]
    if missing:
        raise NativeLibraryError(f"{path} does not export {missing}")
    lib.sdnet_abi_version.restype = ctypes.c_int
    lib.sdnet_error_string.restype = ctypes.c_char_p
    lib.sdnet_error_string.argtypes = [ctypes.c_int]
    lib.sdnet_decode_workspace_bytes.restype = ctypes.c_int
    lib.sdnet_decode_workspace_bytes.argtypes = [ctypes.c_int] * 8 + [ctypes.POINTER(ctypes.c_size_t)]
    lib.sdnet_decode_launch.restype = ctypes.c_int
    lib.sdnet_decode_launch.argtypes = [ctypes.POINTER(SdnetDecodeParams), ctypes.c_void_p]
    lib.sdnet_gather_wait_launch.restype = ctypes.c_int
    lib.sdnet_gather_wait_launch.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_uint32, ctypes.c_void_p]
    lib.sdnet_match_launch.restype = ctypes.c_int
    lib.sdnet_match_launch.argtypes = [ctypes.POINTER(SdnetMatchParams), ctypes.c_void_p]
    lib.sdnet_match_objects_launch.restype = ctypes.c_int
    lib.sdnet_match_objects_launch.argtypes = [ctypes.POINTER(SdnetObjectMatchParams), ctypes.c_void_p]
    lib.sdnet_sweep_launch.restype = ctypes.c_int
    lib.sdnet_sweep_launch.argtypes = [ctypes.POINTER(SdnetSweepParams), ctypes.c_void_p]
    lib.sdnet_decode_peaks_path.restype = ctypes.c_int
    lib.sdnet_decode_peaks_path.argtypes = [ctypes.POINTER(SdnetDecodeParams)]
    lib.sdnet_decode_schedule.restype = ctypes.c_int
    lib.sdnet_decode_schedule.argtypes = [ctypes.POINTER(SdnetDecodeParams), ctypes.POINTER(SdnetSchedule)]
    lib.sdnet_decode_launch_timed.restype = ctypes.c_int
    lib.sdnet_decode_launch_timed.argtypes = [ctypes.POINTER(SdnetDecodeParams), ctypes.c_void_p,
                                              ctypes.POINTER(ctypes.c_float)]
    lib.sdnet_suppress_launch.restype = ctypes.c_int
    lib.sdnet_suppress_launch.argtypes = [ctypes.POINTER(SdnetTensor4)] + [ctypes.c_int] * 6 + [ctypes.c_void_p, ctypes.c_void_p]
    lib.sdnet_suppress_into_launch.restype = ctypes.c_int
    lib.sdnet_suppress_into_launch.argtypes = [ctypes.POINTER(SdnetTensor4)] + [ctypes.c_int] * 6 + [ctypes.POINTER(SdnetTensor4), ctypes.c_void_p]
    lib.sdnet_activate_launch.restype = ctypes.c_int
    lib.sdnet_activate_launch.argtypes = [ctypes.POINTER(SdnetTensor4), ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                          ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    lib.sdnet_decode_host_launch.restype = ctypes.c_int
    lib.sdnet_decode_host_launch.argtypes = [ctypes.POINTER(SdnetDecodeParams), ctypes.c_void_p, ctypes.c_size_t,
                                             ctypes.c_void_p]
    if lib.sdnet_abi_version() != ABI_VERSION:
        raise NativeLibraryError(f"ABI mismatch: library {lib.sdnet_abi_version()} != binding {ABI_VERSION}")
    return lib


def error_string(code: int) -> str:
    return load().sdnet_error_string(int(code)).decode()


def check(code: int, what: str):
    """Map the C ABI's return convention onto Python exceptions."""
    if code == 0:
        return
    msg = f"{what}: {error_string(code)} (code {code})"
    if code == -2:
        # mirrors torch.topk's failure for k > H*W in the reference (SURVEY 8b "Error conventions")
        raise RuntimeError(msg)
    if code < 0:
        raise ValueError(msg)
    raise RuntimeError(msg)


def workspace_bytes(B, M, N, H, W, K, P, dtype=DTYPE_F32, lib=None) -> int:
    out = ctypes.c_size_t(0)
    check((lib or load()).sdnet_decode_workspace_bytes(B, M, N, H, W, K, P, dtype, ctypes.byref(out)), "sdnet_decode_workspace_bytes")
    return int(out.value)
