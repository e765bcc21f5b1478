"""
ctypes binding of the C ABI declared in `include/yawb.h` (libyawb.so, built
in-tree by `csrc/build.py`).  No torch types cross this boundary.

There is no CPU fallback: if the shared library is missing, or no CUDA device
is present, the engine raises instead of computing anything on the host.
"""

from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int32, c_int64, c_uint32, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
# YAWB_LIB: development override (kernel variants built side by side)
LIB_PATH = os.environ.get("YAWB_LIB") or os.path.join(_HERE, "csrc", "libyawb.so")

FLAG_EXACT_BRUTEFORCE = 1
FLAG_OUT_DEVICE = 2
FLAG_SECOND_LABELS = 4
LABELS_MIN_VERSION = 101  # first library version that knows FLAG_SECOND_LABELS
BINNED_LABELS_MIN_VERSION = 102  # first library version with yawb_catalog_set_labels
PARTIAL_MIN_VERSION = 103  # first library version with partial uploads and second-role row masks
# yawb_catalog_footprint flags (library version >= 104)
FOOT_WEIGHTED = 1
FOOT_BINNED = 2
FOOT_U8 = 4
FOOT_Z = 8
FOOT_LABELLED = 16
FOOT_MASK = 32
FOOT_FIRST = 64
FOOT_SECOND = 128
FOOT_NO_UPLOAD = 256
ROLE_FIRST = 1
ROLE_SECOND = 2

# every symbol include/yawb.h declares (checked by tests/test_cabi.py)
EXPORTS = (
    "yawb_last_error", "yawb_create", "yawb_destroy", "yawb_upload_catalog", "yawb_free_catalog",
    "yawb_build_index", "yawb_drop_index", "yawb_catalog_info", "yawb_sum_weights", "yawb_count",
    "yawb_host_alloc", "yawb_host_free", "yawb_sync", "yawb_version", "yawb_device_sms",
    "yawb_timer_start", "yawb_timer_stop", "yawb_assign_patches", "yawb_upload_catalog_u8", "yawb_count2",
    "yawb_upload_catalog_z", "yawb_patch_metadata", "yawb_jackknife", "yawb_count4", "yawb_kmeans",
    "yawb_catalog_set_labels", "yawb_upload_catalog_patches", "yawb_catalog_set_second_rows",
    "yawb_catalog_footprint", "yawb_count_footprint", "yawb_memory_stats", "yawb_memory_reset_peak",
    "yawb_memory_parked",
    "yawb_memory_release",
)


class YawbStats(ctypes.Structure):
    _fields_ = [
        ("kernel_ms", c_double),
        ("index_ms", c_double),
        ("pair_tests", c_uint64),
        ("pair_tests_naive", c_uint64),
        ("rechecks", c_uint64),
        ("work_items", c_uint64),
        ("launches", c_uint64),
        ("plan_ms", c_double),
    ]

    def as_dict(self) -> dict:
        return {name: getattr(self, name) for name, _ in self._fields_}


class YawbError(RuntimeError):
    pass


_lib = None


def load(build_if_missing: bool = False) -> ctypes.CDLL:
    """Load libyawb.so; raises `YawbError` if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH) and build_if_missing:
        from .csrc import build as _build

        _build.build()
    if not os.path.exists(LIB_PATH):
        raise YawbError(
            f"{LIB_PATH} not found: build it with `python yet_another_wizz_b200/csrc/build.py` "
            "(the engine has no CPU fallback)"
        )
    lib = ctypes.CDLL(LIB_PATH)
    lib.yawb_last_error.restype = c_char_p
    lib.yawb_last_error.argtypes = []
    lib.yawb_version.restype = c_int
    lib.yawb_create.argtypes = [c_int, POINTER(c_void_p)]
    lib.yawb_destroy.argtypes = [c_void_p]
    lib.yawb_device_sms.argtypes = [c_void_p]
    lib.yawb_sync.argtypes = [c_void_p]
    lib.yawb_timer_start.argtypes = [c_void_p]
    lib.yawb_timer_stop.argtypes = [c_void_p, POINTER(c_double)]
    lib.yawb_host_alloc.argtypes = [POINTER(c_void_p), c_uint64]
    lib.yawb_host_free.argtypes = [c_void_p]
    lib.yawb_upload_catalog.argtypes = [
        c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, POINTER(c_void_p),
    ]
    lib.yawb_upload_catalog_u8.argtypes = lib.yawb_upload_catalog.argtypes
    lib.yawb_upload_catalog_z.argtypes = [
        c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, POINTER(c_void_p),
    ]
    lib.yawb_upload_catalog_patches.argtypes = [
        c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_void_p,
        POINTER(c_void_p),
    ]
    lib.yawb_catalog_set_second_rows.argtypes = [c_void_p, c_void_p]
    lib.yawb_patch_metadata.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p]
    lib.yawb_jackknife.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]
    lib.yawb_free_catalog.argtypes = [c_void_p]
    lib.yawb_build_index.argtypes = [c_void_p, c_int, POINTER(c_double)]
    lib.yawb_drop_index.argtypes = [c_void_p]
    lib.yawb_catalog_info.argtypes = [c_void_p, POINTER(c_int64), POINTER(c_int64)]
    lib.yawb_sum_weights.argtypes = [c_void_p, c_void_p]
    lib.yawb_assign_patches.argtypes = [c_void_p, c_void_p, c_int64, c_void_p, c_int, c_void_p]
    lib.yawb_kmeans.argtypes = [
        c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, POINTER(c_int), POINTER(c_int),
    ]
    lib.yawb_count.argtypes = [
        c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_uint32,
        c_void_p, c_void_p, POINTER(YawbStats),
    ]
    lib.yawb_count2.argtypes = [
        c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_uint32,
        c_void_p, c_void_p, c_void_p, c_void_p, POINTER(YawbStats),
    ]
    lib.yawb_count4.argtypes = [
        c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_uint32,
        POINTER(c_void_p), POINTER(c_void_p), POINTER(YawbStats),
    ]
    lib.yawb_catalog_footprint.argtypes = [c_int64, c_int, c_int, c_uint32, POINTER(c_int64)]
    lib.yawb_count_footprint.argtypes = [c_int, c_int64, c_int, c_int, c_int, c_int, c_int, POINTER(c_int64)]
    lib.yawb_memory_stats.argtypes = [c_void_p, POINTER(c_int64), POINTER(c_int64), POINTER(c_int64)]
    lib.yawb_memory_parked.argtypes = [c_void_p, POINTER(c_int64)]
    lib.yawb_memory_reset_peak.argtypes = [c_void_p]
    lib.yawb_memory_release.argtypes = [c_void_p]
    if hasattr(lib, "yawb_catalog_set_labels"):  # older libraries lack it: Engine.upload_catalog(n_labels=) refuses
        lib.yawb_catalog_set_labels.argtypes = [c_void_p, c_int]
        lib.yawb_catalog_set_labels.restype = c_int
    for name in EXPORTS:
        if name not in ("yawb_last_error", "yawb_catalog_set_labels"):
            getattr(lib, name).restype = c_int
    lib.yawb_last_error.restype = c_char_p
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().yawb_last_error()
        raise YawbError(msg.decode("utf-8", "replace") if msg else f"yawb error {rc}")
