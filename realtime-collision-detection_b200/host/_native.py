"""ctypes binding of librcd_b200.so (include/rcd.h).  Fails loudly: there is no CPU fallback.

The library is built in-tree by ``realtime-collision-detection_b200/build.py`` (nvcc, sm_100a).
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import numpy as np

_PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.environ.get("RCD_B200_LIB") or os.path.join(_PKG, "librcd_b200.so")  # override: kernel-tuning experiments only

RCD_OK, RCD_EINVAL, RCD_ENODEVICE, RCD_ENOMEM, RCD_ECUDA, RCD_ECAPACITY, RCD_ESTATE = 0, -1, -2, -3, -4, -5, -6
MODE_DETECT, MODE_PREDICT, MODE_COMPUTE_NODE = 0, 1, 2
STEP_APPEND = 0x100
STEP_WITH_DETECT = 0x200
SRC_HOST, SRC_DEVICE = 0, 1
PAT_STATIONARY, PAT_CONSTANT_VELOCITY, PAT_ACCELERATING, PAT_NO_HISTORY = 0, 1, 2, 3
FLAG_PROFILE = 1
FLAG_COUNT_PREDICT_CANDIDATES = 2
FLAG_GRAPH = 4
NUM_STAGES = 10
STAGE_NAMES = ("upload", "keys", "sort", "reorder", "pairs", "narrow", "exact", "download", "total", "qorder")
HALO_RECORD_WORDS = 13

# every symbol include/rcd.h declares (tests/test_abi.py checks the export table against this
# list and against the header itself)
SYMBOLS = (
    "rcd_version", "rcd_last_error", "rcd_create", "rcd_destroy", "rcd_upload", "rcd_set_patterns",
    "rcd_set_owned", "rcd_set_queries", "rcd_step", "rcd_build_index", "rcd_set_compute_node_params", "rcd_truncate", "rcd_invalidate", "rcd_counts", "rcd_download", "rcd_download_unsorted",
    "rcd_download_candidate_counts", "rcd_query_radius", "rcd_classify_patterns", "rcd_halo_pack",
    "rcd_halo_pack_async", "rcd_halo_append", "rcd_history_configure", "rcd_history_append", "rcd_history_reset", "rcd_history_move",
    "rcd_history_classify", "rcd_stage_ms", "rcd_get_stream", "rcd_launch_count", "rcd_pair_tests", "rcd_sync",
    "rcd_ingest_create", "rcd_ingest_destroy", "rcd_ingest_last_error", "rcd_ingest_decode_json",
    "rcd_ingest_counts", "rcd_ingest_set_limit", "rcd_ingest_rejected", "rcd_ingest_id_name", "rcd_ingest_type_name", "rcd_ingest_lookup", "rcd_apply_records",
    "rcd_alerts_configure", "rcd_alerts_update", "rcd_alerts_update_pairs", "rcd_alerts_expire",
    "rcd_alerts_acknowledge", "rcd_alerts_download", "rcd_download_begin", "rcd_download_finish", "rcd_graph_replays", "rcd_pair_exact", "rcd_risk_assessment", "rcd_download_begin_compact", "rcd_summary_begin", "rcd_summary_finish",
    "rcd_download_risk_counts", "rcd_retire", "rcd_retire_stale", "rcd_ingest_release", "rcd_reserve",
    "rcd_alerts_reserve",
)


class RcdConfig(ctypes.Structure):
    _fields_ = [("device", ctypes.c_int32), ("flags", ctypes.c_uint32), ("max_objects", ctypes.c_uint64),
                ("max_pairs", ctypes.c_uint64), ("world_min", ctypes.c_float * 3),
                ("world_max", ctypes.c_float * 3)]


class RcdCounts(ctypes.Structure):
    _fields_ = [("n_objects", ctypes.c_uint64), ("n_owned", ctypes.c_uint64), ("n_candidates", ctypes.c_uint64),
                ("n_potential", ctypes.c_uint64), ("n_pairs", ctypes.c_uint64), ("n_high_risk", ctypes.c_uint64),
                ("n_written", ctypes.c_uint64), ("n_alerts", ctypes.c_uint64 * 4), ("n_exact", ctypes.c_uint64),
                ("n_fallback", ctypes.c_uint64)]


# numpy mirror of rcd_pair (48 bytes)
PAIR_DTYPE = np.dtype([("i", "<u4"), ("j", "<u4"), ("ttc", "<f4"), ("distance", "<f4"), ("rel_speed", "<f4"),
                       ("risk", "<f4"), ("cx", "<f4"), ("cy", "<f4"), ("cz", "<f4"), ("t_closest", "<f4"),
                       ("d_closest", "<f4"), ("priority", "i1"), ("offset", "u1"), ("predicted", "u1"),
                       ("reserved", "u1")])
assert PAIR_DTYPE.itemsize == 48

# numpy mirror of rcd_pair_compact (32 bytes)
PAIR_COMPACT_DTYPE = np.dtype([("i", "<u4"), ("j", "<u4"), ("ttc", "<f4"), ("distance", "<f4"), ("rel_speed", "<f4"),
                               ("risk", "<f4"), ("t_closest", "<f4"), ("priority", "i1"), ("offset", "u1"),
                               ("predicted", "u1"), ("reserved", "u1")])
assert PAIR_COMPACT_DTYPE.itemsize == 32

# numpy mirrors of rcd_object (48 bytes) and rcd_pair_exact_result (72 bytes)
OBJECT_DTYPE = np.dtype([(k, "<f4") for k in ("px", "py", "pz", "vx", "vy", "vz", "ax", "ay", "az", "size", "heading")] +
                        [("type", "<u4")])
assert OBJECT_DTYPE.itemsize == 48
PAIR_EXACT_DTYPE = np.dtype([("hit", "<i4"), ("step", "<i4")] + [(k, "<f8") for k in (
    "collision_time", "distance", "safe_distance", "relative_speed", "cx", "cy", "cz", "risk")])
assert PAIR_EXACT_DTYPE.itemsize == 72

# numpy mirror of rcd_alert_event (40 bytes)
ALERT_REFRESHED, ALERT_CREATED, ALERT_PRIORITY_CHANGED, ALERT_EXPIRED = 0, 1, 2, 3
ALERT_EVENT_DTYPE = np.dtype([("i", "<u4"), ("j", "<u4"), ("alert_id", "<u4"), ("risk", "<f4"), ("ttc", "<f4"),
                              ("distance", "<f4"), ("priority", "i1"), ("old_priority", "i1"), ("kind", "u1"),
                              ("acknowledged", "u1"), ("reserved", "<u4"), ("timestamp", "<f8")])
assert ALERT_EVENT_DTYPE.itemsize == 40


class RcdAlertStats(ctypes.Structure):
    _fields_ = [(k, ctypes.c_uint64) for k in ("n_events", "n_created", "n_changed", "n_refreshed", "n_expired",
                                               "n_live", "n_dropped")]


# numpy mirror of rcd_record (72 bytes): one decoded vehicle message
RECORD_DTYPE = np.dtype([("x", "<f8"), ("y", "<f8"), ("z", "<f8"), ("timestamp", "<f8"), ("vx", "<f4"), ("vy", "<f4"),
                         ("vz", "<f4"), ("ax", "<f4"), ("ay", "<f4"), ("az", "<f4"), ("size", "<f4"),
                         ("heading", "<f4"), ("slot", "<u4"), ("type", "u1"), ("seq", "u1"), ("reserved", "<u2")])
assert RECORD_DTYPE.itemsize == 72


class NativeError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"librcd_b200 error {code}: {message}")
        self.code = code


_lib: Optional[ctypes.CDLL] = None


def load() -> ctypes.CDLL:
    """Load the CUDA library; raise if it was not built (no fallback of any kind)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python realtime-collision-detection_b200/build.py` "
            "(nvcc, sm_100a).  This package has no CPU or PyTorch fallback.")
    L = ctypes.CDLL(LIB_PATH)
    vp, u64, u32, i32, f32 = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int32, ctypes.c_float
    L.rcd_version.restype = ctypes.c_int
    L.rcd_version.argtypes = []
    L.rcd_last_error.restype = ctypes.c_char_p
    L.rcd_last_error.argtypes = [vp]
    L.rcd_create.argtypes = [ctypes.POINTER(RcdConfig), ctypes.POINTER(vp)]
    L.rcd_destroy.argtypes = [vp]
    L.rcd_upload.argtypes = [vp, u64] + [vp] * 13 + [i32]
    L.rcd_set_patterns.argtypes = [vp, u64, vp, i32]
    L.rcd_set_owned.argtypes = [vp, u64]
    if hasattr(L, "rcd_set_queries"):
        L.rcd_set_queries.argtypes = [vp, u64, vp, i32]
    L.rcd_step.argtypes = [vp, i32, f32, f32]
    L.rcd_build_index.argtypes = [vp, f32]
    L.rcd_set_compute_node_params.argtypes = [vp, f32, f32]
    L.rcd_truncate.argtypes = [vp, u64]
    L.rcd_invalidate.argtypes = [vp]
    L.rcd_counts.argtypes = [vp, ctypes.POINTER(RcdCounts)]
    L.rcd_download.argtypes = [vp, vp, u64, ctypes.POINTER(u64)]
    L.rcd_download_unsorted.argtypes = [vp, vp, u64, ctypes.POINTER(u64)]
    L.rcd_download_candidate_counts.argtypes = [vp, vp, u64]
    if hasattr(L, "rcd_download_begin"):
        L.rcd_download_begin.argtypes = [vp, vp, u64]
        L.rcd_download_finish.argtypes = [vp, ctypes.POINTER(RcdCounts), ctypes.POINTER(u64)]
    L.rcd_query_radius.argtypes = [vp, u64, vp, vp, vp, f32, vp, vp, u64]
    L.rcd_classify_patterns.argtypes = [vp, u64, u32, vp, vp, vp]
    L.rcd_halo_pack.argtypes = [vp, i32, i32, vp, vp, f32, vp, u64, vp]
    L.rcd_halo_append.argtypes = [vp, vp, u64]
    if hasattr(L, "rcd_halo_pack_async"):
        L.rcd_halo_pack_async.argtypes = [vp, i32, i32, vp, vp, f32, vp, vp, vp]
    L.rcd_history_configure.argtypes = [vp, u32]
    L.rcd_history_append.argtypes = [vp, u64, vp, vp, vp, vp, vp]
    L.rcd_history_reset.argtypes = [vp, u64, vp]
    L.rcd_history_move.argtypes = [vp, u32, u32]
    L.rcd_history_classify.argtypes = [vp, vp]
    L.rcd_stage_ms.argtypes = [vp, i32, vp]
    L.rcd_get_stream.argtypes = [vp, ctypes.POINTER(vp)]
    L.rcd_launch_count.argtypes = [vp, ctypes.POINTER(u64)]
    L.rcd_pair_tests.argtypes = [vp, ctypes.POINTER(u64)]
    if hasattr(L, "rcd_graph_replays"):
        L.rcd_graph_replays.argtypes = [vp, ctypes.POINTER(u64)]
    L.rcd_sync.argtypes = [vp]
    if hasattr(L, "rcd_summary_begin"):
        L.rcd_download_begin_compact.argtypes = [vp, vp, u64]
        L.rcd_summary_begin.argtypes = [vp, ctypes.c_double, i32]
        L.rcd_summary_finish.argtypes = [vp, vp, u64, ctypes.POINTER(u64), vp, vp, u64, vp]
        L.rcd_download_risk_counts.argtypes = [vp, vp, u64]
    if hasattr(L, "rcd_pair_exact"):
        L.rcd_pair_exact.argtypes = [vp, u64, vp, vp, ctypes.c_double, ctypes.c_double, vp]
        L.rcd_risk_assessment.argtypes = [vp, u64, vp, vp]
    if not hasattr(L, "rcd_ingest_create") and os.environ.get("RCD_B200_LIB"):
        _lib = L
        return L
    L.rcd_ingest_create.argtypes = [ctypes.POINTER(vp)]
    L.rcd_ingest_destroy.argtypes = [vp]
    L.rcd_ingest_last_error.restype = ctypes.c_char_p
    L.rcd_ingest_last_error.argtypes = [vp]
    L.rcd_ingest_decode_json.argtypes = [vp, vp, u64, i32, vp, u64, ctypes.POINTER(u64), ctypes.POINTER(u64),
                                         ctypes.POINTER(u32)]
    L.rcd_ingest_counts.argtypes = [vp, ctypes.POINTER(u64), ctypes.POINTER(u64)]
    L.rcd_ingest_set_limit.argtypes = [vp, u64]
    L.rcd_ingest_rejected.argtypes = [vp, ctypes.POINTER(u64)]
    L.rcd_ingest_id_name.argtypes = [vp, u32, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(u32)]
    L.rcd_ingest_type_name.argtypes = [vp, u32, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(u32)]
    L.rcd_ingest_lookup.argtypes = [vp, ctypes.c_char_p, u32, ctypes.POINTER(u32)]
    L.rcd_apply_records.argtypes = [vp, u64, vp, u32, u64, i32, i32]
    L.rcd_ingest_release.argtypes = [vp, u64, vp, ctypes.POINTER(u64)]
    f64 = ctypes.c_double
    L.rcd_alerts_configure.argtypes = [vp, u64]
    L.rcd_alerts_reserve.argtypes = [vp, u64]
    L.rcd_reserve.argtypes = [vp, u64, u64]
    L.rcd_alerts_update.argtypes = [vp, f64, i32, vp, u64, ctypes.POINTER(RcdAlertStats)]
    L.rcd_alerts_update_pairs.argtypes = [vp, vp, u64, f64, i32, vp, u64, ctypes.POINTER(RcdAlertStats)]
    L.rcd_alerts_expire.argtypes = [vp, f64, f64, vp, u64, ctypes.POINTER(RcdAlertStats)]
    L.rcd_alerts_acknowledge.argtypes = [vp, u64, vp, vp, ctypes.POINTER(u64)]
    L.rcd_alerts_download.argtypes = [vp, vp, u64, ctypes.POINTER(u64)]
    L.rcd_retire.argtypes = [vp, u64, vp, vp, u64, ctypes.POINTER(RcdAlertStats)]
    L.rcd_retire_stale.argtypes = [vp, f64, f64, vp, u64, ctypes.POINTER(u64), vp, u64, ctypes.POINTER(RcdAlertStats)]
    for name in SYMBOLS:
        if not hasattr(L, name) and os.environ.get("RCD_B200_LIB"):
            continue  # an older build loaded for an A/B kernel experiment
        fn = getattr(L, name)
        if name not in ("rcd_last_error", "rcd_version", "rcd_ingest_last_error"):
            fn.restype = ctypes.c_int
    _lib = L
    return L


def check(rc: int, handle=None) -> None:
    if rc != RCD_OK:
        msg = load().rcd_last_error(handle)
        raise NativeError(rc, msg.decode("utf-8", "replace") if msg else "")
