"""The handle's own bookkeeping on the device: kernel-launch counts per frame variant, a refused allocation
in rcd_create, and repeated create / use / destroy cycles."""
import ctypes
import re

import numpy as np
import pytest

from tests.gpu_helpers import compare_pairs
from tests.helpers import f64_frame

pytestmark = pytest.mark.gpu

N_OBJ = 4000

# rcd_launch_count after one frame of each kind on a fresh 4000-object handle.  bench.py reports this
# number as gpu_launches, so it must not move when the host code around the kernels changes.
LAUNCHES = {
    "detect": 15,
    "predict": 15,
    "predict_count_candidates": 15,
    "compute_node": 15,
    "fused": 15,
    "detect_then_predict_appended": 24,
    "fused_graph_replay": 14,
}


def _frame():
    from rcd_b200.host import workloads as W
    return W.uniform_frame(N_OBJ, 7, map_size=800.0, drone_fraction=0.3), W.random_patterns(N_OBJ, 8)


def launch_counts():
    from rcd_b200.host import _native as N
    from rcd_b200.host.engine import FrameEngine
    frame, pat = _frame()
    frames = {
        "detect": lambda e: e.step(N.MODE_DETECT),
        "predict": lambda e: e.step(N.MODE_PREDICT),
        "compute_node": lambda e: e.step(N.MODE_COMPUTE_NODE),
        "fused": lambda e: e.step(N.MODE_PREDICT, with_detect=True),
        "detect_then_predict_appended": lambda e: (e.step(N.MODE_DETECT), e.step(N.MODE_PREDICT, append=True)),
    }
    got = {}
    with FrameEngine(N_OBJ, 64 * N_OBJ) as e:
        for name, step in frames.items():
            e.upload(frame)
            e.set_patterns(pat)
            step(e)
            got[name] = e.launch_count()
    with FrameEngine(N_OBJ, 64 * N_OBJ, count_predict_candidates=True) as e:
        e.upload(frame)
        e.set_patterns(pat)
        e.step(N.MODE_PREDICT)
        got["predict_count_candidates"] = e.launch_count()
    bounds = ((0.0, 0.0, 0.0), (800.0, 800.0, 100.0))
    with FrameEngine(N_OBJ, 64 * N_OBJ, world_bounds=bounds, graph=True) as e:
        for _ in range(3):  # first sighting runs, second is captured, third replays
            e.upload(frame)
            e.set_patterns(pat)
            e.step(N.MODE_PREDICT, with_detect=True)
        assert e.graph_replays() == 1
        got["fused_graph_replay"] = e.launch_count()
    return got


def test_launch_count_of_each_frame_variant():
    assert launch_counts() == LAUNCHES


def test_create_refuses_a_pair_buffer_larger_than_the_device_then_a_normal_handle_works():
    from oracle import oracle as O
    from rcd_b200.host import _native as N
    from rcd_b200.host.engine import FrameEngine
    lib = N.load()
    cfg = N.RcdConfig()
    cfg.max_objects = N_OBJ
    cfg.max_pairs = 1 << 40  # 48-byte records: 52 TB, refused without allocating anything
    cfg.world_min[:] = [1.0, 1.0, 1.0]
    cfg.world_max[:] = [0.0, 0.0, 0.0]
    h = ctypes.c_void_p()
    assert lib.rcd_create(ctypes.byref(cfg), ctypes.byref(h)) == N.RCD_ENOMEM
    assert not h
    msg = lib.rcd_last_error(None)
    assert re.search(rb"\bout\b.*max_pairs", msg), msg
    frame, _ = _frame()
    with FrameEngine(N_OBJ, 64 * N_OBJ) as e:
        e.upload(frame)
        got = e.detect()
    compare_pairs(got, O.frame_A(f64_frame(frame), "detect")["risks"], "detect")


def test_repeated_create_use_destroy_cycles():
    from rcd_b200.host import _native as N
    from rcd_b200.host.engine import FrameEngine
    frame, pat = _frame()
    n = N_OBJ
    rng = np.random.default_rng(5)
    for k in range(20):
        with FrameEngine(n, 64 * n) as e:
            e.alerts_configure(1 << 14)
            e.upload(frame)
            e.set_patterns(pat)
            e.step(N.MODE_PREDICT, with_detect=True)
            e.download_begin(np.zeros(64 * n, N.PAIR_DTYPE))
            pairs, counts = e.download_finish()
            assert len(pairs) == counts["n_pairs"] > 0
            e.step(N.MODE_PREDICT, with_detect=True)
            e.download_begin_compact(np.zeros(64 * n, N.PAIR_COMPACT_DTYPE))
            compact, _ = e.download_finish()
            assert len(compact) == len(pairs)
            e.step(N.MODE_PREDICT, with_detect=True)
            e.summary_begin(100.0 + k)
            ev, st, rc, _ = e.summary_finish(risk_counts=np.zeros(n, np.uint32))
            assert st["n_created"] > 0 and int(rc.sum()) == len(pairs)
            e.alerts_update_pairs(pairs[:100], 101.0 + k)
            e.alerts_acknowledge(pairs["i"][:10], pairs["j"][:10])
            e.alerts_expire(200.0 + k, 30.0)
            e.alerts_download()
            for t in range(3):
                e.history_append(None, frame["px"] + t, frame["py"], frame["pz"], np.full(n, 0.1 * t))
            e.history_reset(np.arange(10, dtype=np.uint32))
            e.history_classify()
            e.query_radius(rng.uniform(0.0, 800.0, (16, 3)), 50.0)
