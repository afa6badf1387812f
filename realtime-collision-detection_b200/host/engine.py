"""Whole-frame engine over the C-ABI: the additive batch API the drop-in classes are built on.

One ``FrameEngine`` owns one ``rcd_handle`` (one GPU, one stream).  Frames are dicts of fp32 SoA
numpy arrays (see ``workloads.py``) or raw device pointers.
"""
from __future__ import annotations

import ctypes
from typing import Dict, Optional, Sequence, Tuple

import numpy as np

from . import _native as N

FRAME_FIELDS = ("px", "py", "pz", "vx", "vy", "vz", "ax", "ay", "az", "size", "heading")


def _as(a, dtype) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=dtype)


def _vp(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


class FrameEngine:
    """Batch interface: upload a frame, run detect / predict / compute-node for every object."""

    def __init__(self, max_objects: int, max_pairs: Optional[int] = None, device: int = 0,
                 world_bounds: Optional[Tuple[Sequence[float], Sequence[float]]] = None, profile: bool = False,
                 count_predict_candidates: bool = False, graph: bool = False):
        self._lib = N.load()
        self._h = ctypes.c_void_p()
        cfg = N.RcdConfig()
        cfg.device = int(device)
        cfg.flags = (N.FLAG_PROFILE if profile else 0) | (
            N.FLAG_COUNT_PREDICT_CANDIDATES if count_predict_candidates else 0) | (N.FLAG_GRAPH if graph else 0)
        cfg.max_objects = int(max(1, max_objects))
        cfg.max_pairs = int(max_pairs if max_pairs is not None else max(4096, 16 * max_objects))
        if world_bounds is None:
            cfg.world_min[:] = [1.0, 1.0, 1.0]
            cfg.world_max[:] = [0.0, 0.0, 0.0]
        else:
            cfg.world_min[:] = [float(v) for v in world_bounds[0]]
            cfg.world_max[:] = [float(v) for v in world_bounds[1]]
        self.max_objects = int(cfg.max_objects)
        self.max_pairs = int(cfg.max_pairs)
        self.device = int(device)
        self.n = 0
        N.check(self._lib.rcd_create(ctypes.byref(cfg), ctypes.byref(self._h)))

    # -- lifetime ---------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.rcd_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def reserve(self, max_objects: Optional[int] = None, max_pairs: Optional[int] = None) -> None:
        """Grow the handle in place (rcd_reserve): None or a value below the current one keeps it.  The objects,
        patterns, trajectory rings, record times, query list and alert table stay on the device; the frame ends."""
        N.check(self._lib.rcd_reserve(self._h, int(max_objects or 0), int(max_pairs or 0)), self._h)
        self.max_objects = max(self.max_objects, int(max_objects or 0))
        self.max_pairs = max(self.max_pairs, int(max_pairs or 0))

    # -- state ------------------------------------------------------------------------------
    def upload(self, frame: Dict[str, np.ndarray], ids: Optional[np.ndarray] = None) -> None:
        """N x update_vehicle (collision_detection.py:74-85) as one SoA copy."""
        arrs = [_as(frame[k], np.float32) for k in FRAME_FIELDS]
        n = int(arrs[0].shape[0])
        typ = _as(frame["type"], np.uint8) if "type" in frame else None
        idv = _as(ids, np.uint32) if ids is not None else None
        self._keep = (arrs, typ, idv)  # keep the host buffers alive until the copies are done
        N.check(self._lib.rcd_upload(self._h, n, *[_vp(a) for a in arrs], _vp(typ), _vp(idv), N.SRC_HOST), self._h)
        self.n = n

    def upload_ptrs(self, n: int, ptrs: Sequence[int], type_ptr: int = 0, id_ptr: int = 0,
                    src: int = N.SRC_DEVICE) -> None:
        """Same, from 11 raw pointers (float32, n entries each, FRAME_FIELDS order) in device memory
        (src=SRC_DEVICE) or host memory (src=SRC_HOST; pinned memory makes the copies asynchronous)."""
        args = [ctypes.c_void_p(int(p)) if p else None for p in ptrs]
        N.check(self._lib.rcd_upload(self._h, int(n), *args, ctypes.c_void_p(type_ptr) if type_ptr else None,
                                     ctypes.c_void_p(id_ptr) if id_ptr else None, int(src)), self._h)
        self.n = int(n)

    def upload_device(self, n: int, ptrs: Sequence[int], type_ptr: int = 0, id_ptr: int = 0) -> None:
        self.upload_ptrs(n, ptrs, type_ptr, id_ptr, N.SRC_DEVICE)

    def upload_host_ptrs(self, n: int, ptrs: Sequence[int], type_ptr: int = 0, id_ptr: int = 0) -> None:
        self.upload_ptrs(n, ptrs, type_ptr, id_ptr, N.SRC_HOST)

    def apply_records(self, records: np.ndarray, n_objects: int, max_seq: int = 0, history: bool = True) -> None:
        """Scatter decoded vehicle messages (``_native.RECORD_DTYPE``, see ``ingest.py``) into the frame:
        N x update_vehicle + N x update_trajectory (warning_system.py:638-678) in one call."""
        rec = np.ascontiguousarray(records, dtype=N.RECORD_DTYPE)
        N.check(self._lib.rcd_apply_records(self._h, int(rec.shape[0]), _vp(rec) if rec.shape[0] else None, int(max_seq),
                                            int(n_objects), 1 if history else 0, N.SRC_HOST), self._h)
        self.n = int(n_objects)

    def apply_records_device(self, n: int, ptr: int, n_objects: int, max_seq: int = 0, history: bool = True) -> None:
        N.check(self._lib.rcd_apply_records(self._h, int(n), ctypes.c_void_p(int(ptr)), int(max_seq), int(n_objects),
                                            1 if history else 0, N.SRC_DEVICE), self._h)
        self.n = int(n_objects)

    def set_patterns_ptr(self, n: int, ptr: int, src: int) -> None:
        N.check(self._lib.rcd_set_patterns(self._h, int(n), ctypes.c_void_p(int(ptr)) if ptr else None, int(src)),
                self._h)

    def set_patterns_device(self, n: int, ptr: int) -> None:
        self.set_patterns_ptr(n, ptr, N.SRC_DEVICE)

    def set_patterns_host_ptr(self, n: int, ptr: int) -> None:
        self.set_patterns_ptr(n, ptr, N.SRC_HOST)

    def set_patterns(self, pattern: Optional[np.ndarray]) -> None:
        if pattern is None:
            N.check(self._lib.rcd_set_patterns(self._h, self.n, None, N.SRC_HOST), self._h)
            return
        p = _as(pattern, np.uint8)
        self._keep_pat = p
        N.check(self._lib.rcd_set_patterns(self._h, int(p.shape[0]), _vp(p), N.SRC_HOST), self._h)

    def set_owned(self, n_owned: int) -> None:
        N.check(self._lib.rcd_set_owned(self._h, int(n_owned)), self._h)

    def set_queries(self, slots: Optional[np.ndarray]) -> None:
        """Query only the listed upload slots (each < n_owned, no repeats) in the following steps; every object
        stays a neighbour.  None: back to every owned object.  The spatial index is kept (rcd_set_queries)."""
        if slots is None:
            N.check(self._lib.rcd_set_queries(self._h, 0, None, N.SRC_HOST), self._h)
            return
        s = _as(slots, np.uint32)
        buf = s if s.shape[0] else np.zeros(1, np.uint32)  # (n = 0 still needs a non-NULL list)
        N.check(self._lib.rcd_set_queries(self._h, int(s.shape[0]), _vp(buf), N.SRC_HOST), self._h)

    def set_queries_device(self, n: int, ptr: int) -> None:
        """Same, from n uint32 slots in device memory (checked on the device; synchronises)."""
        N.check(self._lib.rcd_set_queries(self._h, int(n), ctypes.c_void_p(int(ptr)), N.SRC_DEVICE), self._h)

    def set_compute_node_params(self, prediction_time: float = 5.0, risk_threshold: float = 0.5) -> None:
        N.check(self._lib.rcd_set_compute_node_params(self._h, float(prediction_time), float(risk_threshold)), self._h)

    def truncate(self, n: int) -> None:
        """Drop everything after the first n objects (the halo copies of the previous frame)."""
        N.check(self._lib.rcd_truncate(self._h, int(n)), self._h)
        self.n = int(n)

    def invalidate(self) -> None:
        N.check(self._lib.rcd_invalidate(self._h), self._h)

    # -- retiring departed vehicles (rcd_retire, rcd_retire_stale) -------------------------------------
    def _retire_events(self) -> np.ndarray:
        return self._alert_events(None) if getattr(self, "_alert_cap", 0) else np.zeros(0, N.ALERT_EVENT_DTYPE)

    def retire(self, slots) -> Tuple[np.ndarray, np.ndarray, Dict[str, int]]:
        """remove_vehicle for the listed slots: they keep their place in the frame but have no position, are nobody's
        neighbour and emit nothing; their alerts are dropped.  Returns (slots, EXPIRED events, alert stats)."""
        s = _as(slots, np.uint32)
        ev, st = self._retire_events(), N.RcdAlertStats()
        N.check(self._lib.rcd_retire(self._h, int(s.shape[0]), _vp(s) if s.shape[0] else None, _vp(ev) if ev.shape[0] else None,
                                     ev.shape[0], ctypes.byref(st)), self._h)
        return s, ev[: min(int(st.n_events), ev.shape[0])], self._alert_stats(st)

    def retire_stale(self, now: float, max_age: float) -> Tuple[np.ndarray, np.ndarray, Dict[str, int]]:
        """Retire every slot whose newest applied record is older than max_age at `now` (now - t > max_age).
        Returns (retired slots ascending, EXPIRED events, alert stats).  Record-built frames only."""
        ev, st, n = self._retire_events(), N.RcdAlertStats(), ctypes.c_uint64(0)
        out = np.empty(max(1, self.n), np.uint32)  # (written up to n_retired)
        N.check(self._lib.rcd_retire_stale(self._h, float(now), float(max_age), _vp(out), out.shape[0], ctypes.byref(n),
                                           _vp(ev) if ev.shape[0] else None, ev.shape[0], ctypes.byref(st)), self._h)
        return out[: int(n.value)], ev[: min(int(st.n_events), ev.shape[0])], self._alert_stats(st)

    # -- frames -----------------------------------------------------------------------------
    def step(self, mode: int, search_radius: float = 100.0, time_window: float = 10.0, append: bool = False,
             with_detect: bool = False) -> None:
        """One frame for every owned object (or the set_queries list).  ``append``: keep the pairs / totals of the previous step of this
        frame.  ``with_detect`` (predict mode): also run detect_collisions(search_radius, time_window) in the
        same pass -- the result of step(DETECT) + step(PREDICT, append=True) for one sweep over the data."""
        m = int(mode) | (N.STEP_APPEND if append else 0) | (N.STEP_WITH_DETECT if with_detect else 0)
        N.check(self._lib.rcd_step(self._h, m, float(search_radius), float(time_window)), self._h)

    def build_index(self, cell_radius: float = 100.0) -> None:
        N.check(self._lib.rcd_build_index(self._h, float(cell_radius)), self._h)

    def counts(self) -> Dict[str, int]:
        c = N.RcdCounts()
        N.check(self._lib.rcd_counts(self._h, ctypes.byref(c)), self._h)
        return {"n_objects": c.n_objects, "n_owned": c.n_owned, "n_candidates": c.n_candidates,
                "n_potential": c.n_potential, "n_pairs": c.n_pairs, "n_high_risk": c.n_high_risk,
                "n_written": c.n_written, "n_alerts": [int(v) for v in c.n_alerts], "n_exact": c.n_exact,
                "n_fallback": c.n_fallback}

    def download(self, cap: Optional[int] = None, sort: bool = True, out: Optional[np.ndarray] = None) -> np.ndarray:
        """Emitted pairs as a PAIR_DTYPE array, sorted by (i, j, predicted) unless sort=False.
        `out`: preallocated (e.g. pinned) PAIR_DTYPE buffer to copy into."""
        cap = int(self.max_pairs if cap is None else cap)
        c = self.counts()
        m = min(cap, int(c["n_written"]))
        if out is None:
            out = np.empty(m, N.PAIR_DTYPE)
        m = min(m, out.shape[0])
        got = ctypes.c_uint64(0)
        fn = self._lib.rcd_download if sort else self._lib.rcd_download_unsorted
        N.check(fn(self._h, _vp(out), m, ctypes.byref(got)), self._h)
        return out[: got.value]

    def download_begin(self, out: np.ndarray) -> None:
        """Start delivering the frame just stepped into ``out`` (PAIR_DTYPE, ideally pinned) and return at
        once: the next upload / step can be issued while the copy runs (the handle has twin pair buffers)."""
        self._pending_out = out
        N.check(self._lib.rcd_download_begin(self._h, _vp(out), int(out.shape[0])), self._h)

    def download_finish(self) -> Tuple[np.ndarray, Dict[str, int]]:
        """Wait for the pending delivery; returns (pairs in emission order, totals of that frame)."""
        c, n = N.RcdCounts(), ctypes.c_uint64()
        N.check(self._lib.rcd_download_finish(self._h, ctypes.byref(c), ctypes.byref(n)), self._h)
        out, self._pending_out = self._pending_out, None
        d = {k: int(getattr(c, k)) for k, _ in N.RcdCounts._fields_ if k != "n_alerts"}
        d["n_alerts"] = [int(v) for v in c.n_alerts]
        return out[: int(n.value)], d

    def download_begin_compact(self, out: np.ndarray) -> None:
        """Like download_begin with 32-byte records (``PAIR_COMPACT_DTYPE``): narrowed on the device first."""
        self._pending_out = out
        N.check(self._lib.rcd_download_begin_compact(self._h, _vp(out), int(out.shape[0])), self._h)

    def summary_begin(self, now: float, report_refreshed: bool = False) -> None:
        """Start the summary delivery of the frame just stepped (alert changes + per-object risk counts) and
        return at once; needs alerts_configure."""
        N.check(self._lib.rcd_summary_begin(self._h, float(now), 1 if report_refreshed else 0), self._h)

    def summary_finish(self, events: Optional[np.ndarray] = None, risk_counts: Optional[np.ndarray] = None):
        """Wait for the pending summary: (events, alert stats, risk counts or None, frame totals)."""
        ev = self._alert_events(None) if events is None else events
        st, c, n_ev = N.RcdAlertStats(), N.RcdCounts(), ctypes.c_uint64()
        nrc = 0 if risk_counts is None else int(risk_counts.shape[0])
        N.check(self._lib.rcd_summary_finish(self._h, _vp(ev), ev.shape[0], ctypes.byref(n_ev), ctypes.byref(st),
                                             _vp(risk_counts) if nrc else None, nrc, ctypes.byref(c)), self._h)
        d = {k: int(getattr(c, k)) for k, _ in N.RcdCounts._fields_ if k != "n_alerts"}
        d["n_alerts"] = [int(v) for v in c.n_alerts]
        return ev[: int(n_ev.value)], self._alert_stats(st), risk_counts, d

    def risk_counts(self) -> np.ndarray:
        """Risks emitted per object (as the querying vehicle) in the last frame, upload order."""
        out = np.zeros(self.n, np.uint32)
        N.check(self._lib.rcd_download_risk_counts(self._h, _vp(out), out.shape[0]), self._h)
        return out

    def candidate_counts(self) -> np.ndarray:
        out = np.zeros(int(self.counts()["n_objects"]), np.uint32)
        N.check(self._lib.rcd_download_candidate_counts(self._h, _vp(out), out.shape[0]), self._h)
        return out

    def detect(self, search_radius: float = 100.0, time_window: float = 10.0) -> np.ndarray:
        self.step(N.MODE_DETECT, search_radius, time_window)
        return self.download()

    def predict(self) -> np.ndarray:
        self.step(N.MODE_PREDICT)
        return self.download()

    def compute_node(self, search_radius: float = 100.0) -> np.ndarray:
        self.step(N.MODE_COMPUTE_NODE, search_radius)
        return self.download()

    # -- queries ----------------------------------------------------------------------------
    def query_radius(self, queries, radius: float):
        """get_nearby_vehicles / query_nearby for a batch of points -> list of id arrays."""
        q = _as(queries, np.float32).reshape(-1, 3)
        nq = q.shape[0]
        qx, qy, qz = (np.ascontiguousarray(q[:, k]) for k in range(3))
        offs = np.zeros(nq + 1, np.uint64)
        cap = max(1024, 64 * nq)
        for _ in range(3):
            ids = np.zeros(cap, np.uint32)
            rc = self._lib.rcd_query_radius(self._h, nq, _vp(qx), _vp(qy), _vp(qz), float(radius), _vp(offs),
                                            _vp(ids), cap)
            if rc == N.RCD_ECAPACITY:
                cap = int(offs[nq]) + 16
                continue
            N.check(rc, self._h)
            break
        else:  # pragma: no cover
            raise N.NativeError(N.RCD_ECAPACITY, "query_radius: result buffer kept overflowing")
        return [ids[int(offs[k]): int(offs[k + 1])].copy() for k in range(nq)]

    def classify_patterns(self, samples: np.ndarray, count: np.ndarray) -> np.ndarray:
        """samples: float64 [n, stride, 4] (x, y, z, t) in timestamp order; count: valid samples."""
        s = _as(samples, np.float64)
        n, stride = int(s.shape[0]), int(s.shape[1])
        c = _as(count, np.uint32)
        out = np.zeros(n, np.uint8)
        N.check(self._lib.rcd_classify_patterns(self._h, n, stride, _vp(s), _vp(c), _vp(out)), self._h)
        return out

    # -- the detector's per-pair helpers (collision_detection.py:296-389) ------------------------------------
    def pair_exact(self, a: np.ndarray, b: np.ndarray, time_window: float = 10.0, time_step: float = 0.1) -> np.ndarray:
        """_precise_collision_detection + _risk_assessment for explicit pairs (OBJECT_DTYPE arrays) -> PAIR_EXACT_DTYPE."""
        aa, bb = np.ascontiguousarray(a, dtype=N.OBJECT_DTYPE), np.ascontiguousarray(b, dtype=N.OBJECT_DTYPE)
        out = np.zeros(aa.shape[0], dtype=N.PAIR_EXACT_DTYPE)
        N.check(self._lib.rcd_pair_exact(self._h, aa.shape[0], _vp(aa), _vp(bb), float(time_window), float(time_step), _vp(out)),
                self._h)
        return out

    def risk_assessment(self, records: np.ndarray) -> np.ndarray:
        """records: float64 [n, 7] = heading_i, heading_j, same type (1 / 0), collision_time, distance, safe_distance,
        relative_speed -> risk level (collision_detection.py:344-389)."""
        r = _as(records, np.float64).reshape(-1, 7)
        out = np.zeros(r.shape[0], np.float64)
        N.check(self._lib.rcd_risk_assessment(self._h, r.shape[0], _vp(r), _vp(out)), self._h)
        return out

    # -- device-resident trajectory history ---------------------------------------------------------
    def history_configure(self, max_history: int = 100) -> None:
        N.check(self._lib.rcd_history_configure(self._h, int(max_history)), self._h)

    def history_append(self, slots, x, y, z, t) -> None:
        """One (x, y, z, t) float64 sample for each listed slot (slots=None: 0..n-1)."""
        xs, ys, zs, ts = (_as(a, np.float64) for a in (x, y, z, t))
        sl = None if slots is None else _as(slots, np.uint32)
        N.check(self._lib.rcd_history_append(self._h, int(xs.shape[0]), _vp(sl), _vp(xs), _vp(ys), _vp(zs), _vp(ts)),
                self._h)

    def history_reset(self, slots) -> None:
        sl = _as(slots, np.uint32)
        N.check(self._lib.rcd_history_reset(self._h, int(sl.shape[0]), _vp(sl)), self._h)

    def history_move(self, dst: int, src: int) -> None:
        N.check(self._lib.rcd_history_move(self._h, int(dst), int(src)), self._h)

    def history_classify(self, want_codes: bool = True) -> Optional[np.ndarray]:
        out = np.zeros(self.n, np.uint8) if want_codes else None
        N.check(self._lib.rcd_history_classify(self._h, _vp(out)), self._h)
        return out

    # -- alert lifecycle (warning_system.py:120-197, 259-285, 488-517) ----------------------
    def alerts_configure(self, max_alerts: int) -> None:
        N.check(self._lib.rcd_alerts_configure(self._h, int(max_alerts)), self._h)
        self._alert_cap = int(max_alerts)

    def alerts_reserve(self, max_alerts: int) -> None:
        """Grow the alert table to max_alerts live alerts, keeping every live alert and the alert numbering."""
        N.check(self._lib.rcd_alerts_reserve(self._h, int(max_alerts)), self._h)
        self._alert_cap = max(self._alert_cap, int(max_alerts))

    @staticmethod
    def _alert_stats(st: "N.RcdAlertStats") -> Dict[str, int]:
        return {k: int(getattr(st, k)) for k, _ in N.RcdAlertStats._fields_}

    def _alert_events(self, cap: Optional[int]) -> np.ndarray:
        return np.zeros(self._alert_cap if cap is None else int(cap), dtype=N.ALERT_EVENT_DTYPE)

    def alerts_update(self, now: float, report_refreshed: bool = False, cap: Optional[int] = None):
        """process_collision_risks on the pairs of the last frame; returns (events, stats)."""
        ev, st = self._alert_events(cap), N.RcdAlertStats()
        N.check(self._lib.rcd_alerts_update(self._h, float(now), 1 if report_refreshed else 0, _vp(ev), ev.shape[0],
                                            ctypes.byref(st)), self._h)
        return ev[: min(int(st.n_events), ev.shape[0])], self._alert_stats(st)

    def alerts_update_pairs(self, pairs: np.ndarray, now: float, report_refreshed: bool = False, cap: Optional[int] = None):
        p = np.ascontiguousarray(pairs, dtype=N.PAIR_DTYPE)
        ev, st = self._alert_events(cap), N.RcdAlertStats()
        N.check(self._lib.rcd_alerts_update_pairs(self._h, _vp(p) if p.shape[0] else None, p.shape[0], float(now),
                                                  1 if report_refreshed else 0, _vp(ev), ev.shape[0], ctypes.byref(st)), self._h)
        return ev[: min(int(st.n_events), ev.shape[0])], self._alert_stats(st)

    def alerts_expire(self, now: float, max_age: float = 30.0, cap: Optional[int] = None):
        ev, st = self._alert_events(cap), N.RcdAlertStats()
        N.check(self._lib.rcd_alerts_expire(self._h, float(now), float(max_age), _vp(ev), ev.shape[0], ctypes.byref(st)), self._h)
        return ev[: min(int(st.n_events), ev.shape[0])], self._alert_stats(st)

    def alerts_acknowledge(self, i, j) -> int:
        ii, jj = _as(i, np.uint32), _as(j, np.uint32)
        found = ctypes.c_uint64()
        N.check(self._lib.rcd_alerts_acknowledge(self._h, ii.shape[0], _vp(ii), _vp(jj), ctypes.byref(found)), self._h)
        return int(found.value)

    def alerts_download(self, cap: Optional[int] = None) -> np.ndarray:
        ev = self._alert_events(cap)
        n = ctypes.c_uint64()
        N.check(self._lib.rcd_alerts_download(self._h, _vp(ev), ev.shape[0], ctypes.byref(n)), self._h)
        return ev[: int(n.value)]

    # -- slabs ------------------------------------------------------------------------------
    def halo_pack(self, slab_lo, slab_hi, self_rank: int, halo: float, out_ptr: int, cap: int) -> np.ndarray:
        lo = _as(slab_lo, np.float32)
        hi = _as(slab_hi, np.float32)
        counts = np.zeros(lo.shape[0], np.uint64)
        N.check(self._lib.rcd_halo_pack(self._h, int(lo.shape[0]), int(self_rank), _vp(lo), _vp(hi), float(halo),
                                        ctypes.c_void_p(int(out_ptr)) if out_ptr else None, int(cap), _vp(counts)),
                self._h)
        return counts.astype(np.int64)

    def halo_pack_async(self, slab_lo, slab_hi, self_rank: int, halo: float, out_ptr: int, peer_offset: np.ndarray,
                        counts_ptr: int) -> None:
        """Single-pass pack into fixed per-peer regions of a device buffer; counts stay on the device."""
        lo, hi = _as(slab_lo, np.float32), _as(slab_hi, np.float32)
        off = _as(peer_offset, np.uint64)
        N.check(self._lib.rcd_halo_pack_async(self._h, int(lo.shape[0]), int(self_rank), _vp(lo), _vp(hi), float(halo),
                                              ctypes.c_void_p(int(out_ptr)), _vp(off), ctypes.c_void_p(int(counts_ptr))), self._h)

    def halo_append(self, rec_ptr: int, n_records: int) -> None:
        N.check(self._lib.rcd_halo_append(self._h, ctypes.c_void_p(int(rec_ptr)) if rec_ptr else None,
                                          int(n_records)), self._h)
        self.n += int(n_records)

    # -- instrumentation -----------------------------------------------------------------------
    def stage_ms(self, mode: int = N.MODE_DETECT) -> Dict[str, float]:
        ms = np.zeros(N.NUM_STAGES, np.float32)
        N.check(self._lib.rcd_stage_ms(self._h, int(mode), _vp(ms)), self._h)
        return {name: float(ms[k]) for k, name in enumerate(N.STAGE_NAMES)}

    def cuda_stream(self) -> int:
        """The handle's cudaStream_t as an integer (wrap with torch.cuda.ExternalStream)."""
        s = ctypes.c_void_p()
        N.check(self._lib.rcd_get_stream(self._h, ctypes.byref(s)), self._h)
        return int(s.value or 0)

    def launch_count(self) -> int:
        v = ctypes.c_uint64(0)
        N.check(self._lib.rcd_launch_count(self._h, ctypes.byref(v)), self._h)
        return int(v.value)

    def pair_tests(self) -> int:
        """(query, neighbour) tests of the pair kernel's fp32 filter in the last frame."""
        v = ctypes.c_uint64(0)
        N.check(self._lib.rcd_pair_tests(self._h, ctypes.byref(v)), self._h)
        return int(v.value)

    def graph_replays(self) -> int:
        n = ctypes.c_uint64()
        N.check(self._lib.rcd_graph_replays(self._h, ctypes.byref(n)), self._h)
        return int(n.value)

    def sync(self) -> None:
        N.check(self._lib.rcd_sync(self._h), self._h)
