"""Drop-in for src/collision/collision_detection.py: ``CollisionDetector`` and
``CollisionPredictionModel`` with the reference's signatures and return types (SURVEY.md 8b).

Per-vehicle calls are served from whole-frame GPU results: the first ``detect_collisions`` /
``predict_collisions`` after an update runs one frame for every vehicle (csrc/rcd_pairs.cuh);
the following calls are O(1) look-ups until a vehicle changes.  The additive batch entry points
``detect_all`` / ``predict_all`` return every vehicle's risks at once.
"""
from __future__ import annotations

import time
from typing import Any, Dict, List, Optional, Set, Tuple

import numpy as np

from . import _native as N
from .models import CollisionRisk, Position, Vector, Vehicle
from .spatial_index import SpatialIndex

SAFE_DISTANCE_DEFAULT = 5.0
MAX_WARNING_TIME = 10.0
MAX_RELATIVE_SPEED = 50.0
WEIGHT_DISTANCE, WEIGHT_TIME, WEIGHT_SPEED, WEIGHT_ANGLE, WEIGHT_TYPE = 0.3, 0.3, 0.2, 0.1, 0.1


_FRAME_STAMP = [0]


def _make_risk(r, ids: List[str], rid: str, now: float) -> CollisionRisk:
    return CollisionRisk(
        id=rid, vehicle_id=ids[int(r["i"])], other_vehicle_id=ids[int(r["j"])],
        time_to_collision=float(r["ttc"]), distance=float(r["distance"]), relative_speed=float(r["rel_speed"]),
        risk_level=float(r["risk"]),
        collision_position=Position(float(r["cx"]), float(r["cy"]), float(r["cz"])), timestamp=now,
        is_predicted=bool(r["predicted"]), alert_priority=int(r["priority"]),
        time_to_closest=float(r["t_closest"]), closest_distance=float(r["d_closest"]))


class RiskList(list):
    """The ``List[CollisionRisk]`` the reference returns -- a real ``list`` -- whose ``CollisionRisk`` objects are built
    from the rows of the frame's pair table the first time anything looks at an element (iteration, indexing, ``+``,
    a mutator ...).  ``len(risks)`` / ``if risks:`` cost nothing per risk, which is all the reference's perf harness
    does with the result (performance_test.py:802-809).  Risk ids are ``risk-<frame>-<row>`` (unique per process; the
    reference draws a uuid4 per risk, collision_detection.py:157).  C extensions that read a list's storage directly
    (``json``) should be handed ``list(risks)``."""

    def __init__(self, pairs: np.ndarray, ids: List[str], tag: str, now: float):
        super().__init__()
        self._pairs, self._ids, self._tag, self._now = pairs, ids, tag, now
        self._pending = pairs.shape[0] > 0

    def _fill(self) -> None:
        if self._pending:
            self._pending = False
            list.extend(self, [_make_risk(r, self._ids, f"risk-{self._tag}-{k}", self._now) for k, r in enumerate(self._pairs)])

    @property
    def table(self) -> np.ndarray:
        """The underlying rows (``_native.PAIR_DTYPE``; i / j are slots of the object table)."""
        return self._pairs

    def __len__(self) -> int:
        return int(self._pairs.shape[0]) if self._pending else list.__len__(self)

    def __bool__(self) -> bool:
        return len(self) > 0

    def __reduce__(self):
        return (list, (list(self),))


def _filled(name):
    base = getattr(list, name)

    def method(self, *a, **kw):
        self._fill()
        return base(self, *a, **kw)

    method.__name__ = name
    return method


for _name in ("__iter__", "__getitem__", "__setitem__", "__delitem__", "__contains__", "__reversed__", "__add__", "__iadd__",
              "__mul__", "__rmul__", "__imul__", "__eq__", "__ne__", "__lt__", "__le__", "__gt__", "__ge__", "__repr__",
              "append", "extend", "insert", "pop", "remove", "sort", "reverse", "clear", "count", "index", "copy"):
    setattr(RiskList, _name, _filled(_name))
RiskList.__hash__ = None
RiskList.__radd__ = lambda self, other: list(other) + list(self)


def _risks_from_pairs(pairs: np.ndarray, ids: List[str], tag: Optional[str] = None) -> RiskList:
    if tag is None:
        _FRAME_STAMP[0] += 1
        tag = f"{_FRAME_STAMP[0]:x}"
    return RiskList(pairs, ids, tag, time.time())


def _rows_for(spatial_index: SpatialIndex, vehicle_ids, kind: str, frame) -> Dict[str, List[CollisionRisk]]:
    """{id: risks} for the known ids among `vehicle_ids`, from frame(slots) = (pairs, starts, counts)."""
    table = spatial_index._table
    slots = sorted({table.slot_of[v] for v in vehicle_ids if v in table.slot_of})
    if not slots:
        return {}
    sl = np.asarray(slots, np.uint32)
    pairs, starts, _ = frame(sl)
    tag = f"{kind}{spatial_index._frames.frames_run:x}"
    return {table.ids[s]: _risks_from_pairs(pairs[starts[s]:starts[s + 1]], table.ids, f"{tag}-{s:x}")
            for s in slots if starts[s + 1] > starts[s]}


class CollisionDetector:
    def __init__(self, spatial_index: SpatialIndex):
        self.spatial_index = spatial_index
        self.vehicle_cache: Dict[str, Vehicle] = {}
        self._collision_risks: Dict[str, Dict[str, CollisionRisk]] = {}
        self._latest: Dict[str, RiskList] = {}  # results not yet folded into collision_risks (built on first read)
        self.stats = {"total_detections": 0, "potential_collisions": 0, "high_risk_collisions": 0,
                      "avg_detection_time_ms": 0.0, "max_detection_time_ms": 0.0}
        self._counted: Set[Tuple] = set()

    # -- updates (collision_detection.py:74-108) ----------------------------------------------
    def update_vehicle(self, vehicle: Vehicle) -> None:
        self.vehicle_cache[vehicle.id] = vehicle
        idx = self.spatial_index
        idx.vehicle_positions[vehicle.id] = vehicle.position
        p, v, a = vehicle.position, vehicle.velocity, vehicle.acceleration
        idx._table.set_state(vehicle.id, (p.x, p.y, p.z), (v.x, v.y, v.z), (a.x, a.y, a.z), vehicle.heading,
                             vehicle.size, vehicle.type)
        idx.stats["total_vehicles"] = len(idx.vehicle_positions)

    def update_vehicles_batch(self, vehicles) -> None:
        for v in vehicles:
            self.update_vehicle(v)

    @property
    def collision_risks(self) -> Dict[str, Dict[str, CollisionRisk]]:
        """vehicle id -> {other id -> latest CollisionRisk} (collision_detection.py:168-172), brought up to date with
        the detect_collisions results returned since the last read."""
        for vid, risks in self._latest.items():
            self._collision_risks.setdefault(vid, {}).update({r.other_vehicle_id: r for r in risks})
        self._latest.clear()
        return self._collision_risks

    def remove_vehicle(self, vehicle_id: str) -> None:
        self.vehicle_cache.pop(vehicle_id, None)
        self.spatial_index.remove_vehicle(vehicle_id)
        risks_by_vehicle = self.collision_risks
        risks_by_vehicle.pop(vehicle_id, None)
        for risks in risks_by_vehicle.values():
            risks.pop(vehicle_id, None)

    # -- queries --------------------------------------------------------------------------------
    def _frame(self, search_radius: float, time_window: float, slots: Optional[np.ndarray] = None):
        frames = self.spatial_index._frames
        t0 = time.perf_counter()
        ran_before = frames.frames_run
        pairs, starts, counts = frames.run(N.MODE_DETECT, search_radius, time_window, slots=slots)
        if frames.frames_run != ran_before:  # a new frame was computed: fold its totals into the stats
            ms = (time.perf_counter() - t0) * 1e3
            n = max(1, self.spatial_index._table.n)
            self.stats["potential_collisions"] += int(counts["n_potential"])
            self.stats["high_risk_collisions"] += int(counts["n_high_risk"])
            self.stats["max_detection_time_ms"] = max(self.stats["max_detection_time_ms"], ms / n)
            self._frame_ms_per_vehicle = ms / n
        return pairs, starts, counts

    def detect_collisions(self, vehicle_id: str, search_radius: float = 100.0, time_window: float = 10.0) -> List[CollisionRisk]:
        if vehicle_id not in self.vehicle_cache:
            return []
        table = self.spatial_index._table
        pairs, starts, _counts = self._frame(search_radius, time_window)
        s = table.slot_of[vehicle_id]
        risks = _risks_from_pairs(pairs[starts[s]:starts[s + 1]], table.ids, f"d{self.spatial_index._frames.frames_run:x}-{s:x}")
        if risks:
            if vehicle_id in self._latest:  # an older unread result: fold it in first (later results win per other id)
                _ = self.collision_risks
            self._latest[vehicle_id] = risks
        self.stats["total_detections"] += 1
        k = self.stats["total_detections"]
        ms = getattr(self, "_frame_ms_per_vehicle", 0.0)
        self.stats["avg_detection_time_ms"] = (self.stats["avg_detection_time_ms"] * (k - 1) + ms) / k
        return risks

    def detect_all(self, search_radius: float = 100.0, time_window: float = 10.0) -> Dict[str, List[CollisionRisk]]:
        """Additive batch API: every vehicle's risks from one GPU frame."""
        table = self.spatial_index._table
        if table.n == 0:
            return {}
        pairs, starts, _ = self._frame(search_radius, time_window)
        out: Dict[str, List[CollisionRisk]] = {}
        tag = f"d{self.spatial_index._frames.frames_run:x}"
        for s in np.flatnonzero(np.diff(starts)):
            out[table.ids[int(s)]] = _risks_from_pairs(pairs[starts[s]:starts[s + 1]], table.ids, f"{tag}-{int(s):x}")
        return out

    def detect_for(self, vehicle_ids, search_radius: float = 100.0, time_window: float = 10.0) -> Dict[str, List[CollisionRisk]]:
        """Additive batch API: the risks of the listed vehicles only, keyed like ``detect_all`` (vehicles without a
        risk are left out); unknown ids are skipped.  A whole frame memoised with the same parameters answers
        without GPU work; otherwise one GPU frame queries just these vehicles (every vehicle stays a neighbour) --
        the partitioned queries of CollisionDetectionSystem._process_shard (collision_system.py:423-459)."""
        return _rows_for(self.spatial_index, vehicle_ids, "d",
                         lambda slots: self._frame(search_radius, time_window, slots))

    def get_collision_risks(self, vehicle_id: str) -> List[CollisionRisk]:
        return list(self.collision_risks.get(vehicle_id, {}).values())

    def _spatial_filtering(self, vehicle_id: str, position: Position, search_radius: float) -> Set[str]:
        near = self.spatial_index.get_nearby_vehicles(position, search_radius)
        near.discard(vehicle_id)
        return near

    def _predict_position(self, vehicle: Vehicle, time_delta: float) -> Position:
        p, v, a, t = vehicle.position, vehicle.velocity, vehicle.acceleration, time_delta
        return Position(x=p.x + v.x * t + 0.5 * a.x * t * t, y=p.y + v.y * t + 0.5 * a.y * t * t,
                        z=p.z + v.z * t + 0.5 * a.z * t * t)

    def _calculate_safe_distance(self, vehicle1: Vehicle, vehicle2: Vehicle) -> float:
        return (vehicle1.size + vehicle2.size) / 2 + SAFE_DISTANCE_DEFAULT

    # -- the per-pair helpers the prediction model calls on the detector (collision_detection.py:821-830) ----
    def _object_record(self, vehicle: Vehicle) -> np.ndarray:
        o = np.zeros(1, dtype=N.OBJECT_DTYPE)
        p, v, a = vehicle.position, vehicle.velocity, vehicle.acceleration
        o[0] = (p.x, p.y, p.z, v.x, v.y, v.z, a.x, a.y, a.z, vehicle.size, vehicle.heading,
                self.spatial_index._table.type_code(vehicle.type))
        return o

    def _engine(self):
        frames = self.spatial_index._frames
        frames._ensure_engine()
        return frames.engine

    def _precise_collision_detection(self, vehicle: Vehicle, other_vehicle: Vehicle, time_window: float,
                                     time_step: float = 0.1) -> Optional[Dict[str, Any]]:
        """:296-342 for one pair, evaluated by the device function the frame kernels use (rcd_pair_exact): first
        sample t = k * time_step, k < int(time_window / time_step), with distance <= safe distance."""
        r = self._engine().pair_exact(self._object_record(vehicle), self._object_record(other_vehicle), time_window, time_step)[0]
        if not r["hit"]:
            return None
        return {"collision_time": float(r["collision_time"]),
                "collision_position": Position(float(r["cx"]), float(r["cy"]), float(r["cz"])),
                "distance": float(r["distance"]), "safe_distance": float(r["safe_distance"]),
                "relative_speed": float(r["relative_speed"])}

    def _risk_assessment(self, vehicle: Vehicle, other_vehicle: Vehicle, collision_info: Dict[str, Any]) -> float:
        """:344-389 (+ _get_type_factor :498-513) for one collision_info, on the device (rcd_risk_assessment)."""
        rec = np.array([[vehicle.heading, other_vehicle.heading, 1.0 if vehicle.type == other_vehicle.type else 0.0,
                         collision_info["collision_time"], collision_info["distance"], collision_info["safe_distance"],
                         collision_info.get("relative_speed", 0.0)]], np.float64)
        return float(self._engine().risk_assessment(rec)[0])

    def get_stats(self) -> Dict[str, Any]:
        return self.stats


class CollisionPredictionModel:
    """Trajectory histories live twice: in ``trajectory_history`` (the reference's public attribute)
    and in ring buffers on the GPU (rcd_history_*), which are fed incrementally, so classifying every
    vehicle each frame costs one kernel instead of re-staging up to 100 samples per vehicle.  Both keep
    the last 100 samples in arrival order; the classifier sorts them by timestamp, like the reference (:638)."""

    def __init__(self, collision_detector: CollisionDetector):
        self.collision_detector = collision_detector
        self.max_history_length = 100
        self.prediction_horizon = 10.0
        self.prediction_step = 0.5
        self.trajectory_history: Dict[str, List[Tuple[Position, float]]] = {}
        self.stats = {"total_predictions": 0, "avg_prediction_time_ms": 0.0}
        self._hist_version = 0
        self._pattern_key = None
        self._patterns: Optional[np.ndarray] = None
        # device rings
        self._pending: List[Tuple[str, float, float, float, float]] = []
        self._events_seen = 0
        self._ring_generation = -1

    def update_trajectory(self, vehicle_id: str, position: Position, timestamp: float) -> None:
        h = self.trajectory_history.setdefault(vehicle_id, [])
        h.append((position, timestamp))
        if len(h) > self.max_history_length:
            self.trajectory_history[vehicle_id] = h[-self.max_history_length:]
        self._pending.append((vehicle_id, position.x, position.y, position.z, timestamp))
        self._hist_version += 1

    # -- device rings ------------------------------------------------------------------------------
    def _append_rounds(self, engine, samples_by_slot: Dict[int, List[Tuple[float, float, float, float]]]) -> None:
        """rcd_history_append takes one sample per slot and call: r-th samples go in round r."""
        r = 0
        while True:
            batch = [(s, v[r]) for s, v in samples_by_slot.items() if len(v) > r]
            if not batch:
                break
            arr = np.array([b[1] for b in batch], np.float64).reshape(-1, 4)
            engine.history_append(np.array([b[0] for b in batch], np.uint32), arr[:, 0], arr[:, 1], arr[:, 2], arr[:, 3])
            r += 1

    def _sync_rings(self, frames) -> None:
        table = self.collision_detector.spatial_index._table
        engine = frames.engine
        if self._ring_generation != frames.engine_generation:
            # a new handle: rebuild every ring from the host copies
            engine.history_configure(self.max_history_length)
            seed = {s: [(p.x, p.y, p.z, t) for p, t in self.trajectory_history.get(table.ids[s], [])]
                    for s in range(table.n)}
            self._append_rounds(engine, {s: v for s, v in seed.items() if v})
            self._ring_generation = frames.engine_generation
            self._events_seen = len(table.events)
            self._pending.clear()
            return
        reseed = set()
        for ev in table.events[self._events_seen:]:
            if ev[0] == "move":
                dst, src = ev[1], ev[2]
                if src in reseed:  # the moved vehicle is itself new: its ring is rebuilt at the new slot, never copied
                    reseed.discard(src)
                    reseed.add(dst)
                else:
                    engine.history_move(dst, src)
                    reseed.discard(dst)  # whatever was pending for the slot's previous occupant is void
            else:  # a (possibly recycled) slot got a new vehicle
                reseed.add(ev[1])
        self._events_seen = len(table.events)
        by_slot: Dict[int, List[Tuple[float, float, float, float]]] = {}
        if reseed:
            live = [s for s in reseed if s < table.n]
            if live:
                engine.history_reset(np.array(live, np.uint32))
            for s in live:  # the reference keeps a removed vehicle's history: it continues on re-insertion
                hist = self.trajectory_history.get(table.ids[s], [])
                if hist:
                    by_slot[s] = [(p.x, p.y, p.z, t) for p, t in hist]
        reseeded_ids = {table.ids[s] for s in by_slot}
        for vid, x, y, z, t in self._pending:
            s = table.slot_of.get(vid)
            if s is not None and vid not in reseeded_ids:
                by_slot.setdefault(s, []).append((x, y, z, t))
        self._pending.clear()
        self._append_rounds(engine, by_slot)

    def _classify_on_device(self, frames) -> None:
        table = self.collision_detector.spatial_index._table
        key = (self._hist_version, table.version, frames.engine_generation)
        if key != self._pattern_key or frames._flags_uploaded != key:
            self._sync_rings(frames)
            self._patterns = frames.engine.history_classify(want_codes=True)
            self._pattern_key = key
            frames.flags_set_on_device(key)

    def trajectory_patterns(self) -> np.ndarray:
        """Pattern code of every indexed vehicle (collision_detection.py:623-711), classified on the
        GPU; 3 = fewer than 2 samples (-> detect path, :590-592)."""
        frames = self.collision_detector.spatial_index._frames
        table = self.collision_detector.spatial_index._table
        if table.n == 0:
            return np.zeros(0, np.uint8)
        frames.sync_objects()
        self._classify_on_device(frames)
        return self._patterns

    def _frame(self, slots: Optional[np.ndarray] = None):
        frames = self.collision_detector.spatial_index._frames
        return frames.run(N.MODE_PREDICT, 100.0, 10.0, prepare=self._classify_on_device, slots=slots)

    def predict_collisions(self, vehicle_id: str) -> List[CollisionRisk]:
        det = self.collision_detector
        if vehicle_id not in det.vehicle_cache:
            return []
        table = det.spatial_index._table
        t0 = time.perf_counter()
        pairs, starts, _ = self._frame()
        s = table.slot_of[vehicle_id]
        risks = _risks_from_pairs(pairs[starts[s]:starts[s + 1]], table.ids,
                                  f"p{det.spatial_index._frames.frames_run:x}-{s:x}")
        self.stats["total_predictions"] += 1
        k = self.stats["total_predictions"]
        ms = (time.perf_counter() - t0) * 1e3
        self.stats["avg_prediction_time_ms"] = (self.stats["avg_prediction_time_ms"] * (k - 1) + ms) / k
        return risks

    def predict_all(self) -> Dict[str, List[CollisionRisk]]:
        table = self.collision_detector.spatial_index._table
        if table.n == 0:
            return {}
        pairs, starts, _ = self._frame()
        out: Dict[str, List[CollisionRisk]] = {}
        tag = f"p{self.collision_detector.spatial_index._frames.frames_run:x}"
        for s in np.flatnonzero(np.diff(starts)):
            out[table.ids[int(s)]] = _risks_from_pairs(pairs[starts[s]:starts[s + 1]], table.ids, f"{tag}-{int(s):x}")
        return out

    def predict_for(self, vehicle_ids) -> Dict[str, List[CollisionRisk]]:
        """``predict_all`` for the listed vehicles only (see ``CollisionDetector.detect_for``)."""
        return _rows_for(self.collision_detector.spatial_index, vehicle_ids, "p", self._frame)

    def get_stats(self) -> Dict[str, Any]:
        return {**self.stats, "trajectory_history_count": len(self.trajectory_history)}
