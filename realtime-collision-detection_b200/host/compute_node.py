"""Drop-in for the three hot-path classes of src/compute/compute_node.py:20-321 (surface B):
``SpatialIndex`` (uniform grid, cell 10 m), ``VehicleState`` and ``CollisionDetector``.

``SpatialIndex.query_nearby`` and ``CollisionDetector.detect_collisions`` run on the GPU
(RCD_MODE_COMPUTE_NODE / rcd_query_radius); ``detect_collisions_for_all`` is the additive batch
form of ComputeNode._detect_collisions_for_all (:592-642).
"""
from __future__ import annotations

import time
from typing import Dict, List, Optional

import numpy as np

from . import _native as N
from .engine import FrameEngine
from .models import ComputeNodeCollisionRisk as CollisionRisk
from .models import LocationData, Position, Vector
from .object_table import FrameCache, ObjectTable


class SpatialIndex:
    def __init__(self, cell_size: float = 10.0, device: int = 0):
        self.cell_size = cell_size
        self.positions: Dict[str, Position] = {}
        self._table = ObjectTable()
        self._frames = FrameCache(self._table, device)

    def _get_cell(self, position: Position):
        cs = self.cell_size
        return (int(position.x / cs), int(position.y / cs), int(position.z / cs))

    def insert(self, vehicle_id: str, position: Position):
        self.positions[vehicle_id] = position
        self._table.set_position(vehicle_id, position.x, position.y, position.z)

    def remove(self, vehicle_id: str) -> bool:
        if vehicle_id not in self.positions:
            return False
        del self.positions[vehicle_id]
        self._table.remove(vehicle_id)
        return True

    def query_nearby(self, position: Position, radius: float) -> List[str]:
        if self._table.n == 0:
            return []
        self._frames.sync_objects()
        hits = self._frames.engine.query_radius([(position.x, position.y, position.z)], radius)[0]
        ids = self._table.ids
        return [ids[int(s)] for s in hits]

    def get_position(self, vehicle_id: str) -> Optional[Position]:
        return self.positions.get(vehicle_id)

    def get_all_vehicles(self) -> List[str]:
        return list(self.positions.keys())

    def get_vehicle_count(self) -> int:
        return len(self.positions)


class VehicleState:
    """compute_node.py:152-212 (host bookkeeping only)."""

    def __init__(self, vehicle_id: str, max_history: int = 10):
        self.vehicle_id = vehicle_id
        self.max_history = max_history
        self.history: List[LocationData] = []
        self.last_update = 0

    def update(self, location_data: LocationData):
        self.history.append(location_data)
        if len(self.history) > self.max_history:
            self.history.pop(0)
        self.last_update = time.time()

    def get_current_location(self) -> Optional[LocationData]:
        return self.history[-1] if self.history else None

    def predict_position(self, time_delta: float) -> Optional[Position]:
        if len(self.history) < 2:
            return None
        c = self.history[-1]
        return Position(x=c.position.x + c.velocity.x * time_delta, y=c.position.y + c.velocity.y * time_delta,
                        z=c.position.z + c.velocity.z * time_delta)


def _stage(states: List[VehicleState]):
    n = len(states)
    f = {k: np.zeros(n, np.float32) for k in ("px", "py", "pz", "vx", "vy", "vz", "ax", "ay", "az", "size", "heading")}
    f["type"] = np.zeros(n, np.uint8)
    hist = np.zeros(n, np.uint8)
    for k, st in enumerate(states):
        loc = st.get_current_location()
        f["px"][k], f["py"][k], f["pz"][k] = loc.position.x, loc.position.y, loc.position.z
        f["vx"][k], f["vy"][k], f["vz"][k] = loc.velocity.x, loc.velocity.y, loc.velocity.z
        f["heading"][k] = loc.heading
        hist[k] = 1 if len(st.history) >= 2 else 0
    return f, hist


def _risks(pairs: np.ndarray, ids: List[str]) -> List[CollisionRisk]:
    now = time.time()
    return [CollisionRisk.create(vehicle_id1=ids[int(r["i"])], vehicle_id2=ids[int(r["j"])], risk_level=float(r["risk"]),
                                 estimated_collision_time=now + float(r["ttc"]),
                                 position=Position(float(r["cx"]), float(r["cy"]), float(r["cz"])),
                                 relative_velocity=float(r["rel_speed"])) for r in pairs]


class CollisionDetector:
    def __init__(self, prediction_time: float = 5.0, risk_threshold: float = 0.5, device: int = 0):
        self.prediction_time = prediction_time
        self.risk_threshold = risk_threshold
        self.device = device
        self._engine: Optional[FrameEngine] = None

    def _eng(self, n: int) -> FrameEngine:
        cap = max(1024, 2 * n)
        if self._engine is None:
            self._engine = FrameEngine(cap, device=self.device)
            self._engine.set_compute_node_params(self.prediction_time, self.risk_threshold)
        elif self._engine.max_objects < n:  # grow in place (the parameters stay), FrameEngine's default pair buffer
            self._engine.reserve(cap, max(4096, 16 * cap))
        return self._engine

    def detect_collisions(self, vehicle: VehicleState, nearby_vehicles: Dict[str, VehicleState]) -> List[CollisionRisk]:
        """compute_node.py:229-321 for one vehicle against an explicit neighbour set: the vehicle
        and its neighbours are staged as one small frame in which only the vehicle is queried."""
        if not vehicle.get_current_location():
            return []
        others = [(oid, st) for oid, st in nearby_vehicles.items()
                  if oid != vehicle.vehicle_id and st.get_current_location()]
        states = [vehicle] + [st for _, st in others]
        ids = [vehicle.vehicle_id] + [oid for oid, _ in others]
        frame, hist = _stage(states)
        eng = self._eng(len(states))
        eng.upload(frame)
        eng.set_patterns(hist)
        eng.set_owned(1)
        # every listed neighbour is a candidate (the caller already applied its search radius);
        # the pair function itself drops pairs farther apart than 50 m (:262)
        return _risks(eng.compute_node(search_radius=1.0e9), ids)

    def detect_collisions_for_all(self, states: Dict[str, VehicleState], search_radius: float = 100.0) -> Dict[str, List[CollisionRisk]]:
        """Batch form of ComputeNode._detect_collisions_for_all (:592-642): query_nearby(search_radius)
        + detect_collisions for every vehicle with a location, in one GPU frame."""
        live = [(vid, st) for vid, st in states.items() if st.get_current_location()]
        if not live:
            return {}
        ids = [vid for vid, _ in live]
        frame, hist = _stage([st for _, st in live])
        eng = self._eng(len(live))
        eng.upload(frame)
        eng.set_patterns(hist)
        out: Dict[str, List[CollisionRisk]] = {}
        for r in _risks(eng.compute_node(search_radius=search_radius), ids):
            out.setdefault(r.vehicle_id1, []).append(r)
        return out
