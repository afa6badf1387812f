"""Host-side staging of per-vehicle API calls into the SoA frame the GPU consumes.

The reference API is per vehicle and string keyed (update_vehicle(Vehicle), insert(id, Position));
the GPU works on whole frames.  ``ObjectTable`` keeps an id <-> dense slot map and fp32 SoA
arrays so that every per-vehicle call is O(1); ``FrameCache`` uploads the table when it changed
and memoises whole-frame results, so N per-vehicle queries cost one GPU frame.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import numpy as np

from . import _native as N
from .engine import FRAME_FIELDS, FrameEngine


class ObjectTable:
    def __init__(self, capacity: int = 1024):
        self.capacity = int(capacity)
        self.n = 0
        self.ids: List[str] = []
        self.slot_of: Dict[str, int] = {}
        self.f = {k: np.zeros(self.capacity, np.float32) for k in FRAME_FIELDS}
        self.type = np.zeros(self.capacity, np.uint8)
        self.flag = np.full(self.capacity, 2, np.uint8)  # pattern code / has-history flag
        self.type_codes: Dict[str, int] = {}
        self.version = 0
        # slot events since the table was created: ("new", slot, id) / ("move", dst, src); consumers
        # (the device-resident trajectory rings) keep their own read position
        self.events: List[Tuple] = []

    def _grow(self):
        self.capacity *= 2
        for k in FRAME_FIELDS:
            self.f[k] = np.concatenate([self.f[k], np.zeros_like(self.f[k])])
        self.type = np.concatenate([self.type, np.zeros_like(self.type)])
        self.flag = np.concatenate([self.flag, np.full_like(self.flag, 2)])

    def type_code(self, name: Optional[str]) -> int:
        code = self.type_codes.get(name)
        if code is None:
            code = len(self.type_codes)
            if code > 255:
                raise ValueError("more than 256 distinct vehicle types")
            self.type_codes[name] = code
        return code

    def slot(self, vid: str) -> int:
        s = self.slot_of.get(vid)
        if s is None:
            if self.n == self.capacity:
                self._grow()
            s = self.n
            self.n += 1
            self.ids.append(vid)
            self.slot_of[vid] = s
            for k in FRAME_FIELDS:
                self.f[k][s] = 0.0
            self.type[s] = 0
            self.flag[s] = 2
            self.events.append(("new", s, vid))
        return s

    def set_position(self, vid: str, x: float, y: float, z: float) -> int:
        s = self.slot(vid)
        self.f["px"][s], self.f["py"][s], self.f["pz"][s] = x, y, z
        self.version += 1
        return s

    def set_state(self, vid: str, p, v, a, heading: float, size: float, type_name: Optional[str]) -> int:
        s = self.slot(vid)
        f = self.f
        f["px"][s], f["py"][s], f["pz"][s] = p
        f["vx"][s], f["vy"][s], f["vz"][s] = v
        f["ax"][s], f["ay"][s], f["az"][s] = a
        f["heading"][s], f["size"][s] = heading, size
        self.type[s] = self.type_code(type_name)
        self.version += 1
        return s

    def remove(self, vid: str) -> bool:
        s = self.slot_of.pop(vid, None)
        if s is None:
            return False
        last = self.n - 1
        if s != last:  # keep the table dense: move the last object into the hole
            moved = self.ids[last]
            for k in FRAME_FIELDS:
                self.f[k][s] = self.f[k][last]
            self.type[s] = self.type[last]
            self.flag[s] = self.flag[last]
            self.ids[s] = moved
            self.slot_of[moved] = s
            self.events.append(("move", s, last))
        self.ids.pop()
        self.n = last
        self.version += 1
        return True

    def frame(self) -> Dict[str, np.ndarray]:
        out = {k: self.f[k][: self.n] for k in FRAME_FIELDS}
        out["type"] = self.type[: self.n]
        return out


class FrameCache:
    """Lazy whole-frame evaluation on the GPU for one ObjectTable."""

    def __init__(self, table: ObjectTable, device: int = 0):
        self.table = table
        self.device = device
        self.engine: Optional[FrameEngine] = None
        self._uploaded = -1
        self._flags_uploaded = None
        self._results: Dict[Tuple, Tuple[np.ndarray, np.ndarray, Dict]] = {}
        self.frames_run = 0
        self.engine_generation = 0  # bumps whenever a new handle replaces the old one (device state is lost)

    def _ensure_engine(self):
        need = max(self.table.n, 1)
        if self.engine is None or self.engine.max_objects < need:
            if self.engine is not None:
                self.engine.close()
            cap = max(1024, 2 * need)
            self.engine = FrameEngine(cap, max_pairs=max(1 << 16, 32 * cap), device=self.device)
            self.engine_generation += 1
            self._uploaded = -1

    def sync_objects(self, flags: Optional[np.ndarray] = None):
        self._ensure_engine()
        t = self.table
        if self._uploaded != t.version:
            self.engine.upload(t.frame())
            self._uploaded = t.version
            self._results.clear()
            self._flags_uploaded = None
        if flags is not None:
            key = flags.tobytes()
            if key != self._flags_uploaded:
                self.engine.set_patterns(flags)
                self._flags_uploaded = key
                self._results.clear()

    def flags_set_on_device(self, key) -> None:
        """The per-object flags were written on the device (rcd_history_classify): remember which
        version they belong to and drop memoised frames if they changed."""
        if key != self._flags_uploaded:
            self._flags_uploaded = key
            self._results.clear()

    def run(self, mode: int, radius: float = 100.0, window: float = 10.0, flags: Optional[np.ndarray] = None,
            prepare=None, slots: Optional[np.ndarray] = None):
        """(pairs sorted by slot i, CSR starts per slot, counts) of one frame, memoised until the
        objects change.  `prepare(cache)` runs after the objects are on the device and again whenever
        the handle had to be replaced (it sets device-side flags).  `slots` (sorted, unique uint32):
        only these objects need their rows -- a memoised whole frame answers, else one frame queries
        just them (rcd_set_queries; its counts are the totals over the slots), memoised per set."""
        self.sync_objects(flags)
        if prepare is not None:
            prepare(self)
        key = (mode, float(radius), float(window))
        hit = self._results.get(key)
        if hit is None and slots is not None:
            key += (slots.tobytes(),)
            hit = self._results.get(key)
        if hit is not None:
            return hit
        eng = self.engine
        eng.set_queries(slots)
        eng.step(mode, radius, window)
        while True:
            counts = eng.counts()
            if counts["n_pairs"] <= eng.max_pairs:
                break
            # the pair buffer overflowed: grow it and run the frame again (counts stay exact)
            self.engine.close()
            cap = self.engine.max_objects
            self.engine = FrameEngine(cap, max_pairs=int(counts["n_pairs"] * 1.5) + 1024, device=self.device)
            self.engine_generation += 1
            self._uploaded = -1
            self._flags_uploaded = None
            self.sync_objects(flags)
            if prepare is not None:
                prepare(self)
            eng = self.engine
            eng.set_queries(slots)
            eng.step(mode, radius, window)
        pairs = eng.download()
        starts = np.searchsorted(pairs["i"], np.arange(self.table.n + 1, dtype=np.uint32), side="left")
        self.frames_run += 1
        res = (pairs, starts, counts)
        self._results[key] = res
        return res

    def close(self):
        if self.engine is not None:
            self.engine.close()
            self.engine = None
