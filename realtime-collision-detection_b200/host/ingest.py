"""Batched ingest of the reference's vehicle wire format (SURVEY.md 8f rank 2).

The reference handles one broker message at a time: ``json.loads`` -> dict ->
``EarlyWarningSystem._handle_vehicle_position`` builds a ``Vehicle`` and calls
``CollisionDetector.update_vehicle`` + ``CollisionPredictionModel.update_trajectory``
(src/collision/warning_system.py:638-678; producer src/test/vehicle_simulator.py:721-752).
``VehicleIngest`` takes whole buffers of those messages instead: the native decoder
(csrc/rcd_ingest.hpp) turns them into fixed records and interns ids / types, and
``FrameEngine.apply_records`` scatters the records into the device-resident frame state and
trajectory rings (csrc/rcd_ingest.cuh).
"""
from __future__ import annotations

import ctypes
from typing import List, Optional, Tuple, Union

import numpy as np

from . import _native as N


class VehicleIngest:
    """Decoder + id table.  A new vehicle id takes the lowest released slot (``release``), else the next fresh one:
    without releases, slot ``k`` of the frame is the k-th distinct vehicle id ever seen."""

    def __init__(self, threads: int = 0):
        self._lib = N.load()
        self._g = ctypes.c_void_p()
        self.threads = int(threads)
        rc = self._lib.rcd_ingest_create(ctypes.byref(self._g))
        if rc != N.RCD_OK:
            raise N.NativeError(rc, "rcd_ingest_create")
        self.bad_messages = 0

    def close(self) -> None:
        if getattr(self, "_g", None) is not None and self._g:
            self._lib.rcd_ingest_destroy(self._g)
            self._g = ctypes.c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc: int) -> None:
        if rc != N.RCD_OK:
            msg = self._lib.rcd_ingest_last_error(self._g)
            raise N.NativeError(rc, msg.decode("utf-8", "replace") if msg else "")

    # -- decode -----------------------------------------------------------------------------
    def decode(self, data: Union[bytes, bytearray, memoryview, str], out: Optional[np.ndarray] = None
               ) -> Tuple[np.ndarray, int]:
        """Decode every message in ``data``; returns (records, max_seq).  Malformed / incomplete
        messages are dropped and counted in ``bad_messages`` (the reference logs and drops them)."""
        if isinstance(data, str):
            data = data.encode("utf-8")
        buf = (ctypes.c_char * len(data)).from_buffer_copy(data) if not isinstance(data, bytes) else data
        n_bytes = len(data)
        # a message of the reference format is > 150 bytes; 64 is a safe lower bound per record
        cap = max(16, n_bytes // 64 + 1) if out is None else int(out.shape[0])
        rec = np.empty(cap, dtype=N.RECORD_DTYPE) if out is None else out
        n, bad, mseq = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint32()
        ptr = ctypes.cast(buf, ctypes.c_void_p) if isinstance(buf, bytes) else ctypes.cast(ctypes.addressof(buf), ctypes.c_void_p)
        rc = self._lib.rcd_ingest_decode_json(self._g, ptr, n_bytes, self.threads, rec.ctypes.data_as(ctypes.c_void_p), cap,
                                              ctypes.byref(n), ctypes.byref(bad), ctypes.byref(mseq))
        if rc == N.RCD_ECAPACITY and out is None and int(n.value) > cap:
            # more (tiny) messages than the estimate: nothing was decoded and no state changed -- once more, with room
            cap = int(n.value)
            rec = np.empty(cap, dtype=N.RECORD_DTYPE)
            rc = self._lib.rcd_ingest_decode_json(self._g, ptr, n_bytes, self.threads, rec.ctypes.data_as(ctypes.c_void_p),
                                                  cap, ctypes.byref(n), ctypes.byref(bad), ctypes.byref(mseq))
        self._check(rc)
        self.bad_messages += int(bad.value)
        return rec[: int(n.value)], int(mseq.value)

    # -- id / type tables -------------------------------------------------------------------
    def set_limit(self, max_ids: int) -> None:
        """At most ``max_ids`` distinct vehicles: messages of further (unknown) vehicles are dropped and counted
        (``bad_messages``, ``rejected``) while the known ones keep being served."""
        self._check(self._lib.rcd_ingest_set_limit(self._g, int(max_ids)))

    def release(self, slots) -> int:
        """Forget the ids of the listed slots (retired vehicles): new ids take them, lowest first, and the id limit
        counts live ids.  ``n_objects`` (slots handed out) does not change.  Returns the number of live ids."""
        s = np.ascontiguousarray(slots, dtype=np.uint32)
        live = ctypes.c_uint64()
        self._check(self._lib.rcd_ingest_release(self._g, int(s.shape[0]), s.ctypes.data_as(ctypes.c_void_p) if s.shape[0]
                                                 else None, ctypes.byref(live)))
        return int(live.value)

    @property
    def rejected(self) -> int:
        n = ctypes.c_uint64()
        self._check(self._lib.rcd_ingest_rejected(self._g, ctypes.byref(n)))
        return int(n.value)

    @property
    def n_objects(self) -> int:
        n = ctypes.c_uint64()
        self._check(self._lib.rcd_ingest_counts(self._g, ctypes.byref(n), None))
        return int(n.value)

    @property
    def n_types(self) -> int:
        n = ctypes.c_uint64()
        self._check(self._lib.rcd_ingest_counts(self._g, None, ctypes.byref(n)))
        return int(n.value)

    def id_of(self, slot: int) -> str:
        p, ln = ctypes.c_char_p(), ctypes.c_uint32()
        self._check(self._lib.rcd_ingest_id_name(self._g, int(slot), ctypes.byref(p), ctypes.byref(ln)))
        return ctypes.string_at(p, ln.value).decode("utf-8", "surrogatepass")

    def type_of(self, code: int) -> str:
        p, ln = ctypes.c_char_p(), ctypes.c_uint32()
        self._check(self._lib.rcd_ingest_type_name(self._g, int(code), ctypes.byref(p), ctypes.byref(ln)))
        return ctypes.string_at(p, ln.value).decode("utf-8", "surrogatepass")

    def slot_of(self, vehicle_id: str) -> Optional[int]:
        b = vehicle_id.encode("utf-8", "surrogatepass")
        s = ctypes.c_uint32()
        rc = self._lib.rcd_ingest_lookup(self._g, b, len(b), ctypes.byref(s))
        if rc == N.RCD_ESTATE:
            return None
        self._check(rc)
        return int(s.value)

    def ids(self) -> List[str]:
        return [self.id_of(k) for k in range(self.n_objects)]


class VehiclePositionStream:
    """Batched counterpart of ``EarlyWarningSystem._handle_vehicle_position`` +
    ``_detect_all_vehicles`` (src/collision/warning_system.py:638-714): message buffers in,
    one GPU frame for every vehicle out.  Object state and trajectory rings stay on the device;
    the host keeps only the id table."""

    def __init__(self, max_objects: int, max_pairs: Optional[int] = None, world_bounds=None, device: int = 0,
                 threads: int = 0, max_history: int = 100):
        from .engine import FrameEngine
        self.engine = FrameEngine(max_objects, max_pairs, device=device, world_bounds=world_bounds)
        self.engine.history_configure(max_history)
        self.ingest = VehicleIngest(threads=threads)
        self.ingest.set_limit(max_objects)  # a full frame rejects new vehicles, it does not fail every later batch
        self.messages_applied = 0

    def close(self) -> None:
        self.ingest.close()
        self.engine.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def reserve(self, max_objects: Optional[int] = None, max_pairs: Optional[int] = None,
                max_alerts: Optional[int] = None) -> None:
        """Grow the frame (vehicles, pair buffer) and the alert table in place: every ring, record time and live alert
        stays on the device.  The ingest id limit follows ``max_objects``, so new vehicles are taken again."""
        self.engine.reserve(max_objects, max_pairs)
        if max_alerts is not None:
            self.engine.alerts_reserve(max_alerts)
        self.ingest.set_limit(self.engine.max_objects)

    def handle_messages(self, data) -> int:
        """Decode and apply a buffer of vehicle messages; returns how many were applied."""
        rec, max_seq = self.ingest.decode(data)
        if len(rec):
            self.engine.apply_records(rec, self.ingest.n_objects, max_seq, history=True)
            self.messages_applied += len(rec)
        return len(rec)

    def _retired(self, slots: np.ndarray, events: np.ndarray, alerts) -> List[str]:
        # the alert manager drops the events while id_of still names the departed vehicles; then the slots are freed
        ids = [self.ingest.id_of(int(k)) for k in slots]
        if alerts is not None:
            alerts.retire_vehicles(events, ids)
        if len(slots):
            self.ingest.release(slots)
        return ids

    def remove_vehicles(self, ids, alerts=None) -> List[str]:
        """``remove_vehicle`` for the listed vehicle ids (unknown ids are skipped): their slots stop taking part in
        frames and are handed to the next new vehicles.  ``alerts``: the ``AlertManager`` attached to this engine,
        whose alerts of the departed vehicles are dropped too.  Returns the ids that were removed."""
        slots = sorted({s for s in (self.ingest.slot_of(v) for v in ids) if s is not None})
        _, ev, _ = self.engine.retire(np.asarray(slots, np.uint32))
        return self._retired(np.asarray(slots, np.uint32), ev, alerts)

    def retire_stale(self, now: float, max_age: float, alerts=None) -> List[str]:
        """Remove every vehicle whose newest message is older than ``max_age`` at ``now`` (now - timestamp >
        max_age); returns their ids in slot order."""
        slots, ev, _ = self.engine.retire_stale(now, max_age)
        return self._retired(slots, ev, alerts)

    def detect_all_vehicles(self, predict: bool = True) -> np.ndarray:
        """``predict_collisions`` (or ``detect_collisions``) for every vehicle: pairs with i / j = slots
        (``ingest.id_of``), sorted by (i, j)."""
        if self.engine.n == 0:
            return np.zeros(0, dtype=N.PAIR_DTYPE)
        if predict:
            self.engine.history_classify(want_codes=False)
            return self.engine.predict()
        return self.engine.detect()
