"""Alert part of src/collision/warning_system.py (SURVEY.md 8a a14, 8f rank 3): the alert gate, priority
tiers, message tiers and the alert table, with the reference's attribute shapes and method names
(``AlertManager``, :48-517) so that callers -- and anything that logs or matches alert messages --
see the same objects and the same bytes.

Two ways to feed it:
  * ``process_collision_risks(risks)`` -- the reference's per-risk walk (:259-285), for risks that are
    already on the host;
  * ``attach_engine`` + ``process_frame`` -- the alert table lives on the GPU next to the frames
    (csrc/rcd_alerts.cuh), a frame's risks are folded in without leaving the device and only the changes
    (created alerts, priority changes, expiries) come back; the host dicts are updated from those events.
Queueing to the broker, resend loops and the asyncio plumbing are out of scope (I/O glue).
"""
from __future__ import annotations

import heapq
import time
import uuid
from typing import Any, Callable, Dict, List, Optional, Tuple

from .models import AlertInfo, CollisionRisk

RISK_LEVEL_LOW = 0.3
RISK_LEVEL_MEDIUM = 0.6
RISK_LEVEL_HIGH = 0.8
PRIORITY_LOW, PRIORITY_MEDIUM, PRIORITY_HIGH, PRIORITY_CRITICAL = 0, 1, 2, 3
ALERT_MAX_AGE = 30.0  # _cleanup_expired_alerts, :497


def alert_message(risk_level: float, other_vehicle_id: str, time_to_collision: float, distance: float) -> str:
    """The message tiers of warning_system.py:313-329, byte for byte (the strings are part of the data
    contract: consumers log and match them)."""
    if risk_level >= RISK_LEVEL_HIGH:
        return (f"紧急警告：与车辆 {other_vehicle_id} 可能在 {time_to_collision:.1f} 秒后发生碰撞，"
                f"当前距离 {distance:.1f} 米，请立即采取避让措施！")
    if risk_level >= RISK_LEVEL_MEDIUM:
        return (f"警告：与车辆 {other_vehicle_id} 可能在 {time_to_collision:.1f} 秒后发生碰撞，"
                f"当前距离 {distance:.1f} 米，请注意避让。")
    return f"注意：与车辆 {other_vehicle_id} 距离较近（{distance:.1f} 米），请保持安全距离。"


class AlertManager:
    def __init__(self, broker=None):
        self.broker = broker
        self.alerts: Dict[str, AlertInfo] = {}                # alert_id -> AlertInfo (:60)
        self.vehicle_alerts: Dict[str, Dict[str, str]] = {}   # vehicle_id -> {other_id -> alert_id} (:61)
        self._queue: List[AlertInfo] = []                     # alert_queue: heap ordered by AlertInfo.__lt__ (:64)
        self._queue_dirty = False                             # a queued alert changed priority: heapify before use
        self.alert_callbacks: Dict[str, List[Callable]] = {}  # vehicle_id -> [callback, ...] (:67)
        self.stats = {"total_alerts": 0, "active_alerts": 0}
        self._engine = None
        self._id_of = None
        self._index_of = None
        self._by_number: Dict[int, str] = {}  # device alert number -> alert_id

    # -- classification ----------------------------------------------------------------------------
    def _get_priority(self, risk_level: float, time_to_collision: float) -> int:
        """warning_system.py:287-311 (the same thresholds the kernels apply to every pair)."""
        if risk_level >= RISK_LEVEL_HIGH and time_to_collision < 3.0:
            return PRIORITY_CRITICAL
        if risk_level >= RISK_LEVEL_HIGH or time_to_collision < 5.0:
            return PRIORITY_HIGH
        if risk_level >= RISK_LEVEL_MEDIUM:
            return PRIORITY_MEDIUM
        return PRIORITY_LOW

    def _generate_alert_message(self, risk: CollisionRisk) -> str:
        return alert_message(risk.risk_level, risk.other_vehicle_id, risk.time_to_collision, risk.distance)

    def _priority_of(self, risk: CollisionRisk) -> int:
        prio = getattr(risk, "alert_priority", -1)  # classified on the GPU together with the pair
        return prio if prio >= 0 else self._get_priority(risk.risk_level, risk.time_to_collision)

    # -- the table (:120-257) ------------------------------------------------------------------------
    def create_alert(self, risk: CollisionRisk) -> AlertInfo:
        alert_info = AlertInfo(id=f"alert-{uuid.uuid4()}", vehicle_id=risk.vehicle_id, other_vehicle_id=risk.other_vehicle_id,
                               risk_level=risk.risk_level, time_to_collision=risk.time_to_collision,
                               message=self._generate_alert_message(risk), priority=self._priority_of(risk),
                               timestamp=time.time())
        self._store(alert_info)
        return alert_info

    def _store(self, alert_info: AlertInfo) -> None:
        self.alerts[alert_info.id] = alert_info
        self.vehicle_alerts.setdefault(alert_info.vehicle_id, {})[alert_info.other_vehicle_id] = alert_info.id
        if self._queue_dirty:
            self._queue.append(alert_info)
        else:
            heapq.heappush(self._queue, alert_info)
        self.stats["total_alerts"] += 1
        self.stats["active_alerts"] = len(self.alerts)

    @property
    def alert_queue(self) -> List[AlertInfo]:
        """The priority queue the sending loop pops from (:64, :219-257).  The reference rebuilds the whole heap for
        every priority change (:186-191: filter, heapify, push -- the same set of alerts afterwards); here a change only
        marks the heap, and it is put in order once, when somebody looks at it."""
        if self._queue_dirty:
            heapq.heapify(self._queue)
            self._queue_dirty = False
        return self._queue

    @alert_queue.setter
    def alert_queue(self, value: List[AlertInfo]) -> None:
        self._queue = value
        self._queue_dirty = False

    def _requeue(self, alert_info: AlertInfo) -> None:
        self._queue_dirty = True  # the alert is queued already (every live alert is): its place is fixed on the next read

    def update_alert(self, risk: CollisionRisk) -> Optional[AlertInfo]:
        alert_id = self.vehicle_alerts.get(risk.vehicle_id, {}).get(risk.other_vehicle_id)
        alert_info = self.alerts.get(alert_id) if alert_id is not None else None
        if alert_info is None:
            return None
        old_priority = alert_info.priority
        alert_info.risk_level = risk.risk_level
        alert_info.time_to_collision = risk.time_to_collision
        alert_info.priority = self._priority_of(risk)
        alert_info.message = self._generate_alert_message(risk)
        alert_info.timestamp = time.time()
        if alert_info.priority != old_priority:  # the queue only hears of priority changes (:186-191)
            self._requeue(alert_info)
        return alert_info

    def acknowledge_alert(self, alert_id: str) -> bool:
        a = self.alerts.get(alert_id)
        if a is None:
            return False
        a.acknowledged = True
        if self._engine is not None and self._index_of is not None:
            i, j = self._index_of(a.vehicle_id), self._index_of(a.other_vehicle_id)
            if i is not None and j is not None:
                self._engine.alerts_acknowledge([i], [j])
        return True

    def get_alerts_for_vehicle(self, vehicle_id: str) -> List[AlertInfo]:
        alerts = [self.alerts[a] for a in self.vehicle_alerts.get(vehicle_id, {}).values() if a in self.alerts]
        return sorted(alerts, key=lambda a: (a.priority, -a.timestamp), reverse=True)

    def register_alert_callback(self, vehicle_id: str, callback: Callable) -> None:
        self.alert_callbacks.setdefault(vehicle_id, []).append(callback)

    def unregister_alert_callback(self, vehicle_id: str, callback: Callable) -> None:
        if vehicle_id in self.alert_callbacks:
            self.alert_callbacks[vehicle_id] = [cb for cb in self.alert_callbacks[vehicle_id] if cb != callback]

    def process_collision_risks(self, risks: List[CollisionRisk]) -> List[AlertInfo]:
        """:259-285: drop risks below RISK_LEVEL_LOW, update the alert of (vehicle, other vehicle) or create it."""
        alerts = []
        for risk in risks:
            if risk.risk_level < RISK_LEVEL_LOW:
                continue
            alert_info = self.update_alert(risk)
            if not alert_info:
                alert_info = self.create_alert(risk)
            alerts.append(alert_info)
        return alerts

    def _drop(self, alert_ids) -> None:
        gone = set()
        for alert_id in alert_ids:
            a = self.alerts.pop(alert_id, None)
            if a is None:
                continue
            gone.add(alert_id)
            self.vehicle_alerts.get(a.vehicle_id, {}).pop(a.other_vehicle_id, None)
        if gone:
            self.alert_queue = [a for a in self.alert_queue if a.id not in gone]
            heapq.heapify(self.alert_queue)
        self.stats["active_alerts"] = len(self.alerts)

    def _cleanup_expired_alerts(self, now: Optional[float] = None) -> None:
        """:488-517: acknowledged, or older than 30 s."""
        now = time.time() if now is None else now
        self._drop([k for k, a in self.alerts.items() if a.acknowledged or now - a.timestamp > ALERT_MAX_AGE])

    # -- device table (csrc/rcd_alerts.cuh): the same lifecycle for whole frames ----------------------
    def attach_engine(self, engine, id_of, max_alerts: int = 1 << 20, index_of=None) -> None:
        """Keep the alert table on the GPU next to the frames of ``engine`` (a ``FrameEngine``); ``id_of(k)``
        maps the caller ids of the pairs back to vehicle id strings, ``index_of(id)`` the other way (needed
        only for ``acknowledge_alert`` to reach the device table).  Call again after the engine was replaced:
        the live alerts are folded into the new table."""
        self._engine, self._id_of, self._index_of = engine, id_of, index_of
        engine.alerts_configure(max_alerts)
        if self.alerts and index_of is not None:  # migrate what is alive (a FrameCache grew into a new handle)
            import numpy as np
            from . import _native as N
            live = [a for a in self.alerts.values() if index_of(a.vehicle_id) is not None and index_of(a.other_vehicle_id) is not None]
            p = np.zeros(len(live), dtype=N.PAIR_DTYPE)
            for k, a in enumerate(live):
                p[k]["i"], p[k]["j"] = index_of(a.vehicle_id), index_of(a.other_vehicle_id)
                p[k]["risk"], p[k]["ttc"], p[k]["priority"] = a.risk_level, a.time_to_collision, a.priority
            ev, _ = engine.alerts_update_pairs(p, time.time())
            # (the created events come back in arbitrary order: match them by key)
            by_key = {(index_of(a.vehicle_id), index_of(a.other_vehicle_id)): a.id for a in live}
            self._by_number = {int(e["alert_id"]): by_key[(int(e["i"]), int(e["j"]))] for e in ev}

    def _apply_event(self, e) -> AlertInfo:
        from . import _native as N
        vid, other = self._id_of(int(e["i"])), self._id_of(int(e["j"]))
        number = int(e["alert_id"])
        msg = alert_message(float(e["risk"]), other, float(e["ttc"]), float(e["distance"]))
        alert_id = self._by_number.get(number)
        a = self.alerts.get(alert_id) if alert_id is not None else None
        if a is None:
            a = AlertInfo(id=f"alert-{number}", vehicle_id=vid, other_vehicle_id=other, risk_level=float(e["risk"]),
                          time_to_collision=float(e["ttc"]), message=msg, priority=int(e["priority"]),
                          timestamp=float(e["timestamp"]), acknowledged=bool(e["acknowledged"]))
            self._by_number[number] = a.id
            self._store(a)
        else:
            old = a.priority
            a.risk_level, a.time_to_collision, a.message = float(e["risk"]), float(e["ttc"]), msg
            a.priority, a.timestamp = int(e["priority"]), float(e["timestamp"])
            if a.priority != old or int(e["kind"]) == N.ALERT_PRIORITY_CHANGED:
                self._requeue(a)
        return a

    def process_frame(self, now: Optional[float] = None, report_refreshed: bool = False) -> List[AlertInfo]:
        """process_collision_risks (:259-285) for every risk of the engine's last frame, on the device.
        Returns only what the reference's queue would hear about: created alerts and priority changes
        (plus refreshed ones on request); ``alerts`` / ``vehicle_alerts`` / ``alert_queue`` follow those."""
        ev, st = self._engine.alerts_update(time.time() if now is None else now, report_refreshed)
        out = [self._apply_event(e) for e in ev]
        self.stats["active_alerts"] = st["n_live"]
        return out

    def _drop_events(self, ev) -> List[Tuple[str, str]]:
        """Drop the alerts of the device table's EXPIRED events from the host dicts; returns their (vehicle, other) keys."""
        self._drop([self._by_number.pop(int(e["alert_id"]), None) for e in ev])
        return [(self._id_of(int(e["i"])), self._id_of(int(e["j"]))) for e in ev]

    def cleanup_expired(self, now: Optional[float] = None, max_age: float = ALERT_MAX_AGE) -> List[Tuple[str, str]]:
        """_cleanup_expired_alerts (:488-517) on the device table; returns the (vehicle, other) keys that were dropped."""
        ev, st = self._engine.alerts_expire(time.time() if now is None else now, max_age)
        keys = self._drop_events(ev)
        self.stats["active_alerts"] = st["n_live"]
        return keys

    def retire_vehicles(self, ev, vehicle_ids) -> List[Tuple[str, str]]:
        """The host side of retiring vehicles on the attached engine (``FrameEngine.retire`` / ``retire_stale``): drop
        the alerts of its EXPIRED events -- call while ``id_of`` still names the departed vehicles -- and forget the
        departed vehicles' per-vehicle entries.  Returns the (vehicle, other) keys that were dropped."""
        keys = self._drop_events(ev)
        for v in vehicle_ids:
            self.vehicle_alerts.pop(v, None)
        return keys

    def acknowledge(self, vehicle_id_index: int, other_vehicle_index: int) -> bool:
        """acknowledge_alert (:199-213) addressed by the pair's caller ids (device table)."""
        found = self._engine.alerts_acknowledge([vehicle_id_index], [other_vehicle_index]) == 1
        if found and self._id_of is not None:
            alert_id = self.vehicle_alerts.get(self._id_of(vehicle_id_index), {}).get(self._id_of(other_vehicle_index))
            if alert_id in self.alerts:
                self.alerts[alert_id].acknowledged = True
        return found

    def get_stats(self) -> Dict[str, Any]:
        return dict(self.stats)
