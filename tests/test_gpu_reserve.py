"""Growing a handle in place (rcd_reserve, rcd_alerts_reserve): a grown handle steps like one created at the final size,
a step right after a reserve equals the step before it, the frame state, rings, record times, query list and alerts
survive, a refused reserve leaves the handle as it was, and the class-level code keeps one handle for its whole life."""
import ctypes

import numpy as np
import pytest

from tests.test_gpu_retire import BOUNDS, TOTALS, _messages

pytestmark = pytest.mark.gpu


def _N():
    from rcd_b200.host import _native as N
    return N


def _W():
    from rcd_b200.host import workloads as W
    return W


def _same_alerts(ea, eb):
    """Alert events or downloads of two handles: the same records, and the same new alert numbers handed out.  (Which
    pair gets which number within one fold depends on the order the device threads create them, so a record's number
    is compared only as part of the set of numbers a call created.)"""
    N = _N()
    assert len(ea) == len(eb)
    created = [np.sort(e["alert_id"][e["kind"] == N.ALERT_CREATED]) for e in (ea, eb)]
    assert np.array_equal(*created)
    xa, xb = ea.copy(), eb.copy()
    xa["alert_id"] = 0
    xb["alert_id"] = 0
    assert np.sort(xa).tobytes() == np.sort(xb).tobytes()


def _same_step(a, b, run, exact_grid=True):
    """Step both engines: the same records and totals; the same pair tests when both grids are sized alike."""
    run(a)
    run(b)
    assert a.download().tobytes() == b.download().tobytes()
    ca, cb = a.counts(), b.counts()
    assert ca["n_pairs"] <= a.max_pairs and cb["n_pairs"] <= b.max_pairs
    keys = TOTALS if exact_grid else [k for k in TOTALS if k not in ("n_exact", "n_fallback")]
    assert all(ca[k] == cb[k] for k in keys), (ca, cb)
    if exact_grid:
        assert a.pair_tests() == b.pair_tests()
    return ca


def _modes():
    N = _N()
    return [
        lambda e: e.step(N.MODE_DETECT, 100.0, 10.0),
        lambda e: e.step(N.MODE_PREDICT),
        lambda e: e.step(N.MODE_COMPUTE_NODE, 80.0),
    ]


# ---- 1. a grown handle equals a handle created at the final size ------------------------------------------------------
def test_grown_stream_equals_a_stream_created_at_the_final_size():
    N, W = _N(), _W()
    from rcd_b200.host.ingest import VehiclePositionStream
    n0, n1 = 3000, 6000
    ids = [f"veh-{k}" for k in range(n1)]
    rng = np.random.default_rng(91)
    f = W.uniform_frame(n1, 92, map_size=2000.0, drone_fraction=0.3)
    q = np.sort(rng.choice(n0, 900, replace=False)).astype(np.uint32)
    with VehiclePositionStream(4096, 1 << 18, world_bounds=BOUNDS) as a, \
            VehiclePositionStream(1 << 16, 1 << 20, world_bounds=BOUNDS) as b:
        for s in (a, b):
            s.engine.alerts_configure(1 << 16)
        grown = False
        for r in range(7):
            t = 100.0 + 0.5 * r
            if r == 3:  # a query list, then the reserve: the list, rings, record times and alerts stay
                for s in (a, b):
                    s.engine.set_queries(q)
                a.reserve(1 << 16, 1 << 20)
                assert a.engine.max_objects == 1 << 16 and a.engine.max_pairs == 1 << 20
                grown = True
                _same_step(a.engine, b.engine, _modes()[0])
                for s in (a, b):
                    s.engine.set_queries(None)
            live = n0 if r < 3 else n1  # past the old capacity once grown
            talk = [k for k in range(live) if not (r == 6 and k % 10 == 0)]  # the last batch leaves some silent
            msg = _messages(f, ids, t, talk)
            for s in (a, b):
                s.handle_messages(msg)
            assert a.ingest.rejected == 0 and a.ingest.n_objects == b.ingest.n_objects == live
            assert np.array_equal(a.engine.history_classify(), b.engine.history_classify())
            for run in _modes():
                _same_step(a.engine, b.engine, run, grown)
            _same_step(a.engine, b.engine, lambda e: e.step(N.MODE_PREDICT, 100.0, 10.0, with_detect=True), grown)
            ea, sa = a.engine.alerts_update(t, report_refreshed=True)
            eb, sb = b.engine.alerts_update(t, report_refreshed=True)
            assert sa == sb
            _same_alerts(ea, eb)
            _same_alerts(a.engine.alerts_download(), b.engine.alerts_download())
            f = W.advance(f, 0.5, rng)
        assert len(a.engine.alerts_download()) > 100
        sa, ea, _ = a.engine.retire_stale(t, 0.4)
        sb, eb, _ = b.engine.retire_stale(t, 0.4)
        assert np.array_equal(sa, sb) and np.array_equal(sa, np.arange(0, n1, 10))
        _same_alerts(ea, eb)
        _same_step(a.engine, b.engine, lambda e: e.step(N.MODE_PREDICT, 100.0, 10.0, with_detect=True))


# ---- 2. a step straight after a reserve equals the step before it -----------------------------------------------------
@pytest.mark.parametrize("case", ["upload", "halo", "query list"])
def test_step_after_reserve_equals_the_step_before(case):
    N, W = _N(), _W()
    from rcd_b200.host.engine import FrameEngine
    n = 3000
    frame = W.hotspot_frame(n, 11, 1000.0, 4, radius_range=(100.0, 250.0))
    with FrameEngine(4096, 1 << 19, world_bounds=BOUNDS) as e:
        e.upload(frame)
        e.set_patterns(W.random_patterns(n, 12))
        if case == "halo":
            e.set_owned(2000)
        if case == "query list":
            e.set_queries(np.sort(np.random.default_rng(13).choice(n, 700, replace=False)))
        for run in _modes() + [lambda x: x.step(N.MODE_PREDICT, 100.0, 10.0, with_detect=True)]:
            run(e)
            before = (e.download().tobytes(), e.counts(), e.pair_tests())
            assert len(before[0]) > 0
            # (up to 16 Ki objects keep the grid of a 4 Ki handle: the pair-test count must not move either)
            e.reserve(e.max_objects + 2048, 2 * e.max_pairs)
            run(e)
            assert (e.download().tobytes(), e.counts(), e.pair_tests()) == before


# ---- 3. pair-buffer overflow recovery ---------------------------------------------------------------------------------
def test_pair_buffer_overflow_recovers_without_losing_alerts():
    N, W = _N(), _W()
    from rcd_b200.host.engine import FrameEngine
    n = 3000
    frame = W.hotspot_frame(n, 21, 1000.0, 4, radius_range=(100.0, 250.0))
    pat = W.random_patterns(n, 22)
    fused = lambda e: e.step(N.MODE_PREDICT, 100.0, 10.0, with_detect=True)
    with FrameEngine(4096, 512, world_bounds=BOUNDS) as a, FrameEngine(4096, 1 << 20, world_bounds=BOUNDS) as b:
        for e in (a, b):
            e.alerts_configure(1 << 16)
            e.upload(frame)
            e.set_patterns(pat)
            fused(e)
        c = a.counts()
        assert c["n_pairs"] > c["n_written"] == 512
        a.reserve(max_pairs=c["n_pairs"])
        fused(a)
        assert a.counts()["n_written"] == c["n_pairs"]
        ea, sa = a.alerts_update(5.0, report_refreshed=True)
        eb, sb = b.alerts_update(5.0, report_refreshed=True)
        assert sa == sb and sa["n_created"] > 512
        _same_alerts(ea, eb)
        _same_alerts(a.alerts_download(), b.alerts_download())


# ---- 4. alert table growth --------------------------------------------------------------------------------------------
def _risk_pairs(n, seed, first=0):
    N = _N()
    rng = np.random.default_rng(seed)
    p = np.zeros(n, N.PAIR_DTYPE)
    p["i"] = np.arange(first, first + n, dtype=np.uint32)
    p["j"] = p["i"] + 1_000_000
    p["risk"] = rng.uniform(0.3, 1.0, n).astype(np.float32)
    p["ttc"] = rng.uniform(0.0, 10.0, n).astype(np.float32)
    p["distance"] = rng.uniform(0.0, 5.0, n).astype(np.float32)
    p["priority"] = rng.integers(0, 4, n)
    p["offset"] = 255
    return p


def test_alert_table_grows_keeping_every_live_alert():
    N = _N()
    from rcd_b200.host.engine import FrameEngine
    lib = N.load()
    with FrameEngine(1024, 1 << 12) as a, FrameEngine(1024, 1 << 12) as b, FrameEngine(1024, 1 << 12) as c:
        assert lib.rcd_alerts_reserve(c._h, 1 << 12) == N.RCD_ESTATE  # never configured
        a.alerts_configure(512)  # a 1024-slot table; downloads see 512 of its alerts
        b.alerts_configure(4096)
        first = _risk_pairs(1500, 31)
        _, st = a.alerts_update_pairs(first, 1.0)
        assert st["n_created"] == 1024 and st["n_dropped"] == 1500 - 1024
        acked = a.alerts_acknowledge(first["i"][::7], first["j"][::7])
        seen = a.alerts_download()
        assert len(seen) == 512 and seen["acknowledged"].any()
        a.alerts_reserve(4096)
        a.alerts_reserve(100)  # smaller: no-op
        held = a.alerts_download()
        # every live alert survives: what the small table showed, record for record (numbers, timestamps, flags)
        assert len(held) == 1024 and np.array_equal(np.sort(held["alert_id"]), np.arange(1024))
        assert set(r.tobytes() for r in seen) <= set(r.tobytes() for r in held)
        kept = first[np.isin(first["i"], held["i"])]
        assert np.array_equal(held["risk"], kept["risk"]) and np.array_equal(held["priority"], kept["priority"])
        assert (held["timestamp"] == 1.0).all()
        assert np.array_equal(held["acknowledged"] != 0, np.isin(held["i"], first["i"][::7]))
        assert acked == held["acknowledged"].sum()
        ev, st = a.alerts_update_pairs(_risk_pairs(1, 32, first=5000), 2.0)
        assert st["n_created"] == 1 and st["n_dropped"] == 0 and int(ev["alert_id"][0]) == 1024  # the next number
        b.alerts_update_pairs(kept, 1.0)
        b.alerts_acknowledge(first["i"][::7], first["j"][::7])
        b.alerts_update_pairs(_risk_pairs(1, 32, first=5000), 2.0)
        # from here on it behaves like a table made at the large size holding the same alerts
        _same_alerts(a.alerts_download(), b.alerts_download())
        more = np.concatenate([first[::3], _risk_pairs(2000, 33, first=10_000)])
        for e in (a, b):
            e.alerts_acknowledge(more["i"][::11], more["j"][::11])
        (ea, sa), (eb, sb) = (e.alerts_update_pairs(more, 20.0, report_refreshed=True) for e in (a, b))
        assert sa == sb and sa["n_dropped"] == 0
        _same_alerts(ea, eb)
        (ea, sa), (eb, sb) = (e.alerts_expire(40.0, 30.0) for e in (a, b))
        assert sa == sb and sa["n_expired"] > 0 and sa["n_live"] > 0
        _same_alerts(ea, eb)
        _same_alerts(a.alerts_download(), b.alerts_download())


# ---- 5. state rules ---------------------------------------------------------------------------------------------------
def test_reserve_state_rules():
    N, W = _N(), _W()
    from rcd_b200.host.engine import FrameEngine
    lib = N.load()
    n = 2000
    frame = W.uniform_frame(n, 41, map_size=800.0, drone_fraction=0.3)
    with FrameEngine(4096, 1 << 18) as e:
        e.alerts_configure(1 << 14)
        e.upload(frame)
        e.step(N.MODE_DETECT)
        c = e.counts()
        for mo, mp in ((0, 0), (100, 0), (0, 16), (4096, 1 << 18)):  # no growth: no-ops, the frame stays
            e.reserve(mo, mp)
        assert e.counts() == c and (e.max_objects, e.max_pairs) == (4096, 1 << 18)
        e.reserve(8192)
        assert (e.max_objects, e.max_pairs) == (8192, 1 << 18)
        for call in (e.counts, e.download, e.pair_tests, lambda: e.alerts_update(1.0),
                     lambda: e.step(N.MODE_PREDICT, append=True)):
            with pytest.raises(N.NativeError) as err:
                call()
            assert err.value.code == N.RCD_ESTATE
        e.step(N.MODE_DETECT)
        e.download_begin(np.zeros(1 << 18, N.PAIR_DTYPE))
        assert lib.rcd_reserve(e._h, 1 << 14, 0) == N.RCD_ESTATE
        pairs, _ = e.download_finish()
        e.step(N.MODE_DETECT)
        e.summary_begin(1.0)
        assert lib.rcd_reserve(e._h, 1 << 14, 0) == N.RCD_ESTATE
        assert lib.rcd_alerts_reserve(e._h, 1 << 15) == N.RCD_ESTATE
        e.summary_finish()
        e.reserve(1 << 14)
        e.alerts_reserve(1 << 15)
        e.step(N.MODE_DETECT)
        assert e.download().tobytes() == np.sort(pairs, order=["i", "j", "predicted"]).tobytes()


def test_graph_replay_after_reserve_recaptures():
    N, W = _N(), _W()
    from rcd_b200.host.engine import FrameEngine
    n = 3000
    frame = W.uniform_frame(n, 51, map_size=1000.0, drone_fraction=0.3)
    pat = W.random_patterns(n, 52)
    bounds = ((0.0, 0.0, 0.0), (1000.0, 1000.0, 100.0))
    with FrameEngine(4096, 1 << 19, world_bounds=bounds, graph=True) as a, \
            FrameEngine(4096, 1 << 19, world_bounds=bounds) as b:
        def frames(k):
            for _ in range(k):
                for e in (a, b):
                    e.upload(frame)
                    e.set_patterns(pat)
                    e.step(N.MODE_PREDICT, 100.0, 10.0, with_detect=True)
                assert a.download().tobytes() == b.download().tobytes() and a.counts() == b.counts()

        frames(3)  # runs, captures, replays
        assert a.graph_replays() == 1
        for e in (a, b):
            e.reserve(8192, 1 << 20)
        frames(3)  # the graphs of the old buffers are gone: captured again, then replayed
        assert a.graph_replays() == 2


# ---- 6. failure atomicity ---------------------------------------------------------------------------------------------
def test_refused_reserve_leaves_the_handle_usable():
    N, W = _N(), _W()
    from rcd_b200.host.engine import FrameEngine
    lib = N.load()
    n = 3000
    frame = W.uniform_frame(n, 61, map_size=1000.0, drone_fraction=0.3)
    with FrameEngine(4096, 1 << 18) as e:
        e.alerts_configure(1 << 14)
        e.history_configure(100)
        e.upload(frame)
        e.set_patterns(W.random_patterns(n, 62))
        e.step(N.MODE_PREDICT, 100.0, 10.0, with_detect=True)
        before = (e.download().tobytes(), e.counts(), e.pair_tests())
        assert lib.rcd_reserve(e._h, 1 << 14, 1 << 40) == N.RCD_ENOMEM  # 48-byte records: 52 TB
        assert b"max_pairs" in lib.rcd_last_error(e._h)
        assert lib.rcd_reserve(e._h, 1 << 30, 0) == N.RCD_EINVAL
        assert (e.download().tobytes(), e.counts(), e.pair_tests()) == before  # the frame is still there
        e.step(N.MODE_PREDICT, 100.0, 10.0, with_detect=True)
        assert (e.download().tobytes(), e.counts(), e.pair_tests()) == before
        e.alerts_update(1.0)


# ---- 7. memory is released --------------------------------------------------------------------------------------------
def _optional_parts(e, n):
    """Every part of a handle made at its first use: rings, record times, query list, delivery twin, compact scratch."""
    N, W = _N(), _W()
    from rcd_b200.host.ingest import VehicleIngest
    f = W.uniform_frame(n, 71, map_size=1000.0)
    with VehicleIngest(threads=1) as g:
        rec, ms = g.decode(_messages(f, [f"m{k}" for k in range(n)], 1.0))
        e.apply_records(rec, g.n_objects, ms)
    e.set_queries(np.arange(0, n, 2))
    e.step(N.MODE_DETECT)
    e.download_begin_compact(np.zeros(e.max_pairs, N.PAIR_COMPACT_DTYPE))
    e.download_finish()


def test_reserve_cycles_release_the_old_buffers():
    import torch
    from rcd_b200.host.engine import FrameEngine
    torch.cuda.init()
    with FrameEngine(4096, 1 << 16) as e:
        _optional_parts(e, 1000)
        for k in range(1, 11):
            e.reserve(4096 + k * 20_000, (1 << 16) + k * 100_000)
        e.sync()
        free_grown = torch.cuda.mem_get_info()[0]
        final = (e.max_objects, e.max_pairs)
    with FrameEngine(*final) as f:
        _optional_parts(f, 1000)
        f.sync()
        free_fresh = torch.cuda.mem_get_info()[0]
    assert abs(free_grown - free_fresh) <= 64 << 20, (free_grown, free_fresh)


# ---- 8. class level ---------------------------------------------------------------------------------------------------
def test_prediction_model_keeps_one_handle_while_the_vehicle_count_grows():
    from rcd_b200.host.collision_detection import CollisionDetector, CollisionPredictionModel
    from rcd_b200.host.models import Position, Vector, Vehicle
    from rcd_b200.host.spatial_index import SpatialIndex
    from tests.test_gpu_dropin import _oracle_patterns
    rng = np.random.default_rng(81)
    n = 1500  # the first handle holds 1024 vehicles
    pos = rng.uniform(0, 700, (n, 3)) * np.array([1.0, 1.0, 0.1])
    vel = rng.uniform(-8, 8, (n, 3)) * np.array([1.0, 1.0, 0.0])
    acc = rng.uniform(-1.5, 1.5, (n, 3)) * (rng.random((n, 1)) < 0.5) * np.array([1.0, 1.0, 0.0])

    def feed(models, live, t):
        for i in range(live):
            p = pos[i] + vel[i] * t + 0.5 * acc[i] * t * t
            v = Vehicle(id=f"v{i}", position=Position(*map(float, p)), velocity=Vector(*map(float, vel[i])),
                        acceleration=Vector(*map(float, acc[i])), heading=0.0, size=2.0, type="car", timestamp=t)
            for m in models:
                m.collision_detector.update_vehicle(v)
                m.update_trajectory(v.id, v.position, t)

    def risks(m, vids):
        return [sorted((r.vehicle_id, r.other_vehicle_id, r.time_to_collision, r.distance, r.risk_level, r.is_predicted)
                       for r in m.predict_collisions(v)) for v in vids]

    grown = CollisionPredictionModel(CollisionDetector(SpatialIndex()))
    fresh = CollisionPredictionModel(CollisionDetector(SpatialIndex()))
    frames = grown.collision_detector.spatial_index._frames
    for step in range(6):
        feed([grown, fresh], 500 if step < 3 else n, 0.5 * step)
        table = grown.collision_detector.spatial_index._table
        assert np.array_equal(grown.trajectory_patterns(), _oracle_patterns(grown, table)), step
        assert frames.engine_generation == 1
    assert frames.engine.max_objects >= n
    vids = [f"v{i}" for i in range(0, n, 37)]
    assert sum(len(r) for r in risks(grown, vids)) > 0
    assert risks(grown, vids) == risks(fresh, vids)
    assert fresh.collision_detector.spatial_index._frames.engine_generation == 1


def test_compute_node_detector_grows_in_place():
    from rcd_b200.host import compute_node as CN
    from rcd_b200.host.models import LocationData, Position, Vector
    W = _W()
    n = 3000
    f = W.uniform_frame(n, 91, map_size=900.0)
    states = {}
    for i in range(n):
        st = CN.VehicleState(f"v{i}")
        loc = LocationData(vehicle_id=f"v{i}", timestamp=0.0,
                           position=Position(float(f["px"][i]), float(f["py"][i]), float(f["pz"][i])),
                           velocity=Vector(float(f["vx"][i]), float(f["vy"][i]), float(f["vz"][i])),
                           heading=float(f["heading"][i]), vehicle_type="car")
        st.update(loc)
        if i % 3:
            st.update(loc)
        states[f"v{i}"] = st

    def table(out):
        return sorted((r.vehicle_id1, r.vehicle_id2, r.risk_level, r.relative_velocity,
                       r.position.x, r.position.y, r.position.z) for rs in out.values() for r in rs)

    det = CN.CollisionDetector(prediction_time=4.0, risk_threshold=0.4)
    small = dict(list(states.items())[:600])
    det.detect_collisions_for_all(small, 100.0)
    eng = det._engine
    assert eng.max_objects == 1200
    got = table(det.detect_collisions_for_all(states, 100.0))
    assert det._engine is eng and eng.max_objects == 2 * n
    want = table(CN.CollisionDetector(prediction_time=4.0, risk_threshold=0.4).detect_collisions_for_all(states, 100.0))
    assert len(got) > 0 and got == want
