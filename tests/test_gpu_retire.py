"""Retiring departed and silent vehicles from a record-built frame (rcd_retire, rcd_retire_stale, rcd_ingest_release):
a frame with retired slots must step exactly like an upload of its live vehicles, staleness is strict at the float64
boundary, recycled slots start from nothing, and the alerts of departed vehicles go with them."""
import ctypes

import numpy as np
import pytest

from tests.gpu_helpers import feed_rounds as _feed, vehicle_messages as _messages

pytestmark = pytest.mark.gpu

BOUNDS = ((-300.0, -300.0, -10.0), (1300.0, 1300.0, 110.0))
TOTALS = ("n_objects", "n_candidates", "n_potential", "n_pairs", "n_high_risk", "n_written", "n_alerts", "n_exact",
          "n_fallback")


def _N():
    from rcd_b200.host import _native as N
    return N


def _W():
    from rcd_b200.host import workloads as W
    return W


def _frame(kind, n, seed):
    W = _W()
    if kind == "uniform":
        return W.uniform_frame(n, seed, map_size=1000.0, drone_fraction=0.3)
    return W.hotspot_frame(n, seed, 1000.0, 4, radius_range=(100.0, 250.0))


def _same_step(a, b, run, live, n):
    """Step a (frame with retired slots) and b (upload of the live slots, ids = slots): same records, totals, tests."""
    run(a)
    run(b)
    pa, pb = a.download(), b.download()
    assert pa.tobytes() == pb.tobytes()
    ca, cb = a.counts(), b.counts()
    assert ca["n_objects"] == n and ca["n_owned"] == n and cb["n_owned"] == len(live)
    assert all(ca[k] == cb[k] for k in TOTALS if k != "n_objects"), (ca, cb)
    assert a.pair_tests() == b.pair_tests()
    gone = np.setdiff1d(np.arange(n), live)
    cand, risk = a.candidate_counts(), a.risk_counts()
    assert not cand[gone].any() and not risk[gone].any()
    assert np.array_equal(cand[live], b.candidate_counts()) and np.array_equal(risk[live], b.risk_counts())
    return pa, ca


def _modes():
    N = _N()
    return [
        ("detect r100 t10", lambda e: e.step(N.MODE_DETECT, 100.0, 10.0)),
        ("detect r60 t4", lambda e: e.step(N.MODE_DETECT, 60.0, 4.0)),
        ("predict", lambda e: e.step(N.MODE_PREDICT)),
        ("predict + detect", lambda e: e.step(N.MODE_PREDICT, 100.0, 10.0, with_detect=True)),
        ("compute node", lambda e: (e.set_compute_node_params(4.0, 0.4), e.step(N.MODE_COMPUTE_NODE, 80.0))),
    ]


# ---- 1. equivalence with an upload of the live vehicles --------------------------------------------------------------
@pytest.mark.parametrize("kind", ["uniform", "hotspot"])
def test_retired_frame_steps_like_an_upload_of_the_live_vehicles(kind):
    from rcd_b200.host.engine import FrameEngine
    from rcd_b200.host.ingest import VehiclePositionStream
    n = 3000
    ids = [f"veh-{k}" for k in range(n)]
    with VehiclePositionStream(4096, 1 << 21, world_bounds=BOUNDS) as s, FrameEngine(4096, 1 << 21, world_bounds=BOUNDS) as e:
        last = _feed(s, _frame(kind, n, 21), ids, 3, 100.0, 22)
        assert [s.ingest.slot_of(v) for v in ids[:5]] == list(range(5))
        gone = np.sort(np.random.default_rng(23).choice(n, int(0.3 * n), replace=False))
        assert sorted(s.remove_vehicles([ids[k] for k in gone])) == sorted(ids[k] for k in gone)
        live = np.setdiff1d(np.arange(n), gone)
        codes = s.engine.history_classify()
        assert len(set(codes[live].tolist())) >= 2
        e.upload(_W().take(last, live), ids=live.astype(np.uint32))
        e.set_patterns(codes[live])
        for name, run in _modes():
            pairs, c = _same_step(s.engine, e, run, live, n)
            assert len(pairs) > 20, name
            assert not np.isin(pairs["i"], gone).any() and not np.isin(pairs["j"], gone).any()


# A road along y, 4 m wide and 100 m high, with a small radius: one cell across x (nx = 1) and ten layers in z, so the
# tiles made only of retired queries would have an inverted box of (2 - ny)(2 - nz) > 0 rows if they were not empty.
ROAD = ((0.0, 0.0, 0.0), (4.0, 2000.0, 100.0))


@pytest.mark.parametrize("bounds", [ROAD, None], ids=["static", "from-data"])
def test_whole_retired_tiles_on_a_narrow_tall_grid(bounds):
    N = _N()
    from rcd_b200.host.engine import FrameEngine
    from rcd_b200.host.ingest import VehiclePositionStream
    n = 2000
    rng = np.random.default_rng(81)
    f = _W().uniform_frame(n, 82, map_size=2000.0)
    f["px"] = rng.uniform(0.0, 4.0, n).astype(np.float32)
    f["pz"] = rng.uniform(0.0, 100.0, n).astype(np.float32)
    f["vx"] = rng.uniform(-0.5, 0.5, n).astype(np.float32)
    f["vz"] = rng.uniform(-2.0, 2.0, n).astype(np.float32)
    ids = [f"road-{k}" for k in range(n)]
    with VehiclePositionStream(4096, 1 << 20, world_bounds=bounds) as s, FrameEngine(4096, 1 << 20, world_bounds=bounds) as e:
        s.handle_messages(_messages(f, ids, 3.0))
        gone = np.sort(rng.choice(n, 700, replace=False))  # about 22 tiles of retired queries behind the live ones
        s.remove_vehicles([ids[k] for k in gone])
        live = np.setdiff1d(np.arange(n), gone)
        e.upload(_W().take(f, live), ids=live.astype(np.uint32))
        for run in (lambda x: x.step(N.MODE_DETECT, 10.0, 4.0), lambda x: x.step(N.MODE_DETECT, 20.0, 10.0),
                    lambda x: x.step(N.MODE_COMPUTE_NODE, 10.0)):
            _same_step(s.engine, e, run, live, n)
            assert e.pair_tests() > 0 and e.counts()["n_candidates"] > 100


# ---- 2. staleness at the float64 boundary ----------------------------------------------------------------------------
def test_retire_stale_is_strict_at_the_boundary():
    N = _N()
    from rcd_b200.host.engine import FrameEngine
    from rcd_b200.host.ingest import VehiclePositionStream
    max_age = 30.0
    now = float(np.nextafter(30.5, np.inf))
    t_old, t_edge = 0.5, now - max_age
    assert now - t_edge == max_age and now - t_old == np.nextafter(max_age, np.inf)
    n = 600
    kind = np.random.default_rng(31).integers(0, 3, n)  # 0: exactly max_age old, 1: one ulp older, 2: fresh
    ts = np.choose(kind, [t_edge, t_old, now])
    ids = [f"s{k}" for k in range(n)]
    with VehiclePositionStream(1024, 1 << 18, world_bounds=BOUNDS) as s:
        s.handle_messages(_messages(_frame("uniform", n, 32), ids, ts))
        lib, h = N.load(), s.engine._h
        # too little room: RCD_ECAPACITY, the true count, nothing retired
        out = np.zeros(8, np.uint32)
        got = ctypes.c_uint64()
        st = N.RcdAlertStats()
        rc = lib.rcd_retire_stale(h, now, max_age, out.ctypes.data_as(ctypes.c_void_p), 8, ctypes.byref(got), None, 0,
                                  ctypes.byref(st))
        assert rc == N.RCD_ECAPACITY and got.value == int((kind == 1).sum())
        slots, ev, _ = s.engine.retire_stale(now, max_age)
        assert np.array_equal(slots, np.flatnonzero(kind == 1))  # ascending, exactly the older-by-one-ulp ones
        assert len(ev) == 0
        again, _, _ = s.engine.retire_stale(now, max_age)
        assert len(again) == 0
        # nor does the stream-level call
        assert s.retire_stale(now, max_age) == []
        s.engine.step(N.MODE_DETECT, 100.0, 10.0)
        assert s.engine.counts()["n_objects"] == n
    with FrameEngine(1024, 1 << 18, world_bounds=BOUNDS) as e:
        e.upload(_frame("uniform", 100, 33))
        with pytest.raises(N.NativeError) as err:
            e.retire_stale(now, max_age)
        assert err.value.code == N.RCD_ESTATE
        e.upload(_W().empty_frame(0))  # an empty upload starts a record-built frame
        assert len(e.retire_stale(now, max_age)[0]) == 0


# ---- 3. recycled slots: fresh rings, no inherited alerts -------------------------------------------------------------
def test_recycled_slots_start_fresh_and_departed_alerts_go():
    N = _N()
    from rcd_b200.host.ingest import VehiclePositionStream
    from rcd_b200.host.warning_system import AlertManager
    n, k = 2000, 300
    rng = np.random.default_rng(41)
    old_ids = [f"old-{q}" for q in range(n)]
    new_ids = [f"new-{q}" for q in range(k)]
    with VehiclePositionStream(4096, 1 << 21, world_bounds=BOUNDS) as s, \
            VehiclePositionStream(4096, 1 << 21, world_bounds=BOUNDS) as fresh:
        am = AlertManager()
        am.attach_engine(s.engine, s.ingest.id_of, max_alerts=1 << 16)
        _feed(s, _W().uniform_frame(n, 42, map_size=600.0, drone_fraction=0.2), old_ids, 3, 10.0, 43)
        s.engine.history_classify(want_codes=False)
        s.engine.step(N.MODE_DETECT, 100.0, 10.0)
        am.process_frame(now=11.0)
        before = s.engine.alerts_download()
        gone_ids = [old_ids[q] for q in rng.choice(n, k, replace=False)]
        gone = np.array(sorted(s.ingest.slot_of(v) for v in gone_ids), np.uint32)
        want = before[np.isin(before["i"], gone) | np.isin(before["j"], gone)].copy()
        assert len(want) > 10
        want["kind"] = N.ALERT_EXPIRED
        seen = []
        drop = am.retire_vehicles
        am.retire_vehicles = lambda ev, vids: (seen.append(ev.copy()), drop(ev, vids))[1]
        assert sorted(s.remove_vehicles(gone_ids, alerts=am)) == sorted(gone_ids)
        ev = np.sort(seen[0], order=["i", "j"])
        assert ev.tobytes() == np.sort(want, order=["i", "j"]).tobytes()  # event for event
        after = s.engine.alerts_download()
        assert len(after) == len(before) - len(want)
        assert not np.isin(after["i"], gone).any() and not np.isin(after["j"], gone).any()
        assert not any(v in am.vehicle_alerts for v in gone_ids)
        assert not any(a.vehicle_id in gone_ids or a.other_vehicle_id in gone_ids for a in am.alerts.values())
        assert am.stats["active_alerts"] == len(after)
        # new vehicles take the freed slots, lowest first; their rings hold nothing of the previous occupants
        nf = _W().uniform_frame(k, 44, map_size=600.0, drone_fraction=0.2)
        _feed(fresh, nf, new_ids, 3, 20.0, 45)
        _feed(s, nf, new_ids, 3, 20.0, 45)
        assert [s.ingest.slot_of(v) for v in new_ids] == gone.tolist()
        assert s.ingest.n_objects == n
        codes, fcodes = s.engine.history_classify(), fresh.engine.history_classify()
        assert len(set(fcodes.tolist())) >= 2
        assert np.array_equal(codes[gone], fcodes[[fresh.ingest.slot_of(v) for v in new_ids]])
        # the next fold creates the alerts of the new occupants: none is a refresh of an inherited one
        s.engine.step(N.MODE_DETECT, 100.0, 10.0)
        ev, _ = s.engine.alerts_update(21.5, report_refreshed=True)
        mine = ev[np.isin(ev["i"], gone) | np.isin(ev["j"], gone)]
        assert len(mine) > 10 and (mine["kind"] == N.ALERT_CREATED).all()


# ---- 4. query lists, graph replay, radius queries --------------------------------------------------------------------
def test_query_lists_graph_replay_and_radius_queries():
    N = _N()
    from rcd_b200.host.engine import FrameEngine
    from rcd_b200.host.ingest import VehicleIngest
    n = 3000
    rng = np.random.default_rng(51)
    ids = [f"q{q}" for q in range(n)]
    with VehicleIngest(threads=1) as g, FrameEngine(4096, 1 << 21, world_bounds=BOUNDS) as a, \
            FrameEngine(4096, 1 << 21, world_bounds=BOUNDS, graph=True) as b:
        rec, ms = g.decode(_messages(_frame("hotspot", n, 52), ids, 5.0))
        for e in (a, b):
            e.apply_records(rec, g.n_objects, ms)

        def both(k):
            for _ in range(k):
                for e in (a, b):
                    e.step(N.MODE_PREDICT, 100.0, 10.0, with_detect=True)
                assert a.download().tobytes() == b.download().tobytes() and a.counts() == b.counts()

        both(4)
        gone = np.sort(rng.choice(n, 800, replace=False)).astype(np.uint32)
        for e in (a, b):
            e.retire(gone)
        both(4)
        assert b.graph_replays() >= 2
        live = np.setdiff1d(np.arange(n), gone)
        q_with = np.sort(rng.choice(n, 1200, replace=False)).astype(np.uint32)
        q_without = q_with[~np.isin(q_with, gone)]
        res = []
        for q in (q_with, q_without):
            a.set_queries(q)
            a.step(N.MODE_DETECT, 100.0, 10.0)
            c = a.counts()
            res.append((a.download().tobytes(), {k: c[k] for k in TOTALS}, a.pair_tests()))
        assert res[0] == res[1] and len(res[0][0]) > 0
        a.set_queries(None)
        hits = a.query_radius([[500.0, 500.0, 50.0]], 5000.0)[0]
        assert np.array_equal(np.sort(hits), live)


# ---- 5. edges --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bounds", [BOUNDS, None], ids=["static", "from-data"])
def test_edges(bounds):
    N = _N()
    from rcd_b200.host.engine import FrameEngine
    from rcd_b200.host.ingest import VehicleIngest
    n = 500
    ids = [f"e{q}" for q in range(n)]
    with VehicleIngest(threads=1) as g, FrameEngine(1024, 1 << 18, world_bounds=bounds) as e:
        assert len(e.retire([])[0]) == 0  # empty frame
        with pytest.raises(N.NativeError) as err:
            e.retire([0])
        assert err.value.code == N.RCD_EINVAL
        rec, ms = g.decode(_messages(_frame("uniform", n, 61), ids, 1.0))
        e.apply_records(rec, g.n_objects, ms)
        e.retire(np.arange(0, n, 3))
        e.step(N.MODE_DETECT, 100.0, 10.0)
        p0, c0, t0 = e.download().tobytes(), e.counts(), e.pair_tests()
        e.retire(np.arange(0, n, 3))  # twice: no-op
        for bad in ([n], [1, n + 7]):
            with pytest.raises(N.NativeError) as err:
                e.retire(np.array(bad, np.uint32))
            assert err.value.code == N.RCD_EINVAL
        e.step(N.MODE_DETECT, 100.0, 10.0)
        assert (e.download().tobytes(), e.counts(), e.pair_tests()) == (p0, c0, t0)
        e.retire(np.arange(n))  # everybody
        for mode in (N.MODE_DETECT, N.MODE_PREDICT, N.MODE_COMPUTE_NODE):
            e.step(mode, 100.0, 10.0)
            c = e.counts()
            assert c["n_pairs"] == 0 and c["n_candidates"] == 0 and e.pair_tests() == 0 and c["n_objects"] == n
        # a record brings a slot back
        e.apply_records(rec[:1], g.n_objects, 0)
        e.step(N.MODE_COMPUTE_NODE, 100.0)
        assert e.counts()["n_candidates"] == 1  # the vehicle finds itself (quirk Q8)


# ---- 6. churn at a full id limit -------------------------------------------------------------------------------------
def test_churn_at_a_full_id_limit():
    N = _N()
    from rcd_b200.host.engine import FrameEngine
    from rcd_b200.host.ingest import VehiclePositionStream
    L, rounds = 1000, 50
    rng = np.random.default_rng(71)
    live = [f"c{q}" for q in range(L)]
    nid = L
    with VehiclePositionStream(L, 1 << 20, world_bounds=BOUNDS) as s, FrameEngine(L, 1 << 20, world_bounds=BOUNDS) as e:
        for r in range(rounds + 1):
            f = _W().uniform_frame(L, 100 + r, map_size=700.0, drone_fraction=0.2)
            t = float(r)
            if r == 0:
                s.handle_messages(_messages(f, live, t))
                continue
            silent = set(rng.choice(L, L // 10, replace=False).tolist())
            talk = [q for q in range(L) if q not in silent]
            s.handle_messages(_messages(f, live, t, talk))
            departed = s.retire_stale(t, 0.5)
            assert sorted(departed) == sorted(live[q] for q in silent)
            for q in sorted(silent):  # newcomers take the rows of the departed
                live[q] = f"c{nid}"
                nid += 1
            s.handle_messages(_messages(f, live, t, sorted(silent)))
            assert s.ingest.rejected == 0 and s.engine.n <= L and s.ingest.n_objects <= L
        slot = np.array([s.ingest.slot_of(v) for v in live])
        assert sorted(slot.tolist()) == list(range(L))
        e.upload(_W().take(f, np.argsort(slot)), ids=np.arange(L, dtype=np.uint32))
        for run in (lambda x: x.step(N.MODE_DETECT, 100.0, 10.0), lambda x: x.step(N.MODE_COMPUTE_NODE, 100.0)):
            pairs, _ = _same_step(s.engine, e, run, np.arange(L), L)
            assert len(pairs) > 20
