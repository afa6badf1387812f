"""The drop-in classes (reference signatures) on the GPU against the reference's golden vectors:
the tests read like the reference's own use of its API (warning_system.py:638-714,
compute_node.py:592-642)."""
import numpy as np
import pytest

from tests.helpers import assert_close, assert_pairs_equal, load_golden

pytestmark = pytest.mark.gpu


def _vehicles(frame):
    from rcd_b200.host.models import Position, Vector, Vehicle
    out = []
    for i in range(len(frame["px"])):
        out.append(Vehicle(id=f"v{i}", position=Position(float(frame["px"][i]), float(frame["py"][i]), float(frame["pz"][i])),
                           velocity=Vector(float(frame["vx"][i]), float(frame["vy"][i]), float(frame["vz"][i])),
                           acceleration=Vector(float(frame["ax"][i]), float(frame["ay"][i]), float(frame["az"][i])),
                           heading=float(frame["heading"][i]), size=float(frame["size"][i]),
                           type=f"type{int(frame['type'][i])}", timestamp=0.0))
    return out


def _table(risks):
    return np.array([[int(r.vehicle_id[1:]), int(r.other_vehicle_id[1:]), r.time_to_collision, r.distance,
                      r.relative_speed, r.risk_level, r.collision_position.x, r.collision_position.y,
                      r.collision_position.z] for r in risks], np.float64).reshape(-1, 9)


def _compare(got, want):
    got = got[np.lexsort((got[:, 1], got[:, 0]))]
    assert_pairs_equal(got[:, :2], want[:, :2])
    assert np.array_equal(np.round(got[:, 2], 5), np.round(want[:, 2], 5))
    for c in range(3, 9):
        assert_close(got[:, c], want[:, c], f"col {c}", 1e-6, 1e-6)


def test_detector_per_vehicle_calls_match_golden():
    from rcd_b200.host.collision_detection import CollisionDetector
    from rcd_b200.host.spatial_index import SpatialIndex
    z, frame = load_golden("detect_dense3d.npz")
    det = CollisionDetector(SpatialIndex())
    for v in _vehicles(frame):
        det.update_vehicle(v)
    assert det.detect_collisions("nobody") == []
    risks = []
    for vid in list(det.vehicle_cache):
        risks += det.detect_collisions(vid)
    _compare(_table(risks), z["risks"])
    assert det.spatial_index._frames.frames_run == 1  # N per-vehicle calls = one GPU frame
    st = det.get_stats()
    assert st["total_detections"] == len(frame["px"]) and st["potential_collisions"] == int(z["stat_potential"])
    assert st["high_risk_collisions"] == int(z["stat_high"])
    some = int(z["risks"][0, 0])
    assert {r.other_vehicle_id for r in det.get_collision_risks(f"v{some}")} == \
        {f"v{int(j)}" for i, j in z["risks"][:, :2] if int(i) == some}
    # removing a vehicle removes its pairs from the next frame
    gone = f"v{int(z['risks'][0, 1])}"
    det.remove_vehicle(gone)
    after = det.detect_all()
    assert all(r.other_vehicle_id != gone for rs in after.values() for r in rs) and gone not in after
    # a non-default radius / window is a new frame with the reference's semantics
    z2, frame2 = load_golden("detect_r60_t4.npz")
    det2 = CollisionDetector(SpatialIndex())
    det2.update_vehicles_batch(_vehicles(frame2))
    risks2 = [r for vid in det2.vehicle_cache for r in det2.detect_collisions(vid, float(z2["R"]), float(z2["T"]))]
    _compare(_table(risks2), z2["risks"])


def test_spatial_index_nearby_matches_golden():
    import os
    from rcd_b200.host.models import Position
    from rcd_b200.host.spatial_index import SpatialIndex
    from tests.helpers import GOLDEN
    z = np.load(os.path.join(GOLDEN, "scalars.npz"))
    idx = SpatialIndex()
    n = len(z["near_frame_px"])
    for i in range(n):
        idx.insert_vehicle(f"v{i}", Position(float(z["near_frame_px"][i]), float(z["near_frame_py"][i]), float(z["near_frame_pz"][i])))
    off = z["near_off"]
    for k in (0, 7, 60, 61, 79):
        q = z["near_q"][k]
        got = idx.get_nearby_vehicles(Position(*[float(c) for c in q]), float(z["near_radius"]))
        assert got == {f"v{int(i)}" for i in z["near_ids"][off[k]:off[k + 1]]}
    batch = idx.get_nearby_vehicles_batch([tuple(map(float, q)) for q in z["near_q"]], float(z["near_radius"]))
    assert [sorted(int(s[1:]) for s in b) for b in batch] == [z["near_ids"][off[k]:off[k + 1]].tolist() for k in range(len(off) - 1)]


def test_prediction_model_classifies_histories_and_matches_golden():
    from rcd_b200.host.collision_detection import CollisionDetector, CollisionPredictionModel
    from rcd_b200.host.models import Position
    from rcd_b200.host.spatial_index import SpatialIndex
    z, frame = load_golden("predict_dense3d.npz")
    det = CollisionDetector(SpatialIndex())
    model = CollisionPredictionModel(det)
    vehicles = _vehicles(frame)
    for v, pat in zip(vehicles, z["pattern"]):
        det.update_vehicle(v)
        p = v.position
        if pat == 3:      # fewer than two samples -> the reference falls back to detect_collisions
            model.update_trajectory(v.id, p, 0.0)
            continue
        for k, t in enumerate((0.0, 1.0, 2.0, 3.0)):
            if pat == 0:    # stationary: mean speed < 0.1
                q = Position(p.x, p.y, p.z)
            elif pat == 1:  # constant velocity: mean acceleration < 0.1
                q = Position(p.x + 3.0 * t, p.y, p.z)
            else:           # accelerating
                q = Position(p.x + 2.0 * t + 0.5 * t * t, p.y, p.z)
            model.update_trajectory(v.id, q, t)
    assert np.array_equal(model.trajectory_patterns(), z["pattern"])
    risks = [r for v in vehicles for r in model.predict_collisions(v.id)]
    _compare(_table(risks), z["risks"])
    assert [r.is_predicted for r in sorted(risks, key=lambda r: (int(r.vehicle_id[1:]), int(r.other_vehicle_id[1:])))] \
        == z["is_predicted"].tolist()
    assert det.spatial_index._frames.frames_run == 1
    # alert classification of the same risks
    from rcd_b200.host.warning_system import AlertManager
    mgr = AlertManager()
    alerts = mgr.process_collision_risks(risks)
    assert len(alerts) == sum(r.risk_level >= 0.3 for r in risks)
    assert all(a.priority == mgr._get_priority(a.risk_level, a.time_to_collision) for a in alerts)


def test_compute_node_classes_match_golden():
    from rcd_b200.host import compute_node as CN
    from rcd_b200.host.models import LocationData, Position, Vector
    z, frame = load_golden("implB_dense.npz")
    n = len(frame["px"])
    index = CN.SpatialIndex()
    states = {}
    for i in range(n):
        loc = LocationData(vehicle_id=f"v{i}", timestamp=0.0,
                           position=Position(float(frame["px"][i]), float(frame["py"][i]), float(frame["pz"][i])),
                           velocity=Vector(float(frame["vx"][i]), float(frame["vy"][i]), float(frame["vz"][i])),
                           heading=float(frame["heading"][i]), vehicle_type="car")
        st = CN.VehicleState(f"v{i}")
        st.update(loc)
        if z["has_history"][i]:
            st.update(loc)
        states[f"v{i}"] = st
        index.insert(f"v{i}", loc.position)
    assert index.get_vehicle_count() == n
    det = CN.CollisionDetector()
    want = z["risks"]  # i j risk ttc rel_speed cx cy cz
    allr = det.detect_collisions_for_all(states, 100.0)
    got = np.array([[int(r.vehicle_id1[1:]), int(r.vehicle_id2[1:]), r.risk_level, r.relative_velocity, r.position.x,
                     r.position.y, r.position.z] for rs in allr.values() for r in rs]).reshape(-1, 7)
    got = got[np.lexsort((got[:, 1], got[:, 0]))]
    assert_pairs_equal(got[:, :2], want[:, :2])
    assert_close(got[:, 2], want[:, 2], "risk", 1e-6, 1e-7)
    assert_close(got[:, 3], want[:, 4], "rel_speed", 1e-6, 1e-7)
    assert_close(got[:, 4:7], want[:, 5:8], "position", 1e-6, 1e-6)
    # the per-vehicle form with an explicit neighbour set (ComputeNode._detect_collisions_for_all)
    for i in np.unique(want[:, 0].astype(int))[:5]:
        near = index.query_nearby(states[f"v{i}"].get_current_location().position, 100.0)
        assert f"v{i}" in near  # quirk Q8: the index returns the querying vehicle
        rs = det.detect_collisions(states[f"v{i}"], {o: states[o] for o in near})
        assert sorted(int(r.vehicle_id2[1:]) for r in rs) == sorted(int(j) for a, j in want[:, :2] if int(a) == i)
        assert all(abs(r.time_to_collision - t) < 1e-3 for r, t in
                   zip(sorted(rs, key=lambda r: int(r.vehicle_id2[1:])), [w[3] for w in want if int(w[0]) == i]))
    assert index.remove("v0") and not index.remove("v0") and index.get_position("v0") is None


def _oracle_patterns(model, table):
    from oracle import oracle as O
    out = []
    for s in range(table.n):
        h = model.trajectory_history.get(table.ids[s], [])
        out.append(O.pattern([(p.x, p.y, p.z, t) for p, t in h]))
    return np.array(out, np.uint8)


def test_device_trajectory_rings_follow_the_host_histories_and_their_late_samples():
    """update_trajectory feeds ring buffers on the GPU incrementally; the classes must equal the
    oracle's classification of the reference-style host histories through ring wrap-around
    (> 100 samples), vehicle removal (slots are recycled by swap-remove), re-insertion and
    samples that arrive with older timestamps than earlier ones."""
    from rcd_b200.host.collision_detection import CollisionDetector, CollisionPredictionModel
    from rcd_b200.host.models import Position, Vector, Vehicle
    from rcd_b200.host.spatial_index import SpatialIndex
    rng = np.random.default_rng(17)
    det = CollisionDetector(SpatialIndex())
    model = CollisionPredictionModel(det)
    n = 60
    kinds = rng.integers(0, 4, n)  # 0 parked, 1 cruising, 2 accelerating, 3 jittery clock (dt = 0 now and then)
    pos = rng.uniform(0, 500, (n, 3))
    vel = rng.uniform(-8, 8, (n, 3))
    acc = rng.uniform(-1.5, 1.5, (n, 3))

    def vehicle(i, t):
        k = kinds[i]
        v = vel[i] * (k > 0)
        a = acc[i] * (k == 2)
        p = pos[i] + v * t + 0.5 * a * t * t
        return Vehicle(id=f"v{i}", position=Position(*map(float, p)), velocity=Vector(*map(float, v)),
                       acceleration=Vector(*map(float, a)), heading=0.0, size=2.0, type="car", timestamp=t)

    table = det.spatial_index._table
    t = 0.0
    for step in range(130):  # 130 samples > max_history_length = 100: the rings wrap
        t += 0.5 if step % 7 else 0.0  # repeated timestamps (dt = 0) are skipped by the classifier
        for i in range(n):
            if i % 5 == 0 and step < 3:
                continue  # late joiners: some vehicles have fewer than 2 samples at first
            v = vehicle(i, t)
            det.update_vehicle(v)
            model.update_trajectory(v.id, v.position, t)
        if step in (1, 2, 50, 129):
            assert np.array_equal(model.trajectory_patterns(), _oracle_patterns(model, table)), step
        if step == 60:  # remove a few vehicles: the table swap-removes, the rings follow
            for i in (3, 17, 59, 0):
                det.remove_vehicle(f"v{i}")
            assert np.array_equal(model.trajectory_patterns(), _oracle_patterns(model, table))
    assert set(model.trajectory_patterns().tolist()) >= {0, 1, 2}
    assert det.spatial_index._frames.engine_generation == 1
    # predictions use the device-side classes
    some = table.ids[5]
    assert isinstance(model.predict_collisions(some), list)
    # late samples (older timestamps than ones already appended) stay in the device rings, which classify them in
    # timestamp order, as the reference classifies its host histories
    late = [i for i in range(n) if kinds[i] == 2 and f"v{i}" in table.slot_of][:6]
    for back in (3.0, 0.25):
        for i in late:
            v = vehicle(i, t - back)
            model.update_trajectory(v.id, v.position, t - back)
        got = model.trajectory_patterns()
        assert np.array_equal(got, _oracle_patterns(model, table)), back
    assert det.spatial_index._frames.engine_generation == 1
    assert isinstance(model.predict_collisions(some), list)


def test_new_vehicle_in_a_recycled_slot_that_is_moved_in_the_same_tick_keeps_its_own_history():
    """The last vehicle is removed (its ring stays behind), a new vehicle takes that slot, and before the next
    frame another removal swap-moves the new vehicle into the hole: the ring must be rebuilt from the new
    vehicle's own samples at its final slot, not copied from the slot's previous occupant."""
    from rcd_b200.host.collision_detection import CollisionDetector, CollisionPredictionModel
    from rcd_b200.host.models import Position, Vector, Vehicle
    from rcd_b200.host.spatial_index import SpatialIndex
    det = CollisionDetector(SpatialIndex())
    model = CollisionPredictionModel(det)
    table = det.spatial_index._table

    def put(vid, x, vx, ax, t):
        v = Vehicle(id=vid, position=Position(x + vx * t + 0.5 * ax * t * t, 0.0, 0.0), velocity=Vector(vx + ax * t, 0.0, 0.0),
                    acceleration=Vector(ax, 0.0, 0.0), heading=0.0, size=2.0, type="car", timestamp=t)
        det.update_vehicle(v)
        model.update_trajectory(vid, v.position, t)

    for k in range(12):  # five accelerating vehicles with long histories; "x" sits in the last slot
        for j, vid in enumerate(("a", "b", "c", "d", "x")):
            put(vid, 100.0 * j, 3.0, 1.5, 0.5 * k)
    assert np.array_equal(model.trajectory_patterns(), _oracle_patterns(model, table))
    assert model.trajectory_patterns()[table.slot_of["x"]] == 2
    # one tick: x leaves, the parked newcomer takes its slot, b leaves -> the newcomer is swap-moved into b's hole
    det.remove_vehicle("x")
    for k in range(3):
        put("new", 900.0, 0.0, 0.0, 6.0 + 0.5 * k)
    det.remove_vehicle("b")
    assert table.slot_of["new"] == 1
    got = model.trajectory_patterns()
    assert np.array_equal(got, _oracle_patterns(model, table))
    assert got[table.slot_of["new"]] == 0  # stationary: x's accelerating history is gone


def test_pair_helpers_match_the_reference_golden():
    """CollisionDetector._precise_collision_detection / _risk_assessment (collision_detection.py:296-389): the same
    hits, float64 values within a few ulp of the reference's own results (x * x vs pow(x, 2.0), CUDA sin vs
    glibc sin: INTEGRATION.md, "last-ulp deviations"), through rcd_pair_exact / rcd_risk_assessment and through
    the drop-in methods."""
    import json
    import os
    from rcd_b200.host import _native as N
    from rcd_b200.host.collision_detection import CollisionDetector
    from rcd_b200.host.engine import FrameEngine
    from rcd_b200.host.models import Position, Vector, Vehicle
    from rcd_b200.host.spatial_index import SpatialIndex
    from tests.helpers import GOLDEN
    d = json.load(open(os.path.join(GOLDEN, "pair_helpers.json"), encoding="utf-8"))
    f = {k[len("frame_"):]: np.asarray(v) for k, v in d["frame"].items()}
    n = len(f["px"])
    objs = np.zeros(n, dtype=N.OBJECT_DTYPE)
    for k in ("px", "py", "pz", "vx", "vy", "vz", "ax", "ay", "az", "size", "heading"):
        objs[k] = f[k]
    objs["type"] = f["type"]
    cols = ("collision_time", "distance", "safe_distance", "relative_speed", "cx", "cy", "cz", "risk")
    with FrameEngine(16, 16) as e:
        for case in d["cases"]:
            ii = np.array([p[0] for p in case["pairs"]]); jj = np.array([p[1] for p in case["pairs"]])
            got = e.pair_exact(objs[ii], objs[jj], case["T"])
            want_hit = np.array([r is not None for r in case["results"]])
            assert np.array_equal(got["hit"].astype(bool), want_hit)
            want = np.array([r for r in case["results"] if r is not None], np.float64)
            g = got[want_hit]
            assert np.array_equal(g["collision_time"], want[:, 0])  # k * 0.1: the same float64 product
            for c, name in enumerate(cols):
                assert_close(g[name], want[:, c], name, 1e-13, 1e-13)
        # _risk_assessment on collision_info records that did not come from the scan
        rng = np.random.default_rng(3)
        rec = np.stack([rng.uniform(-7, 7, 500), rng.uniform(-7, 7, 500), rng.integers(0, 2, 500).astype(float),
                        rng.uniform(0, 15, 500), rng.uniform(0, 12, 500), rng.uniform(5.5, 10, 500), rng.uniform(0, 80, 500)], 1)
        from oracle import oracle as O
        want = np.array([O.risk_level(r[0], r[1], 0, 0 if r[2] else 1, r[3], r[4], r[5], r[6]) for r in rec])
        assert_close(e.risk_assessment(rec), want, "risk", 1e-13, 1e-15)
    # the drop-in methods (what CollisionPredictionModel._detect_at_position calls, :821-830)
    det = CollisionDetector(SpatialIndex())
    vehicles = [Vehicle(id=f"v{i}", position=Position(float(f["px"][i]), float(f["py"][i]), float(f["pz"][i])),
                        velocity=Vector(float(f["vx"][i]), float(f["vy"][i]), float(f["vz"][i])),
                        acceleration=Vector(float(f["ax"][i]), float(f["ay"][i]), float(f["az"][i])), heading=float(f["heading"][i]),
                        size=float(f["size"][i]), type=f"type{int(f['type'][i])}", timestamp=0.0) for i in range(n)]
    case = d["cases"][1]  # time_window = 1.0: the prediction model's call
    seen = 0
    for (i, j), want in list(zip(case["pairs"], case["results"]))[:150]:
        info = det._precise_collision_detection(vehicles[i], vehicles[j], case["T"])
        assert (info is None) == (want is None)
        if info is None:
            continue
        seen += 1
        assert info["collision_time"] == want[0] and abs(info["distance"] - want[1]) <= 1e-12
        assert abs(det._risk_assessment(vehicles[i], vehicles[j], info) - want[7]) <= 1e-13
    assert seen > 10
