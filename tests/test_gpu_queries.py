"""Listed query sets (rcd_set_queries): a step with query set Q emits exactly the rows i in Q of the same step
without a list, with the totals and per-object counts of Q.  Most checks compare a subset step with the rows of
the full frame on the same upload, which works at any size without the CPU oracle; one frame per mode is also
checked against the oracle.  Uploads carry no ids, so a record's i / j are upload slots."""
import numpy as np
import pytest

from tests.gpu_helpers import compare_pairs
from tests.helpers import f64_frame

pytestmark = pytest.mark.gpu

N_OBJ = 20_000


def _N():
    from rcd_b200.host import _native as N
    return N


def _W():
    from rcd_b200.host import workloads as W
    return W


def _frame(kind, n=N_OBJ, seed=11):
    W = _W()
    if kind == "uniform":
        return W.uniform_frame(n, seed, map_size=3000.0, drone_fraction=0.3)
    return W.hotspot_frame(n, seed, 6000.0, 6, radius_range=(300.0, 700.0))


def _sets(n, seed=5):
    rng = np.random.default_rng(seed)
    return {
        "one": np.array([int(rng.integers(n))], np.uint32),
        "1pct": np.sort(rng.choice(n, n // 100, replace=False)).astype(np.uint32),
        "37pct_shuffled": rng.permutation(rng.choice(n, (37 * n) // 100, replace=False)).astype(np.uint32),
        "all_as_list": rng.permutation(n).astype(np.uint32),
    }


# (mode, radius, window, with_detect, patterns, compute-node parameters)
MODES = {
    "detect": (0, 100.0, 10.0, False, None, None),
    "detect_r60_t4": (0, 60.0, 4.0, False, None, None),
    "predict": (1, 100.0, 10.0, False, "mixed", None),
    "fused": (1, 100.0, 10.0, True, "mixed", None),
    "compute_node": (2, 50.0, 10.0, False, "hist", (2.5, 0.25)),
}


class Result:
    def __init__(self, e):
        self.pairs = e.download()
        self.counts = e.counts()
        self.cand = e.candidate_counts()
        self.risk = e.risk_counts()


def _prepare(e, frame, mode_name, n_owned=None):
    mode, R, T, wd, pat, cn = MODES[mode_name]
    n = len(frame["px"])
    e.upload(frame)
    if pat == "mixed":
        e.set_patterns(_W().random_patterns(n, 8))
    elif pat == "hist":
        e.set_patterns((np.random.default_rng(9).random(n) < 0.7).astype(np.uint8))
    if cn is not None:
        e.set_compute_node_params(*cn)
    if n_owned is not None:
        e.set_owned(n_owned)


def _step(e, mode_name, append=False):
    mode, R, T, wd, _pat, _cn = MODES[mode_name]
    e.step(mode, R, T, append=append, with_detect=wd)
    return Result(e)


def _rows(pairs, q):
    return pairs[np.isin(pairs["i"], np.asarray(q, np.uint32))]


def _check_subset(sub, full, q, n):
    """sub: a step with query set q; full: the same step without a list, on the same upload."""
    q = np.asarray(q, np.int64)
    inq = np.zeros(n, bool)
    inq[q] = True
    want = _rows(full.pairs, q)
    assert sub.pairs.tobytes() == want.tobytes(), "sorted records of the subset"
    c = sub.counts
    assert c["n_owned"] == len(q) and c["n_fallback"] == 0
    assert c["n_pairs"] == len(want)
    assert c["n_high_risk"] == int((want["risk"].astype(np.float64) > 0.7).sum())
    assert c["n_alerts"] == np.bincount(want["priority"][want["priority"] >= 0].astype(np.int64), minlength=4).tolist()
    assert c["n_candidates"] == int(full.cand[q].astype(np.int64).sum())
    assert np.array_equal(sub.cand[:n][inq], full.cand[:n][inq]) and not sub.cand[:n][~inq].any()
    assert np.array_equal(sub.risk[:n][inq], full.risk[:n][inq]) and not sub.risk[:n][~inq].any()


@pytest.fixture(scope="module")
def eng():
    from rcd_b200.host.engine import FrameEngine
    e = FrameEngine(max_objects=60_000, max_pairs=4_000_000)
    yield e
    e.close()


# ---- 1. modes x sets ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["uniform", "hotspot"])
@pytest.mark.parametrize("mode_name", list(MODES))
def test_subset_equals_the_rows_of_the_full_frame(eng, kind, mode_name):
    frame = _frame(kind)
    _prepare(eng, frame, mode_name)
    full = _step(eng, mode_name)
    assert full.counts["n_pairs"] > 0 and full.counts["n_pairs"] <= eng.max_pairs
    for name, q in _sets(N_OBJ).items():
        eng.set_queries(q)
        sub = _step(eng, mode_name)
        _check_subset(sub, full, q, N_OBJ)
        if name == "all_as_list":
            for k in ("n_candidates", "n_potential", "n_pairs", "n_high_risk", "n_alerts", "n_owned", "n_written"):
                assert sub.counts[k] == full.counts[k], k
            assert sub.pairs.tobytes() == full.pairs.tobytes()
    eng.set_queries(None)
    again = _step(eng, mode_name)
    assert again.pairs.tobytes() == full.pairs.tobytes() and again.counts == full.counts


# ---- 2. the oracle, filtered by i in Q ----------------------------------------------------------------------------
@pytest.mark.parametrize("mode_name", ["detect", "predict", "compute_node"])
def test_subset_against_the_oracle(eng, mode_name):
    from oracle import oracle as O
    n = 6000
    frame = _W().uniform_frame(n, 21, map_size=1500.0, drone_fraction=0.3)
    q = _sets(n, 6)["37pct_shuffled"]
    _prepare(eng, frame, mode_name)
    eng.set_queries(q)
    got = _step(eng, mode_name)
    mode, R, T, _wd, pat, cn = MODES[mode_name]
    if mode_name == "compute_node":
        hist = (np.random.default_rng(9).random(n) < 0.7)
        ora = O.frame_B(f64_frame(frame), hist, radius=R, prediction_time=cn[0], risk_threshold=cn[1])
    elif mode_name == "predict":
        ora = O.frame_A(f64_frame(frame), "predict", pattern_codes=_W().random_patterns(n, 8))
    else:
        ora = O.frame_A(f64_frame(frame), "detect", R=R, T=T)
    risks = ora["risks"][np.isin(ora["risks"]["i"], q)]
    compare_pairs(got.pairs, risks, mode_name)
    c = got.counts
    assert c["n_pairs"] == len(risks) and c["n_owned"] == len(q) and c["n_fallback"] == 0
    inq = np.zeros(n, bool)
    inq[q] = True
    if mode_name != "predict":  # (predict frames count candidates of pattern-3 objects only)
        assert np.array_equal(got.cand[:n][inq], ora["cand_count"][inq]) and not got.cand[:n][~inq].any()
        assert c["n_candidates"] == int(ora["cand_count"][inq].astype(np.int64).sum())
    if mode_name == "detect":
        assert c["n_potential"] == int(np.isin(ora["potentials"]["i"], q).sum())
    if mode_name != "compute_node":
        assert c["n_high_risk"] == int((risks["risk"] > 0.7).sum())
        assert c["n_alerts"] == np.bincount(risks["priority"][risks["priority"] >= 0], minlength=4).tolist()


# ---- 3. one index, many sets --------------------------------------------------------------------------------------
def test_new_sets_reuse_the_index():
    from rcd_b200.host.engine import FrameEngine
    frame = _frame("hotspot")
    sets = _sets(N_OBJ, 7)
    with FrameEngine(N_OBJ, 4_000_000, profile=True) as e:
        _prepare(e, frame, "detect")
        full = _step(e, "detect")
        launches, sort_ms = [], []
        for name in ("1pct", "37pct_shuffled", "one"):
            e.set_queries(sets[name])
            e.step(0, 100.0, 10.0)
            launches.append(e.launch_count())
            st = e.stage_ms(0)
            sort_ms.append((st["keys"], st["sort"], st["reorder"], st["qorder"]))
            _check_subset(Result(e), full, sets[name], N_OBJ)
        e.set_queries(None)
        nolist = _step(e, "detect")
        assert nolist.pairs.tobytes() == full.pairs.tobytes() and nolist.counts == full.counts
        # the first list builds the slot -> cell-position map once; later sets reuse it and the index
        assert launches[1] == launches[2] == launches[0] - 1
        for keys, sort, reorder, qorder in sort_ms:
            assert keys == sort == reorder == 0.0 and qorder > 0.0
        # a new upload with a list in force would need a rebuilt index: after rcd_invalidate the list stays
        e.set_queries(sets["1pct"])
        e.invalidate()
        e.step(0, 100.0, 10.0)
        assert e.stage_ms(0)["sort"] > 0.0
        _check_subset(Result(e), full, sets["1pct"], N_OBJ)


# ---- 4. halo ----------------------------------------------------------------------------------------------------
def test_listed_queries_with_halo_objects(eng):
    N = _N()
    frame = _frame("uniform")
    k = 15_000
    _prepare(eng, frame, "detect", n_owned=k)
    full = _step(eng, "detect")
    q = np.random.default_rng(3).choice(k, 3000, replace=False).astype(np.uint32)
    eng.set_queries(q)
    sub = _step(eng, "detect")
    _check_subset(sub, full, q, N_OBJ)
    assert (sub.pairs["j"] >= k).any() and (sub.pairs["i"] < k).all()
    with pytest.raises(N.NativeError) as ex:
        eng.set_queries(np.array([1, k], np.uint32))
    assert ex.value.code == N.RCD_EINVAL and "rcd_set_queries" in str(ex.value)


# ---- 5. validation, 7. device lists ------------------------------------------------------------------------------
def test_bad_lists_keep_the_previous_set_and_device_lists_match_host_lists(eng):
    import torch
    N = _N()
    frame = _frame("uniform")
    _prepare(eng, frame, "detect")
    full = _step(eng, "detect")
    q = _sets(N_OBJ, 8)["1pct"]
    eng.set_queries(q)
    first = _step(eng, "detect")
    _check_subset(first, full, q, N_OBJ)
    bad = [np.array([3, 9, 3], np.uint32), np.array([5, N_OBJ], np.uint32), np.array([0, 0xffffffff], np.uint32)]
    for b in bad:
        with pytest.raises(N.NativeError) as ex:
            eng.set_queries(b)
        assert ex.value.code == N.RCD_EINVAL and "rcd_set_queries" in str(ex.value)
        t = torch.from_numpy(b.astype(np.int64).astype(np.uint32).view(np.int32)).cuda()
        with pytest.raises(N.NativeError) as ex:
            eng.set_queries_device(len(b), t.data_ptr())
        assert ex.value.code == N.RCD_EINVAL and "rcd_set_queries" in str(ex.value)
        torch.cuda.synchronize()
        again = _step(eng, "detect")
        assert again.pairs.tobytes() == first.pairs.tobytes() and again.counts == first.counts
    q2 = _sets(N_OBJ, 9)["37pct_shuffled"]
    t = torch.from_numpy(q2.view(np.int32)).cuda()
    torch.cuda.synchronize()
    eng.set_queries_device(len(q2), t.data_ptr())
    dev = _step(eng, "detect")
    eng.set_queries(q2)
    host = _step(eng, "detect")
    assert dev.pairs.tobytes() == host.pairs.tobytes() and dev.counts == host.counts
    _check_subset(dev, full, q2, N_OBJ)
    eng.set_queries(np.zeros(0, np.uint32))  # an empty set: nothing is queried
    empty = _step(eng, "detect")
    assert empty.counts["n_owned"] == 0 and empty.counts["n_pairs"] == 0 and len(empty.pairs) == 0


# ---- 6. lifetime ---------------------------------------------------------------------------------------------------
def test_lifetime_of_a_set(eng):
    import torch
    N = _N()
    frame = _frame("uniform")
    n = N_OBJ
    q = _sets(n, 10)["1pct"]
    _prepare(eng, frame, "detect")
    full = _step(eng, "detect")

    def listed():
        return eng.counts()["n_owned"] == len(q)

    def stepped():
        eng.step(0, 100.0, 10.0)
        return listed()

    # resets: upload, set_owned, truncate
    for reset in (lambda: eng.upload(frame), lambda: eng.set_owned(n), lambda: eng.truncate(n)):
        eng.set_queries(q)
        assert stepped()
        reset()
        assert not stepped() and eng.counts()["n_owned"] == n
    # keeps: set_patterns, invalidate, set_compute_node_params, apply_records (grows the frame), halo_append
    eng.set_queries(q)
    eng.set_patterns(None)
    assert stepped()
    _check_subset(Result(eng), full, q, n)
    eng.invalidate()
    assert stepped()
    eng.set_compute_node_params(5.0, 0.5)
    assert stepped()
    rec = np.zeros(1, N.RECORD_DTYPE)
    s = int(q[0])
    rec[0] = (frame["px"][s], frame["py"][s], frame["pz"][s], 0.0, frame["vx"][s], frame["vy"][s], frame["vz"][s],
              frame["ax"][s], frame["ay"][s], frame["az"][s], frame["size"][s], frame["heading"][s], s,
              frame["type"][s], 0, 0)
    eng.apply_records(rec, n + 10, history=False)  # ten fresh slots at the end
    assert stepped()
    assert (Result(eng).pairs["i"] < n).all()
    eng.truncate(n)
    eng.set_queries(q)
    halo = np.zeros((5, N.HALO_RECORD_WORDS), np.uint32)
    for r in range(5):
        src = int(q[r])  # a faster twin of a queried object: it must show up as a neighbour of its original
        for k, f in enumerate(("px", "py", "pz", "vx", "vy", "vz", "ax", "ay", "az", "size", "heading")):
            halo[r, k] = np.float32(frame[f][src] + (5.0 if f == "vx" else 0.0)).view(np.uint32)
        halo[r, 11] = int(frame["type"][src]) | (2 << 8)
        halo[r, 12] = n + r
    t = torch.from_numpy(halo.view(np.int32)).cuda()
    torch.cuda.synchronize()
    eng.halo_append(t.data_ptr(), 5)
    assert stepped()
    got = Result(eng).pairs
    assert np.isin(got["i"], q).all() and (got["j"] >= n).any()
    # set_queries ends the frame
    eng.truncate(n)
    eng.step(0, 100.0, 10.0)
    eng.set_queries(q)
    with pytest.raises(N.NativeError) as ex:
        eng.step(1, 100.0, 10.0, append=True)
    assert ex.value.code == N.RCD_ESTATE


# ---- 8. graph replay -----------------------------------------------------------------------------------------------
def test_graph_replay_with_lists():
    from rcd_b200.host.engine import FrameEngine
    frame = _frame("hotspot")
    bounds = ((0.0, 0.0, 0.0), (6000.0, 6000.0, 100.0))
    rng = np.random.default_rng(12)
    sets = [np.sort(rng.choice(N_OBJ, 500, replace=False)).astype(np.uint32) for _ in range(6)]
    with FrameEngine(N_OBJ, 4_000_000, world_bounds=bounds) as ref, \
            FrameEngine(N_OBJ, 4_000_000, world_bounds=bounds, graph=True) as g:
        for e in (ref, g):
            _prepare(e, frame, "fused")
        full = _step(ref, "fused")
        plan = sets + [None, sets[0], None, None, sets[1], sets[2], None]
        for q in plan:
            g.set_queries(q)
            got = _step(g, "fused")
            if q is None:
                assert got.pairs.tobytes() == full.pairs.tobytes() and got.counts == full.counts
            else:
                _check_subset(got, full, q, N_OBJ)
        assert g.graph_replays() >= 4


# ---- 9. overflow ---------------------------------------------------------------------------------------------------
def test_overflow_with_a_subset(eng):
    from rcd_b200.host.engine import FrameEngine
    frame = _frame("hotspot")
    q = _sets(N_OBJ, 13)["37pct_shuffled"]
    for mode_name in ("detect", "fused"):
        _prepare(eng, frame, mode_name)
        full = _step(eng, mode_name)
        with FrameEngine(N_OBJ, 64) as small:
            _prepare(small, frame, mode_name)
            small.set_queries(q)
            got = _step(small, mode_name)
        want = _rows(full.pairs, q)
        c = got.counts
        assert c["n_pairs"] == len(want) > 64 and c["n_written"] == 64 and c["n_fallback"] == 0
        assert c["n_candidates"] == int(full.cand[q].astype(np.int64).sum())
        assert np.array_equal(got.risk, np.where(np.isin(np.arange(N_OBJ), q), full.risk[:N_OBJ], 0))
        assert np.array_equal(got.cand[:N_OBJ], np.where(np.isin(np.arange(N_OBJ), q), full.cand[:N_OBJ], 0))
        assert c["n_high_risk"] == int((want["risk"].astype(np.float64) > 0.7).sum())
        assert np.isin(got.pairs["i"], q).all()
        wanted = {r.tobytes() for r in want}
        assert all(r.tobytes() in wanted for r in got.pairs)


# ---- 10. summary delivery ------------------------------------------------------------------------------------------
def test_summary_with_a_subset_matches_the_filtered_pairs():
    from rcd_b200.host.engine import FrameEngine
    frame = _frame("uniform")
    q = _sets(N_OBJ, 14)["37pct_shuffled"]
    with FrameEngine(N_OBJ, 4_000_000) as a, FrameEngine(N_OBJ, 4_000_000) as b:
        for e in (a, b):
            _prepare(e, frame, "fused")
            e.alerts_configure(1_000_000)
        full = _step(b, "fused")
        want_ev, want_st = b.alerts_update_pairs(_rows(full.pairs, q), 1.0)
        a.set_queries(q)
        a.step(1, 100.0, 10.0, with_detect=True)
        a.summary_begin(1.0)
        ev, st, risk, counts = a.summary_finish(risk_counts=np.zeros(N_OBJ, np.uint32))
        assert counts["n_owned"] == len(q) and counts["n_pairs"] == len(_rows(full.pairs, q))
        assert np.array_equal(risk, np.where(np.isin(np.arange(N_OBJ), q), full.risk[:N_OBJ], 0))
        key = ("i", "j", "risk", "ttc", "distance", "priority", "old_priority", "kind")

        def table(e):
            e = np.sort(e, order=["i", "j"])
            return [tuple(r[k] for k in key) for r in e]
        assert len(ev) == len(want_ev) > 0 and table(ev) == table(want_ev)
        for k in ("n_events", "n_created", "n_changed", "n_live"):
            assert st[k] == want_st[k], k


# ---- 11. the bench frame -------------------------------------------------------------------------------------------
def test_bench_frame_one_percent():
    from rcd_b200.host.engine import FrameEngine
    n = 1_000_000
    frame = _W().hotspot_frame(n, 2002, 31623.0, 50)
    bounds = ((0.0, 0.0, 0.0), (31623.0, 31623.0, 100.0))
    q = np.random.default_rng(15).choice(n, n // 100, replace=False).astype(np.uint32)
    with FrameEngine(n, 60_000_000, world_bounds=bounds) as e:
        e.upload(frame)
        e.step(1, 100.0, 10.0, with_detect=True)
        full = Result(e)
        assert full.counts["n_pairs"] <= e.max_pairs
        e.set_queries(q)
        e.step(1, 100.0, 10.0, with_detect=True)
        sub = Result(e)
    _check_subset(sub, full, q, n)


# ---- 12. drop-in ---------------------------------------------------------------------------------------------------
def _vehicles(frame):
    from rcd_b200.host.models import Position, Vector, Vehicle
    return [Vehicle(id=f"v{i}", position=Position(float(frame["px"][i]), float(frame["py"][i]), float(frame["pz"][i])),
                    velocity=Vector(float(frame["vx"][i]), float(frame["vy"][i]), float(frame["vz"][i])),
                    acceleration=Vector(float(frame["ax"][i]), float(frame["ay"][i]), float(frame["az"][i])),
                    heading=float(frame["heading"][i]), size=float(frame["size"][i]),
                    type=f"type{int(frame['type'][i])}", timestamp=0.0) for i in range(len(frame["px"]))]


def _tables(d):
    return {k: v.table.tobytes() for k, v in d.items()}


def test_detect_for_and_predict_for():
    from rcd_b200.host.collision_detection import CollisionDetector, CollisionPredictionModel
    from rcd_b200.host.models import Position
    from rcd_b200.host.spatial_index import SpatialIndex
    n = 3000
    frame = _W().uniform_frame(n, 31, map_size=1200.0)
    ids = [f"v{i}" for i in np.random.default_rng(16).choice(n, 400, replace=False)] + ["nobody", "v1", "v1"]
    known = {v for v in ids if v != "nobody"}

    def fresh():
        det = CollisionDetector(SpatialIndex())
        det.update_vehicles_batch(_vehicles(frame))
        model = CollisionPredictionModel(det)
        for r in range(3):  # histories of three samples: constant-velocity / accelerating patterns
            for i in range(0, n, 2):
                model.update_trajectory(f"v{i}", Position(float(frame["px"][i]) + r, float(frame["py"][i]), 0.0), float(r))
        return det, model

    # the whole frame is memoised: no GPU work
    det, model = fresh()
    frames = det.spatial_index._frames
    all_d = det.detect_all(60.0, 4.0)
    for_d = det.detect_for(ids, 60.0, 4.0)
    assert frames.frames_run == 1
    all_p = model.predict_all()
    for_p = model.predict_for(ids)
    assert frames.frames_run == 2
    assert _tables(for_d) == {k: v for k, v in _tables(all_d).items() if k in known}
    assert _tables(for_p) == {k: v for k, v in _tables(all_p).items() if k in known}
    assert len(for_d) > 0 and len(for_p) > 0
    # nothing memoised: one frame over the listed vehicles only, memoised per set
    det, model = fresh()
    frames = det.spatial_index._frames
    for_d = det.detect_for(ids, 60.0, 4.0)
    assert frames.frames_run == 1 and frames.engine.counts()["n_owned"] == len(known)
    assert _tables(det.detect_for(list(reversed(ids)), 60.0, 4.0)) == _tables(for_d) and frames.frames_run == 1
    assert _tables(for_d) == {k: v for k, v in _tables(det.detect_all(60.0, 4.0)).items() if k in known}
    for_p = model.predict_for(ids)
    assert frames.frames_run == 3 and frames.engine.counts()["n_owned"] == len(known)
    assert _tables(for_p) == {k: v for k, v in _tables(model.predict_all()).items() if k in known}
    assert det.detect_for(["nobody"]) == {}
    # the per-vehicle calls keep their whole-frame behaviour
    vid = sorted(known)[0]
    assert [r.other_vehicle_id for r in det.detect_collisions(vid, 60.0, 4.0)] == \
        [r.other_vehicle_id for r in for_d.get(vid, [])]
