"""Compute-node mode (RCD_MODE_COMPUTE_NODE: SpatialIndex.query_nearby + CollisionDetector.detect_collisions,
src/compute/compute_node.py:98-119, 229-321) against the float64 oracle (oracle.frame_B) across its parameters,
its threshold ties and the paths a frame can take: far-from-origin coordinates, halo objects, one-cell grids,
overflowing queues, graph replay and mode switches on one handle.

Every parameter value here is exactly representable in fp32 (rcd_set_compute_node_params and rcd_step take
floats), so the oracle sees exactly what the device sees."""
import numpy as np
import pytest

from tests.gpu_helpers import compare_counts, compare_pairs
from tests.helpers import f64_frame

pytestmark = pytest.mark.gpu


def _oracle():
    from oracle import oracle as O
    return O


def _W():
    from rcd_b200.host import workloads as W
    return W


def _side(n, density):
    """Side of a square map holding n objects at `density` objects per m^2."""
    return max(40.0, float(np.sqrt(n / density)))


def _hist(n, frac, seed):
    return (np.random.default_rng(seed).random(n) < frac).astype(np.uint8)


def _check_records(got):
    """The fields compare_pairs leaves out in this mode: no alert class, no offset, no stage-2 values."""
    assert (got["priority"] == -1).all(), "compute-node records carry no alert class"
    assert (got["offset"] == 255).all() and (got["predicted"] == 0).all()
    assert (got["t_closest"] == 0).all() and (got["d_closest"] == 0).all()


def _run(e, frame, hist, R=100.0, pt=5.0, thr=0.5):
    e.upload(frame)
    e.set_patterns(hist)
    e.set_compute_node_params(pt, thr)
    return e.compute_node(R)


def _frame_B(frame, hist, R=100.0, pt=5.0, thr=0.5):
    # has_history: any non-zero code (the device packs the code; only 0 means "fewer than two samples")
    return _oracle().frame_B(f64_frame(frame), np.asarray(hist) != 0, radius=R, prediction_time=pt, risk_threshold=thr)


def _check(e, frame, hist, R=100.0, pt=5.0, thr=0.5):
    """One compute-node frame on `e` against frame_B with the same parameters: pair set bit-exact, values to 1e-6,
    totals, per-object candidate counts (self included, quirk Q8), n_fallback == 0.  Returns (got, oracle)."""
    got = _run(e, frame, hist, R, pt, thr)
    ora = _frame_B(frame, hist, R, pt, thr)
    compare_pairs(got, ora["risks"], "compute_node")
    c = e.counts()
    compare_counts(c, e.candidate_counts(), ora, "compute_node")
    assert c["n_written"] == c["n_pairs"] == len(got)
    _check_records(got)
    return got, ora


def _keys(a):
    return (a["i"].astype(np.int64) << 32) | a["j"].astype(np.int64)


@pytest.fixture(scope="module")
def eng():
    from rcd_b200.host.engine import FrameEngine
    e = FrameEngine(max_objects=110_000, max_pairs=2_000_000)
    yield e
    e.close()


# ---- 1. seeded frames -----------------------------------------------------------------------------------------
def _seeded_frame(kind, n, seed):
    W = _W()
    if kind == "uniform":
        return W.uniform_frame(n, seed, map_size=_side(n, 0.01 if n < 50_000 else 0.004), drone_fraction=0.2)
    side = _side(n, 0.004)
    return W.hotspot_frame(n, seed, side, 3, radius_range=(0.15 * side, 0.3 * side), drone_fraction=0.2)


# (generator, objects, has_history fraction, seed, least number of emitted pairs)
SEEDED = [
    ("uniform", 1, 1.0, 1, 0),
    ("uniform", 31, 1.0, 2, 2),
    ("uniform", 2049, 0.5, 3, 40),
    ("hotspot", 4097, 1.0, 4, 200),
    ("uniform", 20000, 0.0, 5, 0),
    ("hotspot", 20000, 0.5, 6, 300),
    ("uniform", 100_000, 1.0, 7, 3000),
]


@pytest.mark.parametrize("kind,n,frac,seed,min_pairs", SEEDED)
def test_seeded_frames(eng, kind, n, frac, seed, min_pairs):
    frame = _seeded_frame(kind, n, seed)
    hist = _hist(n, frac, seed + 1000)
    got, ora = _check(eng, frame, hist)
    assert len(got) >= min_pairs
    c = eng.counts()
    assert c["n_objects"] == c["n_owned"] == n
    assert c["n_candidates"] >= n  # every object finds itself
    if frac == 0.0:
        assert c["n_pairs"] == 0 and c["n_candidates"] > 3 * n  # candidates are still counted
    if 0.0 < frac < 1.0:  # no pair involves an object without history
        assert hist[got["i"]].all() and hist[got["j"]].all()


def test_history_codes_1_2_3_all_mean_has_history(eng):
    """The pattern byte is the has-history flag in this mode: 1, 2 and 3 all mean >= 2 samples."""
    n = 6000
    frame = _seeded_frame("uniform", n, 11)
    codes = np.random.default_rng(12).choice(4, size=n, p=(0.2, 0.2, 0.2, 0.4)).astype(np.uint8)
    got, _ = _check(eng, frame, codes)
    assert len(got) > 100 and (codes[got["i"]] == 3).sum() > 20 and (codes[got["j"]] == 3).sum() > 20
    ones = _run(eng, frame, (codes != 0).astype(np.uint8))
    assert ones.tobytes() == got.tobytes()


# ---- 2. parameter grid ----------------------------------------------------------------------------------------
PREDICTION_TIMES = [0.0, 0.5, 5.0, 30.0]
THRESHOLDS = [-1.0, 0.0, 0.25, 0.5, 1.0, 1.5]
RADII = [10.0, 37.5, 50.0, 100.0, 250.0]
N_GRID = 2000


def _grid_frame():
    """2000 objects on a 300 m map (~170 within 50 m of each), plus
    - pairs with rs = 0: coincident objects with equal velocities (cur = fut = 0) and a convoy (equal velocities,
      3 m apart: fut = cur), risk 0;
    - for every prediction time, 6 pairs 8 m apart that meet at that time (fut ~ 0: risk 1 whatever the radius),
      and for pt = 0, 6 pairs 2 m apart closing at 10 m/s (fut = cur = 2: risk 1)."""
    W = _W()
    f = W.uniform_frame(N_GRID, 21, map_size=300.0, drone_fraction=0.2)
    for k in ("px", "py", "pz", "vx", "vy", "vz"):
        f[k][1:4] = f[k][0]      # objects 0..3: one place, one velocity
        f[k][11:14] = f[k][10]   # objects 10..13: the convoy
    f["px"][11:14] = f["px"][10] + np.float32(3.0) * np.arange(1, 4, dtype=np.float32)
    rng = np.random.default_rng(23)
    a = 20
    for pt in PREDICTION_TIMES:
        for _ in range(6):
            u = rng.normal(size=3)
            u[2] *= 0.2
            u /= np.linalg.norm(u)
            p, v = np.array([f[k][a] for k in ("px", "py", "pz")], np.float64), np.array([f[k][a] for k in ("vx", "vy", "vz")])
            d = (8.0 if pt else 2.0) * u
            w = v - d / pt if pt else v - 10.0 * u
            for c, k in enumerate(("px", "py", "pz")):
                f[k][a + 1] = p[c] + d[c]
            for c, k in enumerate(("vx", "vy", "vz")):
                f[k][a + 1] = w[c]
            a += 2
    return f, _hist(N_GRID, 0.9, 22) | (np.arange(N_GRID) < a).astype(np.uint8)


@pytest.fixture(scope="module")
def grid_frame():
    return _grid_frame()


@pytest.mark.parametrize("pt", PREDICTION_TIMES)
@pytest.mark.parametrize("thr", THRESHOLDS)
def test_parameter_grid(eng, grid_frame, pt, thr):
    frame, hist = grid_frame
    for R in RADII:
        got, ora = _check(eng, frame, hist, R, pt, thr)
        c = eng.counts()
        assert c["n_candidates"] > 3 * N_GRID, R
        keys = set(_keys(got).tolist())
        rs0 = [(0, 1), (1, 0), (2, 3), (10, 11), (11, 10)]  # risk 0: kept exactly when thr <= 0
        assert all((((i << 32) | j) in keys) == (thr <= 0.0) for i, j in rs0), (R, pt, thr)
        if thr > 1.0:  # min(1, rl) < thr for every pair: nothing is emitted, candidates are still counted
            assert c["n_pairs"] == 0
            continue
        assert len(got) >= 12, (R, pt, thr)  # at least the 6 pairs (both directions) planted for this pt
        if thr == 1.0:  # only risks capped at exactly 1.0 survive the strict comparison
            assert (got["risk"] == 1.0).all()
        if pt == 0.0:  # fut == cur: never "moving apart", and the time to collision is prediction_time = 0
            assert (got["ttc"] == 0.0).all()


# ---- 3. pairs placed exactly on the thresholds ---------------------------------------------------------------
# (name, prediction_time, risk_threshold, search_radius, A, B, emitted, expected values of the emitted record)
# A, B = (x, y, z, vx, vy, vz) relative to the pair's base point.  Integer / half-integer / 1/16 values only, so every
# fp64 quantity (cur, fut, rs, rl) is exact and lands on the threshold itself; both directions behave alike.
Z = (0.0, 0.0, 0.0)
TIES = [
    # current_distance > 50 (:262): 50 itself stays
    ("cur == 50", 1.0, 0.5, 100.0, (0, 0, 0, 30, 40, 0), (30, 40, 0) + Z, True, {"distance": 0.0, "risk": 1.0}),
    ("cur == 50, 3-D", 1.0, 0.5, 100.0, (0, 0, 0, 24, 30, 32), (24, 30, 32) + Z, True, {"risk": 1.0}),
    ("cur > 50", 1.0, 0.5, 100.0, (0, 0, 0, 30, 40.5, 0), (30, 40.5, 0) + Z, False, None),
    # moving apart (:284): fut > cur and cur > 4
    ("fut == cur", 1.0, 0.5, 100.0, (0, 0, 0) + Z, (3, 4, 0, -6, -8, 0), True, {"distance": 5.0, "risk": 0.8}),
    ("fut > cur", 1.0, 0.5, 100.0, (0, 0, 0) + Z, (3, 4, 0, -6.5, -8, 0), False, None),
    ("cur == 4, apart", 0.5, 0.5, 100.0, (0, 0, 0) + Z, (4, 0, 0, 20, 0, 0), True, {"distance": 14.0, "ttc": 0.5}),
    ("cur == 4.5, apart", 0.5, 0.5, 100.0, (0, 0, 0) + Z, (4.5, 0, 0, 20, 0, 0), False, None),
    # time to collision (:296-301): fut < 4 and cur > fut
    ("fut == 4", 1.0, 0.5, 100.0, (0, 0, 0) + Z, (10, 0, 0, -6, 0, 0), True, {"ttc": 1.0, "risk": 0.6}),
    ("fut < 4", 1.0, 0.5, 100.0, (0, 0, 0) + Z, (10, 0, 0, -7, 0, 0), True, {"ttc": 6.0 / 7.0, "distance": 3.0}),
    ("ratio < 0.1", 1.0, 0.5, 100.0, (0, 0, 0) + Z, (4.25, 0, 0, -4.25, 0, 0), True, {"ttc": 0.1, "risk": 1.0}),
    ("cur < 4, ratio < 0", 1.0, 0.5, 100.0, (0, 0, 0) + Z, (3, 0, 0, -2, 0, 0), True, {"ttc": 0.1, "risk": 0.8}),
    ("cur < fut < 4", 1.0, 0.0, 100.0, (0, 0, 0) + Z, (2, 0, 0, 1, 0, 0), True, {"ttc": 1.0, "distance": 3.0}),
    # min_distance = max(0.1, fut) (:288)
    ("fut < 0.1", 1.0, 0.5, 100.0, (0, 0, 0) + Z, (10, 0, 0, -9.9375, 0, 0), True, {"distance": 0.0625, "risk": 1.0}),
    ("fut == 0, cur < 4", 1.0, 0.5, 100.0, (0, 0, 0) + Z, (0.5, 0, 0, -0.5, 0, 0), True, {"risk": 1.0, "ttc": 0.1}),
    # risk < threshold (:292) is strict
    ("risk == 0.5", 1.0, 0.5, 100.0, (0, 0, 0) + Z, (18, 0, 0, -10, 0, 0), True, {"risk": 0.5, "distance": 8.0}),
    ("risk < 0.5", 1.0, 0.5, 100.0, (0, 0, 0) + Z, (18.5, 0, 0, -10, 0, 0), False, None),
    ("risk == 1 at thr 1", 1.0, 1.0, 100.0, (0, 0, 0) + Z, (14, 0, 0, -10, 0, 0), True, {"risk": 1.0, "ttc": 1.0}),
    ("risk < 1 at thr 1", 1.0, 1.0, 100.0, (0, 0, 0) + Z, (14, 0, 0, -9.5, 0, 0), False, None),
    ("risk == 0.25", 2.5, 0.25, 37.5, (0, 0, 0) + Z, (20.5, 0, 0, -5, 0, 0), True, {"risk": 0.25, "distance": 8.0}),
    ("rs == 0 at thr 0", 5.0, 0.0, 100.0, (0, 0, 0, 5, 0, 0), (3, 0, 0, 5, 0, 0), True, {"risk": 0.0, "distance": 3.0}),
    ("rs == 0 at thr 0.25", 5.0, 0.25, 100.0, (0, 0, 0, 5, 0, 0), (3, 0, 0, 5, 0, 0), False, None),
    # the search radius (query_nearby, :113-116): distance <= radius
    ("cur == R == 37.5", 2.5, 0.25, 37.5, (0, 0, 0, 9, 12, 0), (22.5, 30, 0) + Z, True, {"risk": 1.0}),
    ("cur > R == 37.5", 2.5, 0.25, 37.5, (0, 0, 0, 9, 12, 0), (22.5, 30.5, 0) + Z, False, None),
    ("cur == R == 50", 5.0, 0.5, 50.0, (0, 0, 0, 6, 8, 0), (30, 40, 0) + Z, True, {"risk": 1.0, "ttc": 4.6}),
    ("cur == R == 10, pt 0", 0.0, 0.5, 10.0, (0, 0, 0) + Z, (6, 8, 0, 0, 0, 20), True, {"distance": 10.0, "ttc": 0.0}),
    ("cur > R == 10, pt 0", 0.0, 0.5, 10.0, (0, 0, 0) + Z, (6, 8.5, 0, 0, 0, 20), False, None),
    ("cur == 4, pt 0", 0.0, 0.5, 10.0, (0, 0, 0) + Z, (0, 4, 0, 0, 0, 20), True, {"distance": 4.0, "ttc": 0.0}),
]


def _tie_frame(cases, seed):
    """Each case's pair on its own base point 500 m apart (so the pairs never meet), among random objects
    (moving, some without history) that share the neighbourhood."""
    W = _W()
    nb = 60
    objs, bases = [], []
    for k, case in enumerate(cases):
        base = np.array([100.0 + 500.0 * k, 200.0, 10.0])
        bases.append(base)
        for o in (case[4], case[5]):
            objs.append(np.concatenate([base + np.asarray(o[:3], np.float64), np.asarray(o[3:], np.float64)]))
    m = len(objs)
    bg = W.uniform_frame(nb * len(cases), seed, map_size=200.0, drone_fraction=0.5)
    shift = np.repeat(np.array(bases)[:, :2] - 100.0, nb, axis=0)
    f = {k: np.zeros(m + len(bg["px"]), np.float32) for k in bg}
    f["type"] = np.zeros(len(f["px"]), np.uint8)
    for c, k in enumerate(("px", "py", "pz", "vx", "vy", "vz")):
        f[k][:m] = np.array(objs)[:, c]
    for k in bg:
        f[k][m:] = bg[k]
    f["px"][m:] = (bg["px"] + shift[:, 0]).astype(np.float32)
    f["py"][m:] = (bg["py"] + shift[:, 1]).astype(np.float32)
    state = np.stack([f[k][:m] for k in ("px", "py", "pz", "vx", "vy", "vz")], 1).astype(np.float64)
    assert np.array_equal(state, np.array(objs)), "tie objects must be exact in fp32"
    hist = np.ones(len(f["px"]), np.uint8)
    hist[m:] = _hist(len(bg["px"]), 0.8, seed)
    return f, hist


def _tie_groups():
    groups = {}
    for case in TIES:
        groups.setdefault(case[1:4], []).append(case)
    return sorted(groups.items())


@pytest.mark.parametrize("params,cases", _tie_groups(), ids=lambda v: "-".join(map(str, v)) if isinstance(v, tuple) else None)
def test_threshold_ties(eng, params, cases):
    """The fp32 filter must let a pair sitting exactly on a threshold through to the fp64 decision, which keeps or
    drops it exactly as the reference does (the oracle emits these pairs at exactly the threshold)."""
    pt, thr, R = params
    frame, hist = _tie_frame(cases, seed=int(100 * pt + 10 * thr + R))
    got, ora = _check(eng, frame, hist, R, pt, thr)
    okeys = _keys(ora["risks"])
    gkeys = _keys(got)
    for k, (name, *_p, emitted, want) in enumerate(cases):
        for i, j in ((2 * k, 2 * k + 1), (2 * k + 1, 2 * k)):
            key = (i << 32) | j
            assert (key in okeys) == emitted, f"{name}: the case is not on the intended side in the oracle"
            assert (key in gkeys) == emitted, name
            if emitted:
                rec = got[gkeys == key][0]
                for field, v in want.items():
                    assert rec[field] == np.float32(v), (name, field, rec[field], v)


# ---- 4. shapes and paths --------------------------------------------------------------------------------------
def test_far_from_origin_with_and_without_clipping_bounds():
    """90 km coordinates (fp32 ulp 8 mm), with the grid fitted to the data and with static bounds that cover only
    the middle of the map, so most objects are clamped into border cells."""
    from rcd_b200.host.engine import FrameEngine
    n = 6000
    frame = _W().uniform_frame(n, 31, map_size=800.0, drone_fraction=0.3)
    for k in ("px", "py"):
        frame[k] = (frame[k] + np.float32(90000.0)).astype(np.float32)
    hist = _hist(n, 0.8, 32)
    for bounds in (None, ((90300.0, 90300.0, 20.0), (90500.0, 90500.0, 60.0))):
        with FrameEngine(n, 1 << 20, world_bounds=bounds) as e:
            for R, pt, thr in ((100.0, 5.0, 0.5), (37.5, 2.5, 0.25), (250.0, 30.0, 0.0)):
                got, _ = _check(e, frame, hist, R, pt, thr)
                assert len(got) > 100, (bounds, R)


def test_owned_prefix_with_halo_objects():
    """set_owned(k): only objects [0, k) are queried; the halo objects [k, n) are neighbours only -- they still
    appear as j, but have no rows and no candidate count of their own (they are another shard's queries)."""
    from rcd_b200.host.engine import FrameEngine
    n, k = 5000, 3111
    frame = _seeded_frame("uniform", n, 41)
    hist = _hist(n, 0.8, 42)
    ora = _frame_B(frame, hist, 100.0, 5.0, 0.25)
    with FrameEngine(n, 1 << 20) as e:
        e.upload(frame)
        e.set_patterns(hist)
        e.set_compute_node_params(5.0, 0.25)
        e.set_owned(k)
        got = e.compute_node(100.0)
        c = e.counts()
        cand = e.candidate_counts()
    rows = ora["risks"][ora["risks"]["i"] < k]
    compare_pairs(got, rows, "compute_node")
    _check_records(got)
    assert (rows["j"] >= k).sum() > 20 and (got["j"] >= k).sum() == (rows["j"] >= k).sum()
    want_cand = np.concatenate([ora["cand_count"][:k], np.zeros(n - k, np.uint32)])
    owned = {"counts": np.array([want_cand.sum(), 0, len(rows), 0]), "cand_count": want_cand}
    compare_counts(c, cand, owned, "compute_node")
    assert c["n_owned"] == k and c["n_objects"] == n
    assert not cand[k:].any()


def test_radius_1e9_puts_everything_in_one_cell(eng):
    """The radius CollisionDetector.detect_collisions uses (every listed neighbour is a candidate): one cell holds the
    whole frame, every object is a candidate of every other one."""
    n = 3000
    frame = _W().uniform_frame(n, 51, map_size=800.0, drone_fraction=0.3)
    hist = _hist(n, 0.7, 52)
    assert float(np.float32(1.0e9)) == 1.0e9
    got, ora = _check(eng, frame, hist, 1.0e9, 5.0, 0.5)
    assert len(got) > 20
    assert (eng.candidate_counts() == n).all() and eng.counts()["n_candidates"] == n * n


@pytest.mark.parametrize("pt,thr", [(5.0, 0.5), (2.5, 0.0)])
def test_overflowing_pair_buffer_and_queues(pt, thr):
    """max_pairs = 64 beside a large engine: the pair queue of k_pairs and the queue k_narrow -> k_exact (both sized
    from max_pairs) run full, so pairs are finished in place by k_pairs' overflow pass and k_narrow's fallback.
    Totals and per-object risk counts stay exact; every stored record is one of the frame's records."""
    from rcd_b200.host.engine import FrameEngine
    n = 12000
    frame = _W().uniform_frame(n, 61, map_size=520.0, drone_fraction=0.3)  # ~350 objects within 50 m of each
    hist = _hist(n, 0.9, 62)
    with FrameEngine(n, 64) as small, FrameEngine(n, 1 << 22) as big:
        everything, ora = _check(big, frame, hist, 100.0, pt, thr)
        assert len(everything) > (70_000 if thr == 0.0 else 2000)  # thr 0: more Q3 entries than the small queue holds
        part = _run(small, frame, hist, 100.0, pt, thr)
        c, cb = small.counts(), big.counts()
        assert c["n_written"] == 64 == len(part) < c["n_pairs"]
        assert c["n_pairs"] == cb["n_pairs"] == len(ora["risks"])
        assert c["n_candidates"] == cb["n_candidates"] == int(ora["counts"][0]) and c["n_fallback"] == 0
        assert np.array_equal(small.candidate_counts(), ora["cand_count"])
        want_rc = np.bincount(ora["risks"]["i"], minlength=n)
        assert np.array_equal(small.risk_counts(), want_rc) and np.array_equal(big.risk_counts(), want_rc)
        assert np.isin(_keys(part), _keys(everything)).all()
        _check_records(part)
        for r in part:  # the stored records are complete, not just the right keys
            assert r.tobytes() == everything[_keys(everything) == _keys(r[None])[0]][0].tobytes()


def test_graph_replay_follows_parameter_and_radius_changes():
    """RCD_FLAG_GRAPH: compute-node frames replay a captured graph once a step's shape has been seen twice.  The
    parameters and the radius are part of that shape: after set_compute_node_params or a new radius a replay must
    not run with the old values, and a graph captured earlier must serve its own values again."""
    from rcd_b200.host.engine import FrameEngine
    n, side = 4000, 700.0
    bounds = ((0.0, 0.0, 0.0), (side, side, 100.0))
    frames = [_W().uniform_frame(n, 71 + k, map_size=side, drone_fraction=0.3) for k in range(4)]
    hist = _hist(n, 0.9, 75)
    phases = [  # (radius, prediction_time, risk_threshold, frames, least replays in the phase)
        (100.0, 5.0, 0.5, 4, 2),   # first sighting, capture, then replays
        (100.0, 2.5, 0.25, 3, 1),
        (100.0, 5.0, 0.5, 2, 2),   # the first phase's graph again
        (50.0, 5.0, 0.5, 3, 1),
        (37.5, 0.0, 1.0, 3, 1),
    ]
    with FrameEngine(n, 1 << 20, world_bounds=bounds) as ref, FrameEngine(n, 1 << 20, world_bounds=bounds, graph=True) as g:
        step = 0
        for R, pt, thr, nf, least in phases:
            before = g.graph_replays()
            for _ in range(nf):
                f = frames[step % len(frames)]
                step += 1
                want, _ = _check(ref, f, hist, R, pt, thr)
                got = _run(g, f, hist, R, pt, thr)
                assert got.tobytes() == want.tobytes() and g.counts() == ref.counts()
                assert np.array_equal(g.candidate_counts(), ref.candidate_counts())
                assert len(got) > (5 if thr == 1.0 else 50)
            assert g.graph_replays() - before >= least, (R, pt, thr)
        # the same upload stepped again with other parameters: the index stays valid, so these steps have shapes of
        # their own (pair kernels only); each shape is captured on its second sighting and replayed on its third
        g.upload(frames[0]); g.set_patterns(hist)
        before = g.graph_replays()
        for pt, thr in ((5.0, 0.5), (5.0, 0.5), (5.0, 0.5), (30.0, 0.25), (30.0, 0.25), (5.0, 0.5), (30.0, 0.25),
                        (0.5, 0.0)):
            g.set_compute_node_params(pt, thr)
            got = g.compute_node(100.0)
            ora = _frame_B(frames[0], hist, 100.0, pt, thr)
            compare_pairs(got, ora["risks"], "compute_node")
            compare_counts(g.counts(), g.candidate_counts(), ora, "compute_node")
        assert g.graph_replays() - before >= 3


def test_mode_switches_on_one_upload():
    """detect, compute-node, predict and compute-node again on one upload, with set_patterns in between: the pattern /
    has-history byte is packed into the cell-ordered state, so each step must see the latest one."""
    from rcd_b200.host.engine import FrameEngine
    n = 5000
    frame = _seeded_frame("uniform", n, 81)
    pat = _W().random_patterns(n, 82)  # predict codes: 0 = stationary, which would mean "no history" here
    hist1, hist2 = _hist(n, 0.6, 83), _hist(n, 0.9, 84)
    sequence = [  # (pattern bytes set before the step, None: keep; the step)
        (pat, lambda x: x.detect()),
        (hist1, lambda x: x.compute_node(100.0)),
        (pat, lambda x: x.predict()),
        (hist2, lambda x: x.compute_node(100.0)),
        (None, lambda x: x.compute_node(50.0)),  # same patterns, other radius: the index is rebuilt
    ]
    with FrameEngine(n, 1 << 20) as e:
        e.upload(frame)
        current = None
        for codes, step in sequence:
            if codes is not None:
                e.set_patterns(codes)
                current = codes
            got = step(e)
            c, cand = e.counts(), e.candidate_counts()
            with FrameEngine(n, 1 << 20) as f:
                f.upload(frame)
                f.set_patterns(current)
                want = step(f)
                wc, wcand = f.counts(), f.candidate_counts()
            assert got.tobytes() == want.tobytes()
            for key in ("n_pairs", "n_candidates", "n_potential", "n_high_risk", "n_alerts", "n_fallback"):
                assert c[key] == wc[key], key
            assert np.array_equal(cand, wcand)
            assert len(got) > 20
        ora = _frame_B(frame, hist2, 50.0)  # the last frame against the oracle as well
        compare_pairs(got, ora["risks"], "compute_node")
        compare_counts(c, cand, ora, "compute_node")


# ---- 5. the host classes with non-default parameters ---------------------------------------------------------
def test_collision_detector_with_non_default_parameters():
    from rcd_b200.host import compute_node as CN
    from rcd_b200.host.models import LocationData, Position, Vector
    n = 3000
    frame = _seeded_frame("uniform", n, 91)
    hist = _hist(n, 0.8, 92)
    states = {}
    for i in range(n):
        loc = LocationData(vehicle_id=f"v{i}", timestamp=0.0,
                           position=Position(float(frame["px"][i]), float(frame["py"][i]), float(frame["pz"][i])),
                           velocity=Vector(float(frame["vx"][i]), float(frame["vy"][i]), float(frame["vz"][i])),
                           heading=float(frame["heading"][i]), vehicle_type="car")
        st = CN.VehicleState(f"v{i}")
        st.update(loc)
        if hist[i]:
            st.update(loc)
        states[f"v{i}"] = st
    det = CN.CollisionDetector(prediction_time=2.5, risk_threshold=0.25)
    ora = _frame_B(frame, hist, 100.0, 2.5, 0.25)["risks"]
    assert len(ora) > 100

    def table(risks):
        t = np.array([[int(r.vehicle_id1[1:]), int(r.vehicle_id2[1:]), r.risk_level, r.relative_velocity,
                       r.position.x, r.position.y, r.position.z] for r in risks]).reshape(-1, 7)
        return t[np.lexsort((t[:, 1], t[:, 0]))]

    def same(got, want):
        from tests.helpers import assert_close, assert_pairs_equal
        assert_pairs_equal(got[:, :2], np.stack([want["i"], want["j"]], 1))
        assert_close(got[:, 2], want["risk"], "risk", 1e-6, 1e-7)
        assert_close(got[:, 3], want["rel_speed"], "rel_speed", 1e-6, 1e-9)
        for c, k in enumerate(("cx", "cy", "cz")):
            assert_close(got[:, 4 + c], want[k], k, 1e-6, 1e-6)

    allr = det.detect_collisions_for_all(states, 100.0)
    same(table([r for rs in allr.values() for r in rs]), ora)
    # the per-vehicle form (set_owned(1), radius 1e9) against the oracle's rows of that vehicle
    px = np.stack([frame[k].astype(np.float64) for k in ("px", "py", "pz")], 1)
    vehicles = np.unique(ora["i"])[:: max(1, len(np.unique(ora["i"])) // 6)][:6]
    for i in list(vehicles) + [int(np.flatnonzero(hist == 0)[0])]:
        near = np.flatnonzero(np.sqrt(((px - px[i]) ** 2).sum(1)) <= 100.0)
        rs = det.detect_collisions(states[f"v{i}"], {f"v{j}": states[f"v{j}"] for j in near})
        want = ora[ora["i"] == i]
        assert len(rs) == len(want) and (len(want) > 0) == bool(hist[i])
        if len(want):
            same(table(rs), want)
