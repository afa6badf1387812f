"""The CPU oracle (oracle/oracle.c) against the golden vectors that the reference's own bytecode
produced under the shim (tests/golden/make_golden.py).  float64 on both sides, same libm:
everything is compared bit-exactly."""
import numpy as np
import pytest

from oracle import oracle as O
import os

from tests.helpers import GOLDEN, f64_frame, load_golden, oracle_risk_table

DETECT = ["detect_dense3d.npz", "detect_2d_noaccel.npz", "detect_r60_t4.npz", "detect_city1k.npz"]
PREDICT = ["predict_dense3d.npz", "predict_2d_allcv.npz", "predict_city300.npz"]


@pytest.mark.parametrize("name", DETECT)
def test_detect_matches_reference_golden(name):
    z, frame = load_golden(name)
    o = O.frame_A(f64_frame(frame), "detect", R=float(z["R"]), T=float(z["T"]), want_candidates=True)
    assert np.array_equal(o["candidates"], z["candidates"])
    pots = np.stack([o["potentials"][c].astype(np.float64) for c in ("i", "j", "tc", "cd")], 1) \
        if len(o["potentials"]) else np.zeros((0, 4))
    assert np.array_equal(pots, z["potentials"])
    assert np.array_equal(oracle_risk_table(o["risks"]), z["risks"])
    assert o["counts"][0] == len(z["candidates"])
    assert o["counts"][1] == int(z["stat_potential"])
    assert o["counts"][3] == int(z["stat_high"])
    assert np.array_equal(np.bincount(z["candidates"][:, 0], minlength=len(frame["px"])), o["cand_count"])
    assert np.all(o["risks"]["offset"] == -1)


@pytest.mark.parametrize("name", PREDICT)
def test_predict_matches_reference_golden(name):
    z, frame = load_golden(name)
    o = O.frame_A(f64_frame(frame), "predict", pattern_codes=z["pattern"])
    assert np.array_equal(oracle_risk_table(o["risks"]), z["risks"])
    # is_predicted is False exactly for the vehicles that fell back to detect (pattern 3)
    assert np.array_equal(z["is_predicted"], z["pattern"][z["risks"][:, 0].astype(int)] != 3)


def test_threads_do_not_change_results():
    z, frame = load_golden("predict_dense3d.npz")
    a = O.frame_A(f64_frame(frame), "predict", pattern_codes=z["pattern"], threads=1)
    b = O.frame_A(f64_frame(frame), "predict", pattern_codes=z["pattern"], threads=4)
    assert a["risks"].tobytes() == b["risks"].tobytes()
    assert np.array_equal(a["cand_count"], b["cand_count"])


def test_implB_matches_reference_golden():
    z, frame = load_golden("implB_dense.npz")
    o = O.frame_B(f64_frame(frame), z["has_history"])
    assert o["counts"][0] == len(z["candidates"])  # query_nearby returns self too (quirk Q8)
    assert np.array_equal(np.bincount(z["candidates"][:, 0], minlength=len(frame["px"])), o["cand_count"])
    r = o["risks"]
    want = z["risks"]  # i j risk ttc_est rel_speed cx cy cz
    assert len(r) == len(want) > 50
    assert np.array_equal(r["i"], want[:, 0]) and np.array_equal(r["j"], want[:, 1])
    assert np.array_equal(r["risk"], want[:, 2])
    # the dataclass field is wall-clock perturbed (quirk Q10): agree to ~1e-4 s only
    assert np.max(np.abs(r["ttc"] - want[:, 3])) < 1e-3
    assert np.array_equal(r["rel_speed"], want[:, 4])
    assert np.array_equal(np.stack([r["cx"], r["cy"], r["cz"]], 1), want[:, 5:8])


def test_scalar_functions_match_reference_golden():
    z = np.load(os.path.join(GOLDEN, "scalars.npz"))
    # trajectory pattern classes
    off = z["hist_off"]
    got = [O.pattern([tuple(r) for r in z["hist"][off[k]:off[k + 1]]]) for k in range(len(off) - 1)]
    assert got == z["hist_class"].tolist()
    assert set(got) == {0, 1, 2, 3}
    # the same histories through the batch entry point, padded with NaN that must never be read
    lens = np.diff(off)
    staged = np.full((len(lens), int(lens.max()) + 3, 4), np.nan)
    for k in range(len(lens)):
        staged[k, :lens[k]] = z["hist"][off[k]:off[k + 1]]
    assert O.patterns(staged, lens).tolist() == z["hist_class"].tolist()
    # alert gate + priority
    assert [O.priority(r, t) for r, t in z["prio_in"]] == z["prio_out"].tolist()
    # grid ids, all four levels (cell = base / 2**level)
    for lvl in range(4):
        cell = (1000.0 / 2 ** lvl, 1000.0 / 2 ** lvl, 100.0 / 2 ** lvl)
        got = np.array([O.grid_id(*p, cell=cell) for p in z["grid_pts"]])
        assert np.array_equal(got, z[f"grid_l{lvl}"])
    # radius queries incl. self (quirk Q8)
    frame = {k[len("near_frame_"):]: z[k] for k in z.files if k.startswith("near_frame_")}
    res = O.query_radius(f64_frame(frame), z["near_q"], float(z["near_radius"]))
    noff = z["near_off"]
    for k, ids in enumerate(res):
        assert np.array_equal(ids, z["near_ids"][noff[k]:noff[k + 1]])


def test_empty_and_single_object_frames():
    from rcd_b200.host import workloads as W
    for n in (0, 1):
        f = W.frame_to_f64(W.uniform_frame(n, 1))
        for mode in ("detect", "predict"):
            o = O.frame_A(f, mode)
            assert o["counts"].tolist() == [0, 0, 0, 0] and len(o["risks"]) == 0
        assert O.frame_B(f)["counts"][0] == n  # a lone vehicle finds itself


def test_pair_helpers_and_alert_messages_match_the_reference_golden():
    """_precise_collision_detection / _risk_assessment (collision_detection.py:296-389) of the oracle against the
    reference's own bytecode, bit for bit in float64; and the alert message tiers (warning_system.py:313-329),
    byte for byte, of the host mirror."""
    import json
    from oracle import oracle as O
    from rcd_b200.host.warning_system import alert_message
    d = json.load(open(os.path.join(GOLDEN, "pair_helpers.json"), encoding="utf-8"))
    f = {k[len("frame_"):]: np.asarray(v, np.float32).astype(np.float64) for k, v in d["frame"].items()}
    obj = lambda i: [f[k][i] for k in ("px", "py", "pz", "vx", "vy", "vz", "ax", "ay", "az", "size")]
    for case in d["cases"]:
        hits = 0
        for (i, j), want in zip(case["pairs"], case["results"]):
            got = O.precise(obj(i), obj(j), case["T"])
            assert (got is None) == (want is None)
            if want is None:
                continue
            hits += 1
            assert list(got) == want[:7]
            risk = O.risk_level(f["heading"][i], f["heading"][j], int(f["type"][i]), int(f["type"][j]), want[0], want[1], want[2], want[3])
            assert risk == want[7]
        assert hits > 100
    for (risk, other, ttc, dist), text in zip(d["messages"]["cases"], d["messages"]["texts"]):
        assert alert_message(risk, other, ttc, dist) == text
        assert alert_message(risk, other, ttc, dist).encode("utf-8") == text.encode("utf-8")
    assert len(d["messages"]["texts"]) > 200
