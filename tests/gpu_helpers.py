"""Comparison of GPU frames (through the C-ABI) with the CPU oracle."""
from __future__ import annotations

import json

import numpy as np

from tests.helpers import assert_close, assert_pairs_equal

# Emitted values are computed in fp64 on the device and rounded once to fp32, so they agree with
# the float64 reference to ~6e-8 relative; the contract (north_star) is 1e-4.  The tests hold the
# tighter 1e-6 so that a regression to fp32-only arithmetic is caught.
RTOL = 1e-6


def compare_pairs(gpu, ora, mode, rtol=RTOL):
    """gpu: PAIR_DTYPE array sorted by (i, j); ora: oracle RISK_DTYPE array sorted by (i, j)."""
    assert_pairs_equal(np.stack([gpu["i"], gpu["j"]], 1), np.stack([ora["i"], ora["j"]], 1), f"{mode} pair set")
    if len(ora) == 0:
        return
    if mode == "compute_node":
        # prediction_time * (cur - 4) / (cur - fut), clamped to >= 0.1: not on a grid, so rounding both sides to a
        # fixed number of decimals would split values that differ only by the fp32 rounding of the record
        assert_close(gpu["ttc"], ora["ttc"], f"{mode} ttc", rtol, 1e-9)
    else:
        # time_to_collision lies on the k*0.1 (+ m*0.5) grid: equal after rounding to 1e-6
        assert np.array_equal(np.round(gpu["ttc"].astype(np.float64), 5), np.round(ora["ttc"], 5)), f"{mode} ttc"
    assert_close(gpu["distance"], ora["distance"], f"{mode} distance", rtol, 1e-9)
    assert_close(gpu["rel_speed"], ora["rel_speed"], f"{mode} rel_speed", rtol, 1e-9)
    assert_close(gpu["risk"], ora["risk"], f"{mode} risk", rtol, 1e-7)
    for c in ("cx", "cy", "cz"):
        assert_close(gpu[c], ora[c], f"{mode} {c}", rtol, 1e-6)
    if mode != "compute_node":
        assert np.array_equal(gpu["priority"].astype(np.int32), ora["priority"]), f"{mode} alert priority"
    if mode == "predict":
        pred = ora["offset"] >= 0
        assert np.array_equal(gpu["predicted"].astype(bool), pred)
        assert np.array_equal(gpu["offset"][pred].astype(np.int32), ora["offset"][pred])


def compare_counts(counts, cand_count, ora, mode, candidates=True):
    """candidates=False: predict frames stepped without RCD_FLAG_COUNT_PREDICT_CANDIDATES."""
    # pairs settled in fp32 are never contradicted by the fp64 stage: the guard bands hold
    assert counts.get("n_fallback", 0) == 0, "fp32-resolved pair had to be redone in fp64"
    if candidates:
        assert counts["n_candidates"] == int(ora["counts"][0]), f"{mode} candidate total"
        assert np.array_equal(cand_count[: len(ora["cand_count"])], ora["cand_count"]), f"{mode} per-object candidates"
    assert counts["n_pairs"] == int(ora["counts"][2]), f"{mode} pair total"
    if mode == "detect":
        assert counts["n_potential"] == int(ora["counts"][1]), "potential_collisions"
    if mode != "compute_node":
        assert counts["n_high_risk"] == int(ora["counts"][3]), "high_risk_collisions"
        prio = np.bincount(ora["risks"]["priority"][ora["risks"]["priority"] >= 0], minlength=4)
        assert counts["n_alerts"] == prio.tolist(), "alerts by priority"


def vehicle_messages(frame, ids, timestamp, order=None):
    """The reference producer's JSON (vehicle_simulator.py:721-752) for the objects of a frame; timestamp: one value
    or one per object."""
    types = ["car", "truck", "bus", "motorcycle", "drone", "tram", "van", "bike"]
    ts = np.broadcast_to(np.asarray(timestamp, np.float64), (len(ids),))
    out = []
    for i in (range(len(ids)) if order is None else order):
        f = lambda k: float(frame[k][i])
        out.append(json.dumps({
            "id": ids[i], "position": {"x": f("px"), "y": f("py"), "z": f("pz")},
            "velocity": {"x": f("vx"), "y": f("vy"), "z": f("vz")},
            "acceleration": {"x": f("ax"), "y": f("ay"), "z": f("az")},
            "heading": f("heading"), "size": f("size"), "type": types[int(frame["type"][i]) % len(types)],
            "timestamp": float(ts[i])}))
    return "\n".join(out)


def feed_rounds(stream, frame, ids, rounds, t0, seed):
    """`rounds` messages per vehicle, 0.5 s apart (trajectory history); returns the frame of the last round."""
    from rcd_b200.host import workloads as W
    rng = np.random.default_rng(seed)
    f = {k: v.copy() for k, v in frame.items()}
    for r in range(rounds):
        last = f
        stream.handle_messages(vehicle_messages(f, ids, t0 + 0.5 * r))
        f = W.advance(f, 0.5, rng)
    return last
