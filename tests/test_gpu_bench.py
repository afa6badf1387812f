"""bench.py --dump-outputs on the GPU: the files hold what the last timed frame computed, checked against the CPU oracle,
and the same arguments give the same files."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.gpu_helpers import compare_pairs
from tests.helpers import f64_frame

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _dump(out):
    # the bench alternates two frames: with 3 warm-up and 2 timed steps the last timed step is frame 1, the last warm-up frame 0
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg1_1k_city", "--steps", "2",
                        "--warmup", "3", "--cpu-budget", "1", "--verify-queries", "0", "--dump-outputs", str(out)],
                       cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    return {f[:-len(".npy")]: (out / f).read_bytes() for f in sorted(os.listdir(out))}


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_frame(tmp_path):
    import bench
    from oracle import oracle as O
    first = _dump(tmp_path / "first")
    assert _dump(tmp_path / "second") == first  # byte for byte
    got = {name: np.load(tmp_path / "first" / f"{name}.npy") for name in first}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) < 64 << 20

    frames = bench.make_frames("cfg1_1k_city", 1, 1000, 2)[0]
    f = f64_frame(frames[1])
    ora = {"detect": O.frame_A(f, "detect")["risks"],
           "predict": O.frame_A(f, "predict", pattern_codes=np.full(1000, 2, np.uint8))["risks"]}
    pairs = {k[len("pairs_"):]: v for k, v in got.items() if k.startswith("pairs_")}
    for flag, mode in enumerate(("detect", "predict")):
        sel = pairs["predicted"] == flag
        compare_pairs({k: v[sel] for k, v in pairs.items()}, ora[mode], mode)
    n_risks = len(ora["detect"]) + len(ora["predict"])
    assert n_risks > 100 and got["total_pairs"].tolist() == [n_risks]
    want = np.bincount(np.concatenate([ora["detect"]["i"], ora["predict"]["i"]]), minlength=1000)
    assert np.array_equal(got["object_ids"], np.arange(1000)) and np.array_equal(got["risk_counts"], want)
