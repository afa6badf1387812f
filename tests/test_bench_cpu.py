"""bench.py pieces that run without a GPU: the reference arm (the CPU oracle timed on the host cores) and the `config`
object both arms of one command must share."""
import json
import os
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg1_1k_city",
                        "--steps", "1", "--warmup", "1"], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "object-updates/s" and d["unit"] == "object-updates/s"
    assert d["higher_is_better"] is True and d["warmup"] >= 3 and d["steps"] == 1 and d["n_gpus"] == 1
    assert d["extrapolated"] is False and d["measured_seconds_per_step"] > 0  # 1000 vehicles: the whole frame is timed
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "object-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["objects"] == 1000 and "gpu_arm" in d["config"] and d["gpu_launches"] == 0


def test_refused_arguments():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], cwd=ROOT, capture_output=True, text=True,
                           timeout=120)
        assert r.returncode == 2 and "error:" in r.stderr, (extra, r.stderr[-2000:])


def test_both_arms_build_the_same_config_object():
    sys.path.insert(0, ROOT)
    import bench
    args = types.SimpleNamespace(max_pairs=32_000_000, graph=False)
    frames, desc, _bounds, _side = bench.make_frames("cfg2_5k_city", 1, 5000, 2)
    a = bench.make_config(args, "cfg2_5k_city", desc, 5000, 5000, 1, 123.4)
    b = bench.make_config(args, "cfg2_5k_city", desc, len(frames[0]["px"]), 5000, 1, 123.4)
    assert a == b and set(a) == {"workload", "objects", "objects_per_gpu", "frame", "gpu_arm"}
    assert bench.make_frames("cfg2_5k_city", 1, 5000, 2)[0] is frames  # cached: the extras re-use generated frames
