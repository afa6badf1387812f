"""Trajectory-ring classification microbenchmark (rcd_history_classify): 1 M slots x 100 samples (H = 100, every ring
full), with 0 %, 1 %, 10 % and 100 % of the rings holding one pair of adjacent samples in swapped arrival order.
    python tools/bench_history.py out.jsonl LIB [LIB ...]
Each LIB (a build of librcd_b200.so) is measured in a child process of its own, the libraries alternating, REPS
rounds.  Call time: host clock around rcd_history_classify + rcd_sync, median of ITERS calls after one warm-up call.
The rings (3.2 GB) are far larger than L2, so every call reads them from HBM.  Prints and writes JSON lines."""
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

N_SLOTS, H, ITERS, REPS = 1 << 20, 100, 15, 3
FRACTIONS = (0.0, 0.01, 0.1, 1.0)


def child(lib):
    sys.path.insert(0, ".")
    from rcd_b200.host import workloads as W
    from rcd_b200.host.engine import FrameEngine
    rng = np.random.default_rng(1)
    p0, v, a = rng.uniform(0, 10000, (N_SLOTS, 3)), rng.uniform(-20, 20, (N_SLOTS, 3)), rng.uniform(-2, 2, (N_SLOTS, 3))
    out = []
    with FrameEngine(N_SLOTS, 1 << 16) as e:
        e.history_configure(H)
        e.upload(W.empty_frame(N_SLOTS))
        for f in FRACTIONS:
            e.history_configure(H)  # empty rings
            late = rng.random(N_SLOTS) < f
            swap_at = rng.integers(0, H - 1, N_SLOTS)  # arrival swap_at + 1 carries the older sample
            for k in range(H):
                tau = np.where(late & (swap_at == k), k + 1, np.where(late & (swap_at + 1 == k), k - 1, k))
                t = 0.1 * tau
                pos = p0 + v * t[:, None] + 0.5 * a * (t * t)[:, None]
                e.history_append(None, pos[:, 0], pos[:, 1], pos[:, 2], 1.7e9 + t)
            codes = e.history_classify()
            ms = []
            for _ in range(ITERS + 1):
                t0 = time.perf_counter()
                e._lib.rcd_history_classify(e._h, None)
                e._lib.rcd_sync(e._h)
                ms.append(1e3 * (time.perf_counter() - t0))
            out.append({"what": "rcd_history_classify", "lib": lib, "slots": N_SLOTS, "H": H, "out_of_order": f,
                        "rings_out_of_order": int(late.sum()), "ms_median": round(float(np.median(ms[1:])), 4),
                        "ms_min": round(float(np.min(ms[1:])), 4), "codes": np.bincount(codes, minlength=4).tolist()})
    print(json.dumps(out))


def main():
    out_path, libs = sys.argv[1], sys.argv[2:]
    lines = []

    def emit(d):
        d["source"] = "tools/bench_history.py"
        print(json.dumps(d), flush=True)
        lines.append(d)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip()
    emit({"what": "device", "nvidia_smi": smi})
    for rep in range(REPS):
        for lib in libs:
            env = dict(os.environ, RCD_B200_LIB=os.path.abspath(lib))
            r = subprocess.run([sys.executable, __file__, "--child", lib], env=env, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError(r.stderr[-3000:])
            for d in json.loads(r.stdout.strip().splitlines()[-1]):
                emit(dict(d, rep=rep))
    with open(out_path, "w") as fh:
        fh.writelines(json.dumps(d) + "\n" for d in lines)


if __name__ == "__main__":
    if sys.argv[1] == "--child":
        child(sys.argv[2])
    else:
        main()
