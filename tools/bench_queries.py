"""Cost of a step over a listed query set (rcd_set_queries) on the indexed 1 M-object bench frame.

    python tools/bench_queries.py --out profiles/r04_queries_n1.jsonl [--reps 10] [--warmup 2]

The bench frame (cfg4_1m_clustered3d, the fused detect + predict mode of bench.py, static bounds) is uploaded and
indexed once.  Then each timed pass is rcd_set_queries with a fresh random set of k slots (so the query order is
rebuilt every pass, the index never) followed by rcd_step; k = 1, 1 k, 10 k, 100 k and 1 M (every object, as a
list).  For comparison: the no-list step on the same index, and the whole frame with the index rebuilt
(rcd_invalidate + rcd_step, what bench.py times per frame).

Timing: CUDA events on the engine's stream around set_queries + step, after `--warmup` untimed passes of the same
kind; a 512 MB buffer is overwritten between timed passes, so every pass starts with a cold L2 (126 MB).  The host
time of the same calls (until the step has been enqueued) is reported beside it.  The per-stage split comes from
a separate run on a handle with RCD_FLAG_PROFILE.  One JSON line per case, then one with the device name and
power limit read in the same process.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SIZES = (1, 1000, 10_000, 100_000, 1_000_000)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--max-pairs", type=int, default=60_000_000)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_queries: no CUDA device (there is nothing to measure without one)")
    from rcd_b200.host import _native as N
    from rcd_b200.host import workloads as W
    from rcd_b200.host.engine import FrameEngine

    n = args.n
    side = 31623.0 * np.sqrt(n / 1_000_000)
    frame = W.hotspot_frame(n, 2002, side, max(1, round(50 * n / 1_000_000)))
    bounds = ((0.0, 0.0, 0.0), (side, side, 100.0))
    rng = np.random.default_rng(2024)
    sizes = [k for k in SIZES if k <= n]
    mode = N.MODE_PREDICT | N.STEP_WITH_DETECT
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")

    def sets(k, count):
        return [rng.choice(n, k, replace=False).astype(np.uint32) for _ in range(count)]

    lines = []
    with FrameEngine(n, args.max_pairs, world_bounds=bounds) as e:
        stream = torch.cuda.ExternalStream(e.cuda_stream())
        e.upload(frame)
        e.step(mode, 100.0, 10.0)  # builds the index
        e.sync()

        def timed(prepare, count):
            dev, host = [], []
            for r in range(args.warmup + count):
                with torch.cuda.stream(stream):
                    flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                t0 = time.perf_counter()
                prepare(r)
                e.step(mode, 100.0, 10.0)
                t1 = time.perf_counter()
                b.record(stream)
                b.synchronize()
                if r >= args.warmup:
                    dev.append(a.elapsed_time(b))
                    host.append((t1 - t0) * 1e3)
            c = e.counts()
            return {"device_ms_p50": float(np.median(dev)), "device_ms_min": float(np.min(dev)),
                    "device_ms_max": float(np.max(dev)), "host_enqueue_ms_p50": float(np.median(host)),
                    "reps": count, "n_owned": int(c["n_owned"]), "n_pairs": int(c["n_pairs"]), "n_fallback": int(c["n_fallback"])}

        for k in sizes:
            qs = sets(k, args.warmup + args.reps)
            res = timed(lambda r: e.set_queries(qs[r]), args.reps)
            lines.append({"case": f"list_{k}", "k": k, **res})
        # (a one-object list in between makes every pass rebuild the whole query order, as a new list would)
        res = timed(lambda r: (e.set_queries(np.arange(1, dtype=np.uint32)), e.set_queries(None)), args.reps)
        lines.append({"case": "no_list_same_index", "k": n, **res})
        res = timed(lambda r: e.invalidate(), args.reps)
        lines.append({"case": "whole_frame_index_rebuilt", "k": n, **res})

    # per-stage split: a separate handle with RCD_FLAG_PROFILE (events around every stage)
    with FrameEngine(n, args.max_pairs, world_bounds=bounds, profile=True) as e:
        e.upload(frame)
        e.step(mode, 100.0, 10.0)
        for k in sizes + [None]:
            q = None if k is None else sets(k, 1)[0]
            stages = []
            for _ in range(3):
                e.set_queries(np.arange(1, dtype=np.uint32))  # (forces a fresh query order for the no-list case too)
                e.set_queries(q)
                e.step(mode, 100.0, 10.0)
                stages.append(e.stage_ms(N.MODE_PREDICT))
            med = {s: float(np.median([st[s] for st in stages])) for s in stages[0]}
            lines.append({"case": f"stages_{'no_list' if k is None else f'list_{k}'}", "k": k or n, "stage_ms": med})

    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as ex:  # (the device name from torch stays)
        smi = f"nvidia-smi unavailable: {ex}"
    lines.append({"case": "device", "torch_name": torch.cuda.get_device_name(0), "nvidia_smi": smi,
                  "workload": f"cfg4_1m_clustered3d, {n} objects, fused detect + predict", "l2_flushed": True})
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")
    for line in lines:
        print(json.dumps(line))


if __name__ == "__main__":
    main()
