"""Growth microbenchmark (rcd_reserve, rcd_alerts_reserve): the call from 1 M to 2 M objects on a record-built frame,
without and with 100-sample trajectory rings, and rcd_alerts_reserve of a table holding about 7 M live alerts.
    python tools/bench_reserve.py [out.jsonl]
Call times: host clock around the call, which synchronises before it returns; every repetition grows a fresh handle
(a reserve grows once).  The rings' share is set beside a strided device copy (torch copy_, one elementwise kernel) of
the same [100][1 M] -> [100][2 M] layout, timed with CUDA events: the alternative to the cudaMemcpy2DAsync the call
uses.  Prints JSON lines."""
import json
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
from rcd_b200.host import _native as N  # noqa: E402
from rcd_b200.host.engine import FrameEngine  # noqa: E402

REPS = 5
N0, N1, H = 1_000_000, 2_000_000, 100
out_path = sys.argv[1] if len(sys.argv) > 1 else None
lines = []


def emit(d):
    d["source"] = "tools/bench_reserve.py"
    print(json.dumps(d), flush=True)
    lines.append(d)


try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip()
except Exception as ex:  # pragma: no cover
    smi = f"nvidia-smi unavailable: {ex}"
emit({"what": "device", "nvidia_smi": smi, "torch_device": torch.cuda.get_device_name(0)})

rec = np.zeros(N0, dtype=N.RECORD_DTYPE)
rng = np.random.default_rng(1)
rec["x"], rec["y"] = rng.uniform(0, 30000, N0), rng.uniform(0, 30000, N0)
rec["size"], rec["timestamp"] = 2.0, 1.0
rec["slot"] = np.arange(N0, dtype=np.uint32)
dev = torch.from_numpy(rec.view(np.uint8).reshape(N0, 72).copy()).cuda()
lib = N.load()
pairs = 1 << 22

for rings in (False, True):
    ms = []
    for _ in range(REPS):
        with FrameEngine(N0, pairs) as e:
            if rings:
                e.history_configure(H)
            e.apply_records_device(N0, dev.data_ptr(), N0, 0, history=rings)
            e.step(N.MODE_DETECT)
            e.sync()
            t0 = time.perf_counter()
            N.check(lib.rcd_reserve(e._h, N1, 0), e._h)
            ms.append((time.perf_counter() - t0) * 1e3)
            e.step(N.MODE_DETECT)
            assert e.counts()["n_objects"] == N0
    emit({"what": "rcd_reserve call", "objects": [N0, N1], "max_pairs": pairs, "rings": H if rings else 0,
          "ring_bytes_copied": N0 * H * 32 if rings else 0, "ms_median": round(float(np.median(ms)), 3),
          "ms_all": [round(x, 3) for x in ms]})

# the ring copy as one strided copy kernel: [H][N0] samples of 32 bytes into the first N0 columns of [H][N1]
src = torch.zeros((H, N0, 4), dtype=torch.float64, device="cuda")
dst = torch.empty((H, N1, 4), dtype=torch.float64, device="cuda")
ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
ms = []
for _ in range(REPS + 1):
    ev[0].record()
    dst[:, :N0].copy_(src)
    ev[1].record()
    torch.cuda.synchronize()
    ms.append(ev[0].elapsed_time(ev[1]))
b = 2 * N0 * H * 32
emit({"what": "ring copy as a strided copy kernel (torch copy_)", "shape": [H, N0, N1], "bytes_read_written": b,
      "ms_median_after_first": round(float(np.median(ms[1:])), 3), "gbs": round(b / (np.median(ms[1:]) * 1e-3) / 1e9, 1)})
del src, dst
torch.cuda.empty_cache()

n_alerts = 7_000_000
ms, live = [], []
p = np.zeros(n_alerts, N.PAIR_DTYPE)
p["i"], p["j"] = rng.integers(0, N0, n_alerts), rng.integers(0, N0, n_alerts)
p["risk"], p["priority"] = 0.5, rng.integers(0, 4, n_alerts)
for _ in range(3):
    with FrameEngine(1 << 16, 1 << 16) as e:
        e.alerts_configure(n_alerts + (n_alerts >> 2))
        _, st = e.alerts_update_pairs(p, 1.0)
        e.sync()
        t0 = time.perf_counter()
        N.check(lib.rcd_alerts_reserve(e._h, 3 * n_alerts), e._h)
        ms.append((time.perf_counter() - t0) * 1e3)
        live.append(int(st["n_live"]))
        assert len(e.alerts_download(cap=1)) == 1
emit({"what": "rcd_alerts_reserve call", "live_alerts": live, "max_alerts": [n_alerts + (n_alerts >> 2), 3 * n_alerts],
      "table_entries": [1 << 25, 1 << 26], "ms_median": round(float(np.median(ms)), 3), "ms_all": [round(x, 3) for x in ms]})

if out_path:
    with open(out_path, "w") as f:
        for d in lines:
            f.write(json.dumps(d) + "\n")
