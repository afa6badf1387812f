"""Ingest microbenchmark (SURVEY.md 8f rank 2): decode throughput of the native decoder next to the
reference's per-message Python path, and the achieved HBM bandwidth of k_apply_records.
    python tools/bench_ingest.py [n_messages]
Prints JSON lines."""
import json
import random
import sys
import time

import numpy as np

sys.path.insert(0, ".")
from rcd_b200.host import _native as N  # noqa: E402
from rcd_b200.host.engine import FrameEngine  # noqa: E402
from rcd_b200.host.ingest import VehicleIngest  # noqa: E402
from tests import ingest_cases as C  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000
rng = random.Random(1)
t0 = time.perf_counter()
base = [C.reference_message(rng, k, 1.7e9 + 1e-3 * k) for k in range(min(n, 100_000))]
# reuse the generated bodies with fresh ids (generation in Python is the slow part of this script)
msgs = [base[k % len(base)].replace(f'"vehicle-{k % len(base)}"', f'"vehicle-{k}"', 1) for k in range(n)]
text = "\n".join(msgs).encode()
print(json.dumps({"what": "generated", "messages": n, "bytes": len(text), "s": round(time.perf_counter() - t0, 2)}))

# reference path: json.loads + the field reads of _handle_vehicle_position, per message
def python_path(text):
    """What the reference does per message (warning_system.py:638-678): json.loads + the field reads."""
    try:
        d = json.loads(text)
        return (d["id"], d["position"]["x"], d["position"]["y"], d["position"]["z"], d["velocity"]["x"], d["velocity"]["y"],
                d["velocity"]["z"], d["acceleration"]["x"], d["acceleration"]["y"], d["acceleration"]["z"], d["heading"],
                d["size"], d["type"], d["timestamp"])
    except Exception:
        return None


sample = msgs[: min(n, 200_000)]
t0 = time.perf_counter()
ok = sum(python_path(m) is not None for m in sample)
dt = time.perf_counter() - t0
print(json.dumps({"what": "reference per-message parse (Python, 1 core)", "messages": len(sample), "ok": ok,
                  "msgs_per_s": round(len(sample) / dt), "MB_per_s": round(sum(map(len, sample)) / dt / 1e6, 1)}))

out = np.empty(n + 16, dtype=N.RECORD_DTYPE)
for threads in (1, 0):
    with VehicleIngest(threads=threads) as g:
        t0 = time.perf_counter()
        rec, mseq = g.decode(text, out=out)
        dt = time.perf_counter() - t0
        print(json.dumps({"what": f"native decode, threads={'all' if threads == 0 else threads}", "messages": len(rec),
                          "msgs_per_s": round(len(rec) / dt), "MB_per_s": round(len(text) / dt / 1e6, 1)}))

try:
    import torch
    assert torch.cuda.is_available()
except Exception as e:  # pragma: no cover
    print(json.dumps({"what": "apply", "skipped": repr(e)}))
    sys.exit(0)

peak = json.load(open("MEASURED_PEAKS.json"))["hbm_gbs"] if __import__("os").path.exists("MEASURED_PEAKS.json") else 6546.2
rec = out[:n]
for order in ("slot order", "random order"):
    r = rec if order == "slot order" else rec[np.random.default_rng(0).permutation(n)]
    dev = torch.from_numpy(r.view(np.uint8).reshape(n, 72).copy()).cuda()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for hist in (False, True):
        with FrameEngine(n, 1 << 16, profile=True) as e:
            if hist:
                e.history_configure(100)
            ms = []
            for it in range(6):
                flush.fill_(it)  # L2 flush: the records were just written / read
                torch.cuda.synchronize()
                e.apply_records_device(n, dev.data_ptr(), n, 0, history=hist)
                e.sync()
                ms.append(e.stage_ms(N.MODE_DETECT)["upload"])
            t = float(np.median(ms[2:]))
            alg = n * (72 + 58 + (32 + 8 if hist else 0))  # (58: the state and the record time)
            print(json.dumps({"what": f"k_apply_records, {order}, history={hist}", "records": n, "ms": round(t, 4),
                              "alg_bytes": alg, "GBps": round(alg / t / 1e6, 1), "frac_of_measured_peak": round(alg / t / 1e6 / peak, 3)}))
