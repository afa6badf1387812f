"""Retirement microbenchmark (rcd_retire_stale, rcd_retire): the call at 1 M and 10 M record-built slots with 1 % of
them stale, without and with a table of ~7 M live alerts; the stale scan (k_stale_count + k_stale_scatter) and the
tombstone kernel (k_retire_slots) as achieved bytes over the data-sheet HBM bandwidth; and the alert purge
(k_alert_rebuild<AlertOfRetired>) next to rcd_alerts_expire (k_alert_rebuild<AlertTooOld>) on the same table.
    python tools/bench_retire.py [out.jsonl]
Call times: host clock around the call, which ends in a device synchronise.  Kernel times: torch.profiler, in
separate repetitions.  Before every timed repetition a 256 MB buffer is written, so the scan's first pass reads
last_seen from HBM, not L2 (its second pass then finds it in L2: 8 / 80 MB).  The ~7 M alerts are explicit pairs with
i, j uniform over the slots (rcd_alerts_update_pairs), so the purge drops about 2 % of them.  Prints JSON lines."""
import ctypes
import json
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
from rcd_b200.host import _native as N  # noqa: E402
from rcd_b200.host.engine import FrameEngine  # noqa: E402

HBM_TBS = 7.7  # HGX B200 data sheet, one GPU
STALE = 0.01
REPS = 7
out_path = sys.argv[1] if len(sys.argv) > 1 else None
lines = []


def emit(d):
    print(json.dumps(d), flush=True)
    lines.append(d)


try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip()
except Exception as ex:  # pragma: no cover
    smi = f"nvidia-smi unavailable: {ex}"
emit({"what": "device", "nvidia_smi": smi, "torch_device": torch.cuda.get_device_name(0)})
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")


def records(n, stale):
    rec = np.zeros(n, dtype=N.RECORD_DTYPE)
    rng = np.random.default_rng(n)
    rec["x"], rec["y"] = rng.uniform(0, 30000, n), rng.uniform(0, 30000, n)
    rec["size"] = 2.0
    rec["slot"] = np.arange(n, dtype=np.uint32)
    rec["timestamp"] = 100.0
    rec["timestamp"][stale] = 0.0
    return torch.from_numpy(rec.view(np.uint8).reshape(n, 72).copy()).cuda()


def kernel_ms(fn, names):
    """Mean device time per repetition of the kernels whose names contain one of `names`."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for it in range(REPS):
            fn(it)
    torch.cuda.synchronize()
    tot = {k: 0.0 for k in names}
    for ev in prof.key_averages():
        for k in names:
            if k in ev.key:
                tot[k] += ev.device_time_total / 1e3 / REPS  # (us -> ms)
    return tot


for n in (1_000_000, 10_000_000):
    k = int(n * STALE)
    stale = np.sort(np.random.default_rng(7).choice(n, k, replace=False))
    dev = records(n, stale)
    dev_stale = dev[torch.from_numpy(stale).cuda()].contiguous()
    for n_alerts in (0, 7_000_000):
        with FrameEngine(n, 1 << 16) as e:
            e.apply_records_device(n, dev.data_ptr(), n, 0, history=False)
            if n_alerts:
                e.alerts_configure(n_alerts + (n_alerts >> 2))
                rng = np.random.default_rng(11)
                p = np.zeros(n_alerts, N.PAIR_DTYPE)
                p["i"], p["j"] = rng.integers(0, n, n_alerts), rng.integers(0, n, n_alerts)
                p["risk"], p["priority"] = 0.5, rng.integers(0, 4, n_alerts)
                _, st = e.alerts_update_pairs(p, 1.0)
                live = st["n_live"]
            else:
                live = 0

            slots_out = np.zeros(k, np.uint32)
            events = np.zeros(1 << 20, N.ALERT_EVENT_DTYPE)
            n_ret, st = ctypes.c_uint64(), N.RcdAlertStats()
            lib = N.load()

            def once(it, e=e):
                # the stale slots come back (state, record time) outside the timed window; from the second repetition
                # on their alerts are gone, and the purge is a rebuild that drops nothing (the same pass over the table)
                e.apply_records_device(k, dev_stale.data_ptr(), n, 0, history=False)
                flush.fill_(it & 0xff)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                N.check(lib.rcd_retire_stale(e._h, 50.0, 30.0, slots_out.ctypes.data_as(ctypes.c_void_p), k, ctypes.byref(n_ret),
                                             events.ctypes.data_as(ctypes.c_void_p) if n_alerts else None,
                                             events.shape[0] if n_alerts else 0, ctypes.byref(st)), e._h)
                dt = time.perf_counter() - t0
                assert n_ret.value == k
                return dt * 1e3, int(st.n_expired)

            ms, purged = [], []
            for it in range(REPS):
                t, x = once(it)
                ms.append(t)
                purged.append(x)
            emit({"what": "rcd_retire_stale call", "slots": n, "stale": k, "live_alerts_before": live,
                  "purged_per_rep": purged, "ms_median_after_first": round(float(np.median(ms[1:])), 4),
                  "ms_all": [round(x, 4) for x in ms]})
            names = ["k_stale_count", "k_scan_tiles", "k_stale_scatter", "k_retire_slots", "AlertOfRetired"]
            kt = kernel_ms(once, names)
            b_count, b_scatter, b_tomb = 8 * n, 8 * n + 4 * k, 70 * k
            row = {"what": "retire kernels", "slots": n, "stale": k, "live_alerts": live,
                   "k_stale_count_ms": round(kt["k_stale_count"], 4), "k_scan_tiles_ms": round(kt["k_scan_tiles"], 4),
                   "k_stale_scatter_ms": round(kt["k_stale_scatter"], 4), "k_retire_slots_ms": round(kt["k_retire_slots"], 4),
                   "count_bytes": b_count, "scatter_bytes": b_scatter, "tombstone_bytes": b_tomb,
                   "count_frac_of_7.7TBs": round(b_count / (kt["k_stale_count"] * 1e-3) / (HBM_TBS * 1e12), 3) if kt["k_stale_count"] else None,
                   "scatter_frac_of_7.7TBs": round(b_scatter / (kt["k_stale_scatter"] * 1e-3) / (HBM_TBS * 1e12), 3) if kt["k_stale_scatter"] else None,
                   "tombstone_frac_of_7.7TBs": round(b_tomb / (kt["k_retire_slots"] * 1e-3) / (HBM_TBS * 1e12), 3) if kt["k_retire_slots"] else None,
                   "count_pass_reads": "HBM (L2 overwritten before each repetition)",
                   "scatter_pass_reads": "L2 (last_seen just read by the count pass)"}
            if n_alerts:
                row["purge_ms"] = round(kt["AlertOfRetired"], 4)
                # rcd_alerts_expire with an age nothing exceeds: the same rebuild, dropping nothing
                kt2 = kernel_ms(lambda it: e.alerts_expire(2.0, 1.0e30, cap=1), ["AlertTooOld"])
                row["expire_ms_same_table"] = round(kt2["AlertTooOld"], 4)
                cap = 1024
                while cap < 2 * (n_alerts + (n_alerts >> 2)):
                    cap <<= 1
                row["table_entries"] = cap
            emit(row)

if out_path:
    with open(out_path, "w") as f:
        for d in lines:
            f.write(json.dumps(d) + "\n")
