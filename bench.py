#!/usr/bin/env python
"""Headline benchmark: object-updates/s and p50/p99 frame latency of the collision hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W

A *step* is one frame = what the reference's perf harness times
(src/test/performance_test.py:794-813): ingest every object, rebuild the spatial index, run
detect_collisions for every object and predict_collisions for every object, deliver the results.

Workload (default): BASELINE.json configs[3] -- 1M mixed vehicles+drones, 3-D, clustered in 50
urban hotspots on a 31.6 km map (reference generator law r = U*radius).  With N GPUs the headline
frame is N x 1M objects on a map of N times the area (same density, 50 hotspots per 1M objects):
weak scaling.  Space is cut into N x-slabs; the cuts start at equal estimated pair work and are
moved during warm-up from the measured frame time of every slab (re-balancing, host/slabs.py);
every frame each GPU packs the objects within the halo width of the other slabs into fixed-size
regions and trades them with one NCCL all_to_all on the engine's stream (nothing in the frame
waits for the host), then runs the frame on owned + halo objects; results are emitted by the owner.

value : whole-job object-updates/s with the frame's object state already in HBM when the timed
        region starts (the engine still ingests it device-to-device every frame).  Timed on the
        device with CUDA events on the engine's stream, max over ranks; L2 is flushed (256 MiB
        write) before every timed frame.
e2e   : same metric through the public host API: pinned host SoA arrays -> H2D -> frame -> delivery
        to host memory, wall clock, max over ranks.  Default delivery = what the reference's consumer
        acts on (warning_system.py:259-285): the alert changes of the frame (process_collision_risks
        folded into the device alert table) + per-object risk counts + totals (rcd_summary_*); the
        full pair records (every CollisionRisk, 48 B each) are measured next to it (`e2e.full_pairs`).
Extra keys at N > 1 (same run, after the headline): `strong_scaling` = configs[3] as written (1M
objects in total over the N slabs); at N = 8 also `configs4_10m` (10M objects, heavy skew).
`verify`: a sample of queries of the headline frame re-computed by the CPU oracle (outside every timed
region) and compared with what the GPUs emitted -- pair set exact, values to 1e-4.
--dump-outputs DIR: what the last device-timed frame computed, as DIR/<name>.npy (see dump_outputs), so that two builds
can be compared output by output on the same seeded frames.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "object-updates/s"
PER_GPU_DEFAULT = 1_000_000
H2D_BYTES_PER_OBJECT = 11 * 4 + 1 + 1 + 4  # 11 fp32 fields + type + trajectory pattern + caller id
FRAME_DESC = "ingest + index + detect-all + predict-all (performance_test.py:794-813)"
L2_DESC = "flushed with a 256 MiB write before every timed frame"


# ----------------------------------------------------------------------------------------------
# workloads
# ----------------------------------------------------------------------------------------------
_FRAME_CACHE = {}


def make_frames(workload: str, n_gpus: int, per_gpu: int, n_frames: int = 2):
    """Global frames (the same on every rank: deterministic seeds) + description."""
    key = (workload, n_gpus, per_gpu, n_frames)
    if key in _FRAME_CACHE:
        return _FRAME_CACHE[key]
    from rcd_b200.host import workloads as W
    n = per_gpu * n_gpus
    if workload == "cfg4_1m_clustered3d":
        side = 31623.0 * np.sqrt(n / 1_000_000)
        f0 = W.hotspot_frame(n, 2002, side, max(1, round(50 * n / 1_000_000)))
        desc = (f"configs[3]: {n} vehicles+drones 3-D, {max(1, round(50 * n / 1_000_000))} hotspots (r=U*radius), "
                f"{side / 1000:.1f} km map")
        bounds = ((0.0, 0.0, 0.0), (side, side, 100.0))
    elif workload in ("cfg5_10m_skew3d", "cfg5_10m_skew3d_uniform_disc"):
        # the reference's radial law r = U * radius piles a Zipf-weighted hotspot up at its centre (density ~ 1/r):
        # 1.8e9 emitted pairs per frame at 10 M objects, more than any pair buffer holds.  SURVEY.md 8d asks for that
        # frame to be reported as it is, next to the variant with objects uniform in each disc (r = sqrt(U) * radius).
        law = "uniform" if workload.endswith("uniform_disc") else "reference"
        side = 100000.0 * np.sqrt(n / 10_000_000)
        f0 = W.hotspot_frame(n, 2003, side, max(1, round(200 * n / 10_000_000)), zipf_s=1.0, radial_law=law)
        desc = (f"configs[4] family: {n} objects 3-D, Zipf(s=1) hotspots ({'r=sqrt(U)*radius' if law == 'uniform' else 'r=U*radius'}), "
                f"{side / 1000:.1f} km map")
        bounds = ((0.0, 0.0, 0.0), (side, side, 100.0))
    elif workload == "cfg3_100k_uniform2d":
        side = 10000.0 * np.sqrt(n / 100_000)
        f0 = W.uniform_frame(n, 2001, map_size=side)
        desc = f"configs[2]: {n} uniform vehicles 2-D, {side / 1000:.1f} km map"
        bounds = ((0.0, 0.0, 0.0), (side, side, 0.0))
    elif workload in ("cfg2_5k_city", "cfg1_1k_city"):
        f0 = W.reference_city_frame(n, 1235 if workload == "cfg2_5k_city" else 1234)
        desc = f"configs[{1 if workload == 'cfg2_5k_city' else 0}]: reference perf-test generator, {n} vehicles, 10 km map"
        side = 10000.0
        bounds = ((0.0, 0.0, 0.0), (side, side, 0.0))
    else:
        raise SystemExit(f"unknown workload {workload}")
    frames = [f0]
    rng = np.random.default_rng(99)
    for _ in range(1, n_frames):  # the reference advances every vehicle between frames (:147-195)
        frames.append(W.advance(frames[-1], 0.05, rng, map_size=(side, side)))
    _FRAME_CACHE[key] = (frames, desc, bounds, side)
    return _FRAME_CACHE[key]


def make_config(args, workload: str, desc: str, n_total: int, per_gpu: int, world: int, halo: float) -> dict:
    """The `config` object: identical in the B200 arm and the reference arm of the same command."""
    return {"workload": f"{workload}: {desc}", "objects": int(n_total), "objects_per_gpu": int(per_gpu), "frame": FRAME_DESC,
            "gpu_arm": {"partition": (f"{world} x-slabs (cuts re-balanced from measured slab times during warm-up), halo "
                                      f"{halo:.0f} m, fixed-size NCCL all_to_all of halo records") if world > 1 else "single GPU",
                        "l2": L2_DESC, "max_pairs": int(args.max_pairs), "cuda_graph": bool(args.graph)}}


# ----------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except ValueError:
                continue
            for k, name in enumerate(names):
                if r[5 + k].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------
# CPU baseline (oracle port of the reference algorithm, all host threads, bounded sample)
# ----------------------------------------------------------------------------------------------
def cpu_frame_seconds(frame, pattern, budget_s: float, plan=None):
    """Time of one reference frame (index + detect-all + predict-all) on the host cores,
    extrapolated from a bounded sample: every `stride`-th object is queried against the FULL
    index; the index build is timed in full.  `plan` = (stride, t_index) of an earlier call skips the sizing runs.
    Returns (seconds_per_frame, description, threads, measured_s, extrapolated, plan)."""
    from oracle import oracle as O
    from rcd_b200.host import workloads as W
    f64 = W.frame_to_f64(frame)
    n = len(frame["px"])
    threads = max(O.max_threads(), os.cpu_count() or 1)  # torchrun exports OMP_NUM_THREADS=1: ask for all cores
    if plan is None:
        # index-only cost (stride so large that only object 0 is queried), once per mode
        t0 = time.perf_counter()
        O.frame_A(f64, "detect", want_potentials=False, query_stride=max(n, 1), risk_cap=1 << 16, threads=threads)
        t_index = time.perf_counter() - t0
        # pilot to size the sample
        stride = max(1, n // 2000)
        t0 = time.perf_counter()
        O.frame_A(f64, "detect", want_potentials=False, query_stride=stride, risk_cap=1 << 22, threads=threads)
        O.frame_A(f64, "predict", pattern_codes=pattern, want_potentials=False, query_stride=stride, risk_cap=1 << 22, threads=threads)
        t_pilot = max(time.perf_counter() - t0 - 2 * t_index, 1e-6)
        per_query = t_pilot / max(1, (n + stride - 1) // stride)
        want = int(min(n, max(2000, budget_s / per_query)))
        stride = max(1, n // want)
    else:
        stride, t_index = plan
    t0 = time.perf_counter()
    O.frame_A(f64, "detect", want_potentials=False, query_stride=stride, risk_cap=1 << 24, threads=threads)
    O.frame_A(f64, "predict", pattern_codes=pattern, want_potentials=False, query_stride=stride, risk_cap=1 << 24, threads=threads)
    t_sample = time.perf_counter() - t0
    queried = (n + stride - 1) // stride
    t_queries = max(t_sample - 2 * t_index, 1e-9)
    t_frame = 2 * t_index + t_queries * (n / queried)
    desc = (f"oracle/oracle.c (float64 port of src/collision, OpenMP {threads} threads): index built over all "
            f"{n} objects, every {stride}-th object queried (detect + predict = {queried} queries each, "
            f"{t_sample:.1f} s measured)" + (", extrapolated to the full frame" if stride > 1 else ""))
    return t_frame, desc, threads, t_sample, stride > 1, (stride, t_index)


def run_reference(args):
    """--impl reference: the reference's algorithm on the host cores (oracle port; the reference
    itself is pure Python and absent from the GPU box)."""
    from rcd_b200.host.slabs import halo_width
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    frames, desc, _bounds, _side = make_frames(args.workload, args.gpus, args.objects_per_gpu, 2)
    n = len(frames[0]["px"])
    pattern = np.full(n, 2, np.uint8)
    steps = args.steps
    budget = max(1.0, min(20.0, 90.0 / (steps + args.warmup)))  # the whole run stays within a few minutes
    times, measured, extrap = [], [], False
    info, plan = None, None
    for k in range(args.warmup + steps):
        t, info, threads, t_meas, ex, plan = cpu_frame_seconds(frames[0], pattern, budget, plan)
        if k >= args.warmup:
            times.append(t)
            measured.append(t_meas)
            extrap = extrap or ex
    t_mean = float(np.mean(times))
    value = n / t_mean
    emit(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "object-updates/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": t_mean * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": make_config(args, args.workload, desc, n, args.objects_per_gpu, args.gpus, halo_width(frames)),
        "extrapolated": bool(extrap), "measured_seconds_per_step": float(np.mean(measured)),
        "cpu_baseline": {"value": value, "unit": "object-updates/s", "cores": threads, "kind": "port", "sample": info},
        "e2e": {"value": value, "unit": "object-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ----------------------------------------------------------------------------------------------
# the B200 arm
# ----------------------------------------------------------------------------------------------
class SlabJob:
    """One workload on this rank: global frames -> this rank's x-slab -> engine (+ halo exchange)."""

    def __init__(self, args, workload: str, per_gpu: int, world: int, rank: int, local_rank: int, cuts=None,
                 profile: bool = True, graph: bool = False, max_pairs=None):
        import torch
        from rcd_b200.host import workloads as W
        from rcd_b200.host.engine import FRAME_FIELDS, FrameEngine
        from rcd_b200.host.slabs import SlabExchange, halo_width, owner_of, slab_bounds
        self.torch, self.FRAME_FIELDS = torch, FRAME_FIELDS
        self.world, self.rank, self.local_rank = world, rank, local_rank
        self.workload, self.per_gpu = workload, per_gpu
        self.frames, self.desc, self.bounds, self.side = make_frames(workload, world, per_gpu, 2)
        frames, bounds, side = self.frames, self.bounds, self.side
        self.n_total = len(frames[0]["px"])
        self.lo, self.hi = cuts if cuts is not None else slab_bounds(frames[0], world, side)
        lo, hi = self.lo, self.hi
        self.halo = halo_width(frames)
        ids_all = np.arange(self.n_total, dtype=np.uint32)
        self.own, self.own_ids = [], []
        n_recv_max = 0
        for f in frames:
            mine = owner_of(f["px"], lo, hi) == rank
            self.own.append(W.take(f, mine))
            self.own_ids.append(ids_all[mine])
            if world > 1:
                x = f["px"]
                n_recv_max = max(n_recv_max, int(((x >= lo[rank] - self.halo) & (x < hi[rank] + self.halo) & ~mine).sum()))
        self.n_own_max = max(len(o["px"]) for o in self.own)
        self.slack = 1.25
        cap = int(self.n_own_max + self.slack * n_recv_max) + 512 * world + 4096
        self.cap = cap
        self.max_pairs = int(args.max_pairs if max_pairs is None else max_pairs)
        # slab bounding box (+ halo) as the static grid bounds: no per-frame bbox round trip
        self.xlo = max(0.0, float(lo[rank]) - self.halo) if np.isfinite(lo[rank]) else 0.0
        self.xhi = min(side, float(hi[rank]) + self.halo) if np.isfinite(hi[rank]) else side
        self.eng_bounds = ((self.xlo, bounds[0][1], bounds[0][2]), (self.xhi, bounds[1][1], bounds[1][2]))
        self.profile, self.graph = profile, graph
        self.eng = FrameEngine(cap, self.max_pairs, device=local_rank, world_bounds=self.eng_bounds, profile=profile and not graph,
                               graph=graph)
        self.stream = torch.cuda.ExternalStream(self.eng.cuda_stream(), device=torch.device("cuda", local_rank))
        self.exch = SlabExchange(self.eng, lo, hi, rank, world, self.halo, self.stream, slack=self.slack) if world > 1 else None
        # device-resident copies of the frames (the engine ingests them device-to-device every step) and pinned host copies
        self.dev, self.pin = [], []
        for f, fid in zip(self.own, self.own_ids):
            n = len(f["px"])
            d = {k: torch.from_numpy(f[k]).cuda() for k in FRAME_FIELDS}
            d["type"] = torch.from_numpy(f["type"]).cuda()
            d["id"] = torch.from_numpy(fid.astype(np.int32)).cuda()
            d["pattern"] = torch.full((n,), 2, dtype=torch.uint8, device="cuda")
            self.dev.append(d)
            p = {k: torch.from_numpy(f[k]).pin_memory() for k in FRAME_FIELDS}
            p["type"] = torch.from_numpy(f["type"]).pin_memory()
            p["id"] = torch.from_numpy(fid.astype(np.int32)).pin_memory()
            p["pattern"] = torch.full((n,), 2, dtype=torch.uint8).pin_memory()
            self.pin.append(p)
        if self.exch is not None:  # size the exchange regions from frame 0 (counting pass + one exchange of sizes)
            self._upload_dev(0)
            self.exch.configure()
        torch.cuda.synchronize()

    # -- one frame ---------------------------------------------------------------------------------
    def _upload_dev(self, k: int) -> None:
        d = self.dev[k % len(self.dev)]
        n = int(d["px"].shape[0])
        self.eng.upload_device(n, [d[f].data_ptr() for f in self.FRAME_FIELDS], d["type"].data_ptr(), d["id"].data_ptr())
        self.eng.set_patterns_device(n, d["pattern"].data_ptr())

    def _upload_host(self, k: int) -> None:
        p = self.pin[k % len(self.pin)]
        n = int(p["px"].shape[0])
        self.eng.upload_host_ptrs(n, [p[f].data_ptr() for f in self.FRAME_FIELDS], p["type"].data_ptr(), p["id"].data_ptr())
        self.eng.set_patterns_host_ptr(n, p["pattern"].data_ptr())

    def frame(self, k: int, host: bool = False, halo_events=None) -> None:
        """Ingest frame k (device-resident copy, or pinned host memory), trade halos, detect-all + predict-all."""
        from rcd_b200.host import _native as N
        (self._upload_host if host else self._upload_dev)(k)
        if self.exch is not None:
            if halo_events is not None:
                halo_events[0].record(self.stream)
            self.exch.exchange()
            if halo_events is not None:
                halo_events[1].record(self.stream)
        self.eng.step(N.MODE_PREDICT, with_detect=True)  # one sweep over the neighbourhoods

    def launches(self) -> int:
        return self.eng.launch_count() + (self.exch.launches_last if self.exch is not None else 0)

    def close(self) -> None:
        self.eng.close()
        self.dev = self.pin = None


def barrier(world: int):
    import torch
    import torch.distributed as dist
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def time_resident(job: SlabJob, steps: int, warmup: int, flush):
    """W warm-up frames, then K device-timed frames (events on the engine's stream, L2 flushed before each)."""
    import torch
    from rcd_b200.host import _native as N
    eng, stream = job.eng, job.stream
    for k in range(warmup):
        job.frame(k)
        eng.sync()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    hev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    stage_acc, launches = {}, 0
    barrier(job.world)
    t0 = time.perf_counter()
    for k in range(steps):
        with torch.cuda.stream(stream):
            flush.zero_()  # L2 flush: 256 MiB write, outside the timed events
            ev[k][0].record(stream)
        job.frame(k, halo_events=hev[k])
        ev[k][1].record(stream)
        if job.profile and not job.graph:  # per-stage times of this frame (synchronises after the end event was recorded)
            for mode in (N.MODE_DETECT, N.MODE_PREDICT):
                for name, ms in eng.stage_ms(mode).items():
                    key = ("detect." if mode == N.MODE_DETECT else "predict.") + name
                    stage_acc[key] = stage_acc.get(key, 0.0) + ms
        launches += job.launches()
    barrier(job.world)
    t_wall = time.perf_counter() - t0
    lat = np.array([a.elapsed_time(b) for a, b in ev], np.float64)
    halo_ms = np.array([a.elapsed_time(b) for a, b in hev], np.float64) if job.exch is not None else np.zeros(steps)
    counts = eng.counts()
    counts["n_tests"] = eng.pair_tests()
    return lat, halo_ms, {k: v / steps for k, v in stage_acc.items()}, launches, counts, t_wall


def time_e2e(job: SlabJob, steps: int, warmup: int, delivery: str, inflight: int, bufs, period: float = 0.0):
    """K frames through the host API from pinned memory: H2D -> (halo) -> frame -> delivery, wall clock.
    delivery 'summary': alert changes + per-object risk counts + totals; 'pairs': every rcd_pair record.
    inflight 2: the delivery of frame k overlaps the kernels of frame k + 1 (twin buffers in the handle).
    period > 0: frames ARRIVE every `period` seconds (the reference harness paces its frames at a target rate,
    performance_test.py:760-830) instead of being submitted as fast as the host can; a frame's latency then runs from its
    arrival time to the arrival of its results."""
    eng = job.eng
    now = [1000.0]

    def begin(k):
        if delivery == "summary":
            now[0] += 0.05
            eng.summary_begin(now[0])
        else:
            eng.download_begin(bufs["pairs"][k % 2])

    def finish(k):
        if delivery == "summary":
            n_own = int(job.pin[k % len(job.pin)]["px"].shape[0])
            ev, st, _rc, _c = eng.summary_finish(bufs["events"], bufs["risk"][:n_own])
            return ev.nbytes + 4 * n_own + 96 + 56, int(st["n_events"])
        got, _c = eng.download_finish()
        return got.nbytes + 96, int(got.shape[0])

    def run(n_frames, period=0.0):
        lat, nbytes, items, t_start = [], 0, 0, {}
        t_origin = time.perf_counter()

        def arrive(k):  # the moment frame k's data is there: now, or the k-th tick of the arrival clock
            if period > 0.0:
                tick = t_origin + k * period
                while time.perf_counter() < tick:
                    pass
                t_start[k] = tick
            else:
                t_start[k] = time.perf_counter()

        if inflight >= 2:
            arrive(0)
            job.frame(0, host=True)
            begin(0)
            for k in range(1, n_frames + 1):
                if k < n_frames:
                    arrive(k)
                    job.frame(k, host=True)
                b, m = finish(k - 1)
                lat.append(time.perf_counter() - t_start[k - 1])
                nbytes += b
                items += m
                if k < n_frames:
                    begin(k)
        else:
            for k in range(n_frames):
                arrive(k)
                job.frame(k, host=True)
                begin(k)
                b, m = finish(k)
                lat.append(time.perf_counter() - t_start[k])
                nbytes += b
                items += m
        return lat, nbytes, items

    run(max(2, min(warmup, 4)))  # allocates the twin buffers, fills the alert table: outside the timed region
    barrier(job.world)
    t0 = time.perf_counter()
    lat, nbytes, items = run(steps, period)
    barrier(job.world)
    t = time.perf_counter() - t0
    return {"t": t, "lat_ms": np.array(lat) * 1e3, "d2h_per_step": nbytes / steps, "items_per_step": items / steps}


def reduce_max(world, vals):
    import torch
    import torch.distributed as dist
    t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t.cpu()]


def reduce_sum(world, vals):
    import torch
    import torch.distributed as dist
    t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return [float(v) for v in t.cpu()]


def gather_list(world, val: float):
    import torch
    import torch.distributed as dist
    t = torch.tensor([val], dtype=torch.float64, device="cuda")
    if world == 1:
        return [float(val)]
    out = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(out, t)
    return [float(o[0]) for o in out]


def rebalance(args, workload, per_gpu, world, rank, local_rank, flush, rounds: int, max_pairs=None):
    """Move the x-cuts towards equal measured frame time per slab: a few short runs, each followed by an
    all-gather of the slabs' frame times and `rebalanced_cuts` (host/slabs.py).  Returns (cuts, history)."""
    from rcd_b200.host.slabs import rebalanced_cuts, slab_bounds
    frames, _d, _b, side = make_frames(workload, world, per_gpu, 2)
    cuts = slab_bounds(frames[0], world, side)
    hist = []
    best = (None, float("inf"))
    for it in range(rounds + 1):
        job = SlabJob(args, workload, per_gpu, world, rank, local_rank, cuts=cuts, profile=False, max_pairs=max_pairs)
        lat, _h, _s, _l, _c, _t = time_resident(job, 3, 2, flush)
        job.close()
        ms = gather_list(world, float(np.mean(lat)))
        hist.append([round(v, 3) for v in ms])
        if max(ms) < best[1]:
            best = (cuts, max(ms))
        if it == rounds:
            break
        cuts = rebalanced_cuts(frames[0]["px"], cuts[0], cuts[1], ms, side)
    return best[0], hist


def verify_frame(job: SlabJob, k: int, n_queries: int):
    """Sampled oracle check of frame k (outside every timed region): every stride-th object of the GLOBAL frame is
    re-computed by the CPU oracle on rank 0 (detect + predict against all objects) and compared with what the
    owners emitted for those queries: pair set exact, values to 1e-4 relative."""
    import torch.distributed as dist
    from oracle import oracle as O  # the checker, never the thing measured
    from rcd_b200.host import workloads as W
    world, rank = job.world, job.rank
    frame = job.frames[k % len(job.frames)]
    n = job.n_total
    stride = max(1, n // max(1, n_queries))
    job.frame(k)
    got = job.eng.download(sort=False)
    c = job.eng.counts()
    overflow = c["n_pairs"] > c["n_written"]
    sel = got[got["i"] % stride == 0].copy()
    parts = [sel]
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, sel)
        flags = [None] * world
        dist.all_gather_object(flags, bool(overflow))
        overflow = any(flags)
    if rank != 0:
        return None
    t0 = time.perf_counter()
    both = np.concatenate(parts)
    f64 = W.frame_to_f64(frame)
    threads = max(O.max_threads(), os.cpu_count() or 1)
    pat = np.full(n, 2, np.uint8)
    res = {"queries": (n + stride - 1) // stride, "stride": stride, "pairs_checked": int(len(both)), "ok": True, "detail": []}
    if overflow:
        res["ok"] = None
        res["detail"].append("pair buffer overflowed on some rank: the emitted records are a subset, counts only")
        return res
    for mode, flag in (("detect", 0), ("predict", 1)):
        ora = O.frame_A(f64, mode, pattern_codes=pat if mode == "predict" else None, want_potentials=False,
                        query_stride=stride, risk_cap=1 << 24, threads=threads)["risks"]
        part = np.sort(both[both["predicted"] == flag], order=["i", "j"])
        same = len(part) == len(ora) and np.array_equal(part["i"], ora["i"]) and np.array_equal(part["j"], ora["j"])
        if not same:
            res["ok"] = False
            res["detail"].append(f"{mode}: pair set differs ({len(part)} emitted vs {len(ora)} oracle)")
            continue
        for fld in ("ttc", "distance", "risk", "rel_speed"):
            a, b = part[fld].astype(np.float64), ora[fld].astype(np.float64)
            bad = np.abs(a - b) > 1e-4 * np.abs(b) + 1e-6
            if bad.any():
                res["ok"] = False
                res["detail"].append(f"{mode}: {fld} differs beyond 1e-4 in {int(bad.sum())} pairs")
        if not np.array_equal(part["priority"].astype(np.int32), ora["priority"].astype(np.int32)):
            res["ok"] = False
            res["detail"].append(f"{mode}: alert class differs")
        res[f"{mode}_pairs"] = int(len(ora))
    res["oracle_seconds"] = round(time.perf_counter() - t0, 2)
    return res


def verify_counts(job: SlabJob, k: int, n_queries: int):
    """Light form of verify_frame for frames whose pair lists are too large to bring back: the number of risks every
    sampled query emits (detect + predict, `rcd_download_risk_counts`) against the CPU oracle's count for that query."""
    import torch.distributed as dist
    from oracle import oracle as O  # the checker, never the thing measured
    from rcd_b200.host import workloads as W
    world, rank = job.world, job.rank
    frame = job.frames[k % len(job.frames)]
    n = job.n_total
    stride = max(1, n // max(1, n_queries))
    job.frame(k)
    job.eng.sync()
    ids = job.own_ids[k % len(job.own_ids)]
    rc = job.eng.risk_counts()[: len(ids)]
    sel = ids % stride == 0
    mine = np.stack([ids[sel].astype(np.int64), rc[sel].astype(np.int64)], 1)
    parts = [mine]
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, mine)
    if rank != 0:
        return None
    t0 = time.perf_counter()
    got = np.concatenate(parts)
    got = got[np.argsort(got[:, 0])]
    f64 = W.frame_to_f64(frame)
    threads = max(O.max_threads(), os.cpu_count() or 1)
    pat = np.full(n, 2, np.uint8)
    want = np.zeros(n, np.int64)
    for mode in ("detect", "predict"):
        ora = O.frame_A(f64, mode, pattern_codes=pat if mode == "predict" else None, want_potentials=False,
                        query_stride=stride, risk_cap=1 << 26, threads=threads)["risks"]
        want += np.bincount(ora["i"].astype(np.int64), minlength=n)
    q = np.arange(0, n, stride)
    ok = len(got) == len(q) and np.array_equal(got[:, 0], q) and np.array_equal(got[:, 1], want[q])
    return {"kind": "risks per sampled query (detect + predict) against the oracle", "queries": int(len(q)), "stride": int(stride),
            "risks_checked": int(want[q].sum()), "ok": bool(ok), "oracle_seconds": round(time.perf_counter() - t0, 2)}


# --dump-outputs: the headline frame emits ~8 M pairs (~400 MB of records), so the pairs of a seeded sample of query
# objects are written; the files stay under 64 MB at every workload
DUMP_SEED = 2026
DUMP_QUERIES = 1 << 15      # query objects whose pair records are written
DUMP_PAIRS_MAX = 1 << 19    # records written at most (64 B each as written)
DUMP_COUNTS_MAX = 1 << 21   # objects whose risk counts are written (all of them up to this many; 12 B each)


def dump_outputs(job: SlabJob, k: int, out_dir: str) -> None:
    """Write what frame k (the last timed frame, still on the device) hands a caller, as DIR/<name>.npy:
      pairs_<field>  the rcd_pair records (rcd_download) whose querying object i is in a seeded sample, sorted by
                     (i, j, predicted), one file per field: i, j in float64, the rest in float32
      risk_counts    risks emitted per object (rcd_download_risk_counts), float32, for the objects in object_ids (float64)
      total_pairs    float64 [pairs the frame emitted], summed over ranks (exact even when the pair buffer overflows)
    Object ids are global and every pair is emitted once, by the owner of i, so the files do not depend on how the frame
    was cut into slabs (as long as no rank's pair buffer overflows: then which records were stored is not fixed)."""
    import torch.distributed as dist
    n, world, rank = job.n_total, job.world, job.rank
    rng = np.random.default_rng(DUMP_SEED)
    queries = np.sort(rng.choice(n, min(n, DUMP_QUERIES), replace=False))
    objects = np.arange(n) if n <= DUMP_COUNTS_MAX else np.sort(rng.choice(n, DUMP_COUNTS_MAX, replace=False))
    pairs = job.eng.download()
    ids = job.own_ids[k % len(job.own_ids)]
    c = job.eng.counts()
    mine = (pairs[np.isin(pairs["i"], queries)], ids, job.eng.risk_counts()[: len(ids)], c["n_pairs"])
    parts = [mine]
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, mine)
    if rank != 0:
        return
    pairs = np.sort(np.concatenate([p[0] for p in parts]), order=["i", "j", "predicted"])[:DUMP_PAIRS_MAX]
    risk = np.zeros(n, np.float32)
    for p in parts:
        risk[p[1]] = p[2]
    out = {f"pairs_{f}": pairs[f].astype(np.float64 if f in ("i", "j") else np.float32)
           for f in pairs.dtype.names if f != "reserved"}
    out["risk_counts"] = risk[objects]
    out["object_ids"] = objects.astype(np.float64)
    out["total_pairs"] = np.array([sum(p[3] for p in parts)], np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measure(args, workload, per_gpu, world, rank, local_rank, flush, steps, warmup, rebalance_rounds, with_e2e=True,
            with_verify=True, sampler=None, max_pairs=None, verify_kind="pairs", verify_queries=None, dump_dir=None):
    """Everything for one workload: (re-balanced) slabs, device-timed frames, end-to-end frames, verification.
    dump_dir: write the outputs of the last device-timed frame there (dump_outputs) before anything else runs a frame."""
    import torch
    from rcd_b200.host import _native as N
    cuts, rb_hist = (None, [])
    if world > 1 and rebalance_rounds > 0:
        cuts, rb_hist = rebalance(args, workload, per_gpu, world, rank, local_rank, flush, rebalance_rounds, max_pairs)
    job = SlabJob(args, workload, per_gpu, world, rank, local_rank, cuts=cuts, profile=True, graph=args.graph, max_pairs=max_pairs)
    lat, halo_ms, stage_ms, launches, counts, t_wall = time_resident(job, steps, warmup, flush)
    if dump_dir is not None:
        dump_outputs(job, steps - 1, dump_dir)
    # a halo region that was too small would have dropped records: look at the device-side counts once, after the frames
    halo_overflow = reduce_max(world, [1.0 if (job.exch is not None and job.exch.overflowed()) else 0.0])[0] > 0
    n_own_mean = float(np.mean([len(o["px"]) for o in job.own]))
    out = {"job": job, "lat": lat, "stage_ms": stage_ms, "launches": launches, "counts": counts, "t_wall": t_wall,
           "rebalance_ms": rb_hist, "halo_overflow": bool(halo_overflow)}
    graph_replays = job.eng.graph_replays() if args.graph else 0
    if args.graph:  # stage breakdown on a profiled twin (outside every timed region)
        twin = SlabJob(args, workload, per_gpu, world, rank, local_rank, cuts=cuts, profile=True, graph=False)
        _l, _h, out["stage_ms"], _n, _c, _t = time_resident(twin, steps, 1, flush)
        twin.close()
    out["graph_replays"] = graph_replays
    # ---- end to end ----------------------------------------------------------------------------------
    e2e = None
    if with_e2e:
        n_pairs_max = reduce_max(world, [float(counts["n_pairs"])])[0]
        eng = job.eng
        eng.alerts_configure(int(max(1 << 20, 3 * n_pairs_max)))
        ev_cap = int(max(1 << 18, min(n_pairs_max, 4 << 20)))
        bufs = {"events": torch.empty(ev_cap * 40, dtype=torch.uint8).pin_memory().numpy().view(N.ALERT_EVENT_DTYPE),
                "risk": torch.empty(job.n_own_max, dtype=torch.int32).pin_memory().numpy().view(np.uint32)}
        runs = {}
        for inflight in ((2, 1) if args.e2e_inflight >= 2 else (1,)):
            runs[inflight] = time_e2e(job, steps, warmup, "summary", inflight, bufs)
        t_best = {k: reduce_max(world, [v["t"]])[0] for k, v in runs.items()}  # every rank must pick the same one
        pick = min(t_best, key=lambda k: t_best[k])
        r = runs[pick]
        e2e = {"t": t_best[pick], "inflight": pick, "lat_ms": r["lat_ms"], "d2h_per_step": r["d2h_per_step"],
               "events_per_step": r["items_per_step"],
               "other": {k: {"ms_per_step": t_best[k] / steps * 1e3, "p99_ms": float(np.percentile(runs[k]["lat_ms"], 99))}
                         for k in runs if k != pick}}
        if 2 in runs:  # frames arriving at a fixed rate below saturation: the latency a periodic feed sees (95 % and 80 % load)
            for tag, slack in (("paced", 1.05), ("paced_80", 1.25)):
                period = slack * t_best[2] / steps
                n_paced = max(steps, 60)  # (a p99 over 20 frames is the maximum: one host hiccup decides it)
                rp = time_e2e(job, n_paced, warmup, "summary", 2, bufs, period=period)
                lat_p = torch.from_numpy(rp["lat_ms"]).cuda()
                if world > 1:
                    import torch.distributed as dist
                    dist.all_reduce(lat_p, op=dist.ReduceOp.MAX)
                lat_p = lat_p.cpu().numpy()
                e2e[tag] = {"period_ms": period * 1e3, "ms_per_step": reduce_max(world, [rp["t"]])[0] / n_paced * 1e3, "frames": n_paced,
                            "p50_ms": float(np.percentile(lat_p, 50)), "p90_ms": float(np.percentile(lat_p, 90)),
                            "p99_ms": float(np.percentile(lat_p, 99)), "max_ms": float(lat_p.max())}
        # full pair records (every CollisionRisk), two frames in flight
        k_full = max(3, min(steps, 10))
        cap_pairs = min(job.max_pairs, int(args.host_pairs_cap))
        bufs["pairs"] = [torch.empty(cap_pairs * 48, dtype=torch.uint8).pin_memory().numpy().view(N.PAIR_DTYPE) for _ in range(2)]
        rf = time_e2e(job, k_full, 2, "pairs", 2, bufs)
        e2e["full"] = {"t": reduce_max(world, [rf["t"]])[0], "steps": k_full, "lat_ms": rf["lat_ms"], "d2h_per_step": rf["d2h_per_step"]}
        bufs.clear()
    out["e2e"] = e2e
    nq = args.verify_queries if verify_queries is None else min(verify_queries, args.verify_queries)
    out["verify"] = None
    if with_verify and nq > 0:
        try:  # (the check never takes the measured line down with it)
            out["verify"] = (verify_frame if verify_kind == "pairs" else verify_counts)(job, 0, nq)
        except Exception as ex:  # noqa: BLE001
            out["verify"] = {"ok": None, "error": f"{type(ex).__name__}: {ex}"[:300]} if rank == 0 else None
    # ---- reduce over ranks (max time, summed counts) ---------------------------------------------------
    t_dev = float(lat.sum()) / 1e3
    out["t_dev"] = reduce_max(world, [t_dev])[0]
    sums = reduce_sum(world, [n_own_mean, float(counts["n_pairs"]), float(counts["n_candidates"]),
                              float(counts["n_objects"] - counts["n_owned"]),
                              e2e["d2h_per_step"] if e2e else 0.0, e2e["full"]["d2h_per_step"] if e2e else 0.0,
                              e2e["events_per_step"] if e2e else 0.0])
    out["objs"], out["n_pairs"], out["n_cand"], out["n_halo"], out["d2h"], out["d2h_full"], out["events"] = sums
    lat_all = torch.from_numpy(lat).cuda()
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(lat_all, op=dist.ReduceOp.MAX)  # a frame is done when its slowest slab is done
    out["lat_all"] = lat_all.cpu().numpy()
    out["per_rank_ms"] = [round(v, 3) for v in gather_list(world, float(np.mean(lat)))]
    out["per_rank_halo_ms"] = [round(v, 4) for v in gather_list(world, float(np.mean(halo_ms)))]
    out["per_rank_objects"] = [int(v) for v in gather_list(world, float(counts["n_objects"]))]
    out["n_own_mean"] = n_own_mean
    return out


def lat_stats(lat):
    return {"p50": float(np.percentile(lat, 50)), "p99": float(np.percentile(lat, 99)),
            "p99_reference_rule": float(np.sort(lat)[min(len(lat) - 1, int(len(lat) * 0.99))]), "max": float(lat.max())}


def run_b200(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
        args.gpus = world
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()  # runs through warm-up and the timed regions (the frames are milliseconds long)
        time.sleep(0.3)
    steps = args.steps
    m = measure(args, args.workload, args.objects_per_gpu, world, rank, local_rank, flush, steps, args.warmup,
                args.rebalance if world > 1 else 0, verify_kind=args.verify_kind, dump_dir=args.dump_outputs)
    clocks = sampler.stop() if rank == 0 else None
    job = m["job"]

    # ---- extra lines BASELINE.json names (after the headline, same process) ------------------------------
    extras = {}
    if world > 1 and args.extras and args.workload == "cfg4_1m_clustered3d" and args.objects_per_gpu == PER_GPU_DEFAULT:
        job.close()
        xs = max(5, min(steps, 10))
        s = measure(args, "cfg4_1m_clustered3d", PER_GPU_DEFAULT // world, world, rank, local_rank, flush, xs, 3,
                    min(args.rebalance, 2), with_e2e=False, verify_queries=1000)
        extras["strong_scaling"] = {
            "workload": f"configs[3] as written: {int(s['objs'])} objects in total over {world} x-slabs", "scaling": "strong",
            "value": s["objs"] * xs / s["t_dev"], "unit": "object-updates/s", "ms_per_step": s["t_dev"] / xs * 1e3,
            "latency_ms": lat_stats(s["lat_all"]), "steps": xs, "per_rank_ms": s["per_rank_ms"],
            "per_rank_halo_ms": s["per_rank_halo_ms"], "pairs_emitted": s["n_pairs"], "halo_objects": s["n_halo"],
            "verify": s["verify"]}
        s["job"].close()
        _FRAME_CACHE.clear()
        if world == 8:
            # the north-star size: 10 M objects on the box, at the configs[3] density (1.25 M per GPU)
            xs = max(5, min(steps, 10))
            s = measure(args, "cfg4_1m_clustered3d", 1_250_000, world, rank, local_rank, flush, xs, 3, min(args.rebalance, 2),
                        with_e2e=False, verify_kind="counts", verify_queries=1000)
            extras["north_star_10m"] = {
                "workload": f"cfg4_1m_clustered3d: {s['job'].desc}", "scaling": "weak (1.25 M objects per GPU)",
                "value": s["objs"] * xs / s["t_dev"], "unit": "object-updates/s", "ms_per_step": s["t_dev"] / xs * 1e3,
                "latency_ms": lat_stats(s["lat_all"]), "steps": xs, "per_rank_ms": s["per_rank_ms"],
                "per_rank_halo_ms": s["per_rank_halo_ms"], "pairs_emitted": s["n_pairs"], "halo_objects": s["n_halo"],
                "verify": s["verify"]}
            s["job"].close()
            _FRAME_CACHE.clear()
            for name in (() if args.skip_configs4 else ("cfg5_10m_skew3d_uniform_disc", "cfg5_10m_skew3d")):
                xs = 3
                # (the queues between the kernels are sized from the pair buffer: 256 M pairs keep this frame out of the
                # overflow pass -- 1.8e9 risks per frame on the box with the reference's radial law)
                big = 256_000_000
                s = measure(args, name, 1_250_000, world, rank, local_rank, flush, xs, 3, 1, with_e2e=False, max_pairs=big,
                            verify_kind="counts", verify_queries=400)
                extras["configs4_10m" + ("_uniform_disc" if name.endswith("disc") else "_reference_law")] = {
                    "workload": f"{name}: {s['job'].desc}", "scaling": "n/a (10M objects on 8 GPUs)",
                    "value": s["objs"] * xs / s["t_dev"], "unit": "object-updates/s", "ms_per_step": s["t_dev"] / xs * 1e3,
                    "candidates_per_s": s["n_cand"] * xs / s["t_dev"], "latency_ms": lat_stats(s["lat_all"]), "steps": xs,
                    "per_rank_ms": s["per_rank_ms"], "pairs_emitted": s["n_pairs"], "candidates": s["n_cand"],
                    "pairs_stored_cap_per_gpu": big,
                    "note": "counts are exact beyond the pair buffer; records past it are not stored", "verify": s["verify"]}
                s["job"].close()
                _FRAME_CACHE.clear()

    if rank == 0:
        from_peaks = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(from_peaks):
            peak, peak_src = float(json.load(open(from_peaks))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        counts = m["counts"]
        n_loc = m["n_own_mean"] + counts["n_objects"] - counts["n_owned"]  # rank 0: owned + halo
        # algorithmic bytes per launch (DESIGN.md "byte model"), rank 0's objects
        npass = max(1, -(-int(np.ceil(np.log2(max(2, eng_ncells(job.bounds, job.xlo, job.xhi))))) // 8))
        model = {"keys": 106.0 * n_loc, "sort": (16.0 * npass - 4.0) * n_loc, "reorder": 112.0 * n_loc,
                 "pairs": 56.0 * n_loc, "narrow": 0.0, "exact": 0.0, "qorder": 0.0}
        kernels = {}
        for key, ms in m["stage_ms"].items():
            mode, name = key.split(".")
            if name in model and ms > 0:
                b = model[name]
                kernels[key] = {"ms": round(ms, 5), "alg_bytes": b, "gbs": round(b / (ms * 1e-3) / 1e9, 2) if b else None}
        dom_key = max((k for k in kernels if kernels[k]["alg_bytes"]), key=lambda k: kernels[k]["ms"])
        dom = kernels[dom_key]
        traffic, ncu_info = None, None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            traffic = tj.get(dom_key)
            ncu_info = tj.get("ncu", {}).get(dom_key)
        pair_tests = None
        if "predict.pairs" in kernels:  # (query, neighbour) tests of the S1 filter on rank 0 per second of its pair kernel
            pair_tests = counts["n_tests"] / (kernels["predict.pairs"]["ms"] * 1e-3)
        cpu = None
        if world == 1:  # the CPU baseline is timed on rank 0 at N=1 only
            cpu_t, cpu_desc, cpu_threads, _tm, ex, _plan = cpu_frame_seconds(job.frames[0], np.full(job.n_total, 2, np.uint8), args.cpu_budget)
            cpu = {"value": job.n_total / cpu_t, "unit": "object-updates/s", "cores": cpu_threads, "kind": "port",
                   "sample": cpu_desc, "extrapolated": bool(ex)}
        e2e = m["e2e"]
        out = {
            "metric": METRIC, "value": m["objs"] * steps / m["t_dev"], "unit": "object-updates/s", "n_gpus": world,
            "steps": steps, "warmup": args.warmup, "ms_per_step": m["t_dev"] / steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32 pre-filter + f64 decisions", "data": "synthetic",
            "config": make_config(args, args.workload, job.desc, job.n_total, args.objects_per_gpu, world, job.halo),
            "latency_ms": lat_stats(m["lat_all"]),
            "frame_totals": {"pairs_emitted": m["n_pairs"], "candidates": m["n_cand"], "halo_objects": m["n_halo"],
                             "pair_tests_rank0": int(counts["n_tests"])},
            "per_rank": {"frame_ms": m["per_rank_ms"], "halo_ms": m["per_rank_halo_ms"], "objects_with_halo": m["per_rank_objects"],
                         "rebalance_rounds_ms": m["rebalance_ms"], "halo_region_overflow": m["halo_overflow"]},
            "e2e": {"value": m["objs"] * steps / e2e["t"], "unit": "object-updates/s",
                    "h2d_bytes_per_step": int(m["objs"] * H2D_BYTES_PER_OBJECT), "d2h_bytes_per_step": int(m["d2h"]),
                    "delivery": "alert changes (rcd_alert_event, 40 B) + per-object risk counts + totals (rcd_summary_begin/_finish)",
                    "alert_events_per_step": m["events"], "ms_per_step": e2e["t"] / steps * 1e3,
                    "p99_ms": float(np.percentile(e2e["lat_ms"], 99)), "frames_in_flight": e2e["inflight"],
                    "other_inflight": e2e["other"],
                    "paced_arrivals": (dict(e2e["paced"], value=m["objs"] / (e2e["paced"]["ms_per_step"] * 1e-3),
                                            note="frames arrive every period_ms (1.05 x the closed-loop step, like the reference "
                                                 "harness's target rate); latency from arrival to delivered results, max over ranks")
                                       if "paced" in e2e else None),
                    "paced_arrivals_80pct_load": (dict(e2e["paced_80"], value=m["objs"] / (e2e["paced_80"]["ms_per_step"] * 1e-3),
                                                       note="the same with frames arriving every 1.25 x the closed-loop step")
                                                  if "paced_80" in e2e else None),
                    "full_pairs": {"value": m["objs"] * e2e["full"]["steps"] / e2e["full"]["t"], "unit": "object-updates/s",
                                   "delivery": "every emitted pair as a 48-byte rcd_pair (rcd_download_begin/_finish), 2 frames in flight",
                                   "d2h_bytes_per_step": int(m["d2h_full"]), "ms_per_step": e2e["full"]["t"] / e2e["full"]["steps"] * 1e3,
                                   "p99_ms": float(np.percentile(e2e["full"]["lat_ms"], 99)), "steps": e2e["full"]["steps"]}},
            "gpu_launches": int(m["launches"]),
            "graph_replays": int(m["graph_replays"]),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": dom_key, "achieved": dom["gbs"], "peak": peak, "unit": "GB/s",
                         "frac": dom["gbs"] / peak, "traffic": traffic, "peak_source": peak_src,
                         "pair_tests_per_s": pair_tests, "ncu": ncu_info,
                         "note": "the pair kernels are fp32-ALU / issue bound (pairs >> bytes): pair_tests_per_s and the ncu "
                                 "issue figures describe them; HBM-bound stages are in `kernels`"},
            "kernels": kernels,
            "cpu_baseline": cpu,
            "verify": m["verify"],
            "wall_s_timed_region": m["t_wall"],
        }
        out.update(extras)
        emit(json.dumps(out))
    if not extras:
        job.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def eng_ncells(bounds, xlo, xhi):
    cell = (100.0 * 1.002 + 0.02) * 0.5
    nx = int((xhi - xlo) / cell) + 1
    ny = int((bounds[1][1] - bounds[0][1]) / cell) + 1
    nz = int((bounds[1][2] - bounds[0][2]) / (2 * cell)) + 1
    return nx * ny * nz + 1


_REAL_STDOUT = None


def quiet_stdout():
    """NCCL and friends print banners to fd 1; the contract is ONE JSON line on stdout.  Everything
    but the final line goes to stderr."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: str):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(line + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--workload", default="cfg4_1m_clustered3d",
                    choices=["cfg1_1k_city", "cfg2_5k_city", "cfg3_100k_uniform2d", "cfg4_1m_clustered3d", "cfg5_10m_skew3d",
                             "cfg5_10m_skew3d_uniform_disc"])
    ap.add_argument("--objects-per-gpu", type=int, default=None)
    ap.add_argument("--max-pairs", type=int, default=32_000_000)
    ap.add_argument("--cpu-budget", type=float, default=15.0, help="seconds of CPU work for the cpu_baseline sample")
    ap.add_argument("--graph", action="store_true",
                    help="replay rcd_step as a CUDA graph (RCD_FLAG_GRAPH): for the small, launch-bound configs")
    ap.add_argument("--e2e-inflight", type=int, default=2,
                    help="frames in flight in the end-to-end leg (2 = the delivery overlaps the next frame)")
    ap.add_argument("--host-pairs-cap", type=int, default=32_000_000,
                    help="pairs per rank the full-pairs end-to-end leg copies back to (pinned) host memory per frame")
    ap.add_argument("--rebalance", type=int, default=3, help="re-balancing rounds of the slab cuts during warm-up (N > 1)")
    ap.add_argument("--verify-queries", type=int, default=2000,
                    help="queries of the headline frame re-computed by the CPU oracle after the timed regions (0 = off)")
    ap.add_argument("--verify-kind", choices=["pairs", "counts"], default="pairs",
                    help="headline check: emitted pair records, or only the per-query risk counts (frames too large to bring back)")
    ap.add_argument("--skip-configs4", action="store_true",
                    help="at N = 8: leave out the two configs[4] lines (10 M heavy-skew objects, 256 M-pair buffers) of the extras")
    ap.add_argument("--no-extras", dest="extras", action="store_false",
                    help="skip the strong-scaling / 10M lines that follow the headline at N > 1")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed frame computed to DIR/<name>.npy (seeded sample of the pairs, per-object "
                         "risk counts, total pairs): for comparing two builds output by output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl b200)")
    if args.objects_per_gpu is None:
        args.objects_per_gpu = {"cfg1_1k_city": 1000, "cfg2_5k_city": 5000, "cfg3_100k_uniform2d": 100_000,
                                "cfg4_1m_clustered3d": PER_GPU_DEFAULT, "cfg5_10m_skew3d": 1_250_000,
                                "cfg5_10m_skew3d_uniform_disc": 1_250_000}[args.workload]
    args.warmup = max(args.warmup, 3)
    quiet_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
