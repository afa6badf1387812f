"""Trajectory pattern codes on the GPU against the float64 oracle, code for code, on every path that feeds them: the
staged classifier (rcd_classify_patterns), the device rings through rcd_history_append / _reset / _move, and the rings
through message ingest (VehiclePositionStream), up to the predict frame that uses the codes.

The oracle's model of a ring: the samples a slot has received, in arrival order, the last H of them; orc_pattern sorts
them by timestamp (stable) before classifying, as the reference does (collision_detection.py:638).  Samples arrive
late here on purpose (a broker reorders, several messages of one vehicle share a batch), and at least half of the
vehicles carry epoch-sized timestamps.  Cases placed near the 0.1 m/s and 0.1 m/s^2 thresholds are held at least a
relative 1e-9 away from them (DESIGN.md section 3: pow vs x*x differ in the last ulp)."""
import numpy as np
import pytest

from tests.gpu_helpers import compare_counts, compare_pairs, vehicle_messages

pytestmark = pytest.mark.gpu

EPOCH = 1.7e9
# vehicle kinds of the sample generator
STATIONARY, CRUISE, ACCEL, DECEL, LATE_ACCEL, LATE_CRUISE, TIE_GLITCH, REPEATED_T, FAR, VERY_LATE, \
    NEAR_SPEED, NEAR_ACCEL, SAME_T = range(13)
LATE_KINDS = (LATE_ACCEL, LATE_CRUISE, TIE_GLITCH, VERY_LATE)
NEAR_KINDS = (NEAR_SPEED, NEAR_ACCEL)  # placed near a threshold, on purpose


def _O():
    from oracle import oracle as O
    return O


def _unit(rng, m):
    u = rng.normal(size=(m, 3))
    return u / np.linalg.norm(u, axis=1, keepdims=True)


def _params(rng, m, kinds):
    """Motion of m vehicle identities; kind[i] drawn from `kinds`."""
    kind = rng.choice(np.asarray(kinds), m)
    P = {"kind": kind}
    epoch = rng.random(m) < 0.6
    P["t0"] = np.where(epoch, EPOCH + rng.uniform(0.0, 1e6, m), rng.uniform(0.0, 100.0, m))
    P["step"] = rng.choice([0.1, 0.5, 1.0, 0.001], m, p=[0.35, 0.35, 0.15, 0.15])
    P["p0"] = rng.uniform(-1000.0, 1000.0, (m, 3))
    P["p0"][kind == FAR] = rng.uniform(-90000.0, 90000.0, ((kind == FAR).sum(), 3))
    speed = rng.uniform(1.0, 25.0, m)
    # near a threshold: |v| or |a| = 0.1 (1 +- d), d log-uniform in [2e-9, 1e-2] (a quarter of them closer than the
    # fp32 rounding of the speed or acceleration)
    d = 10.0 ** rng.uniform(-8.7, -2.0, m) * rng.choice([-1.0, 1.0], m)
    speed = np.where(kind == NEAR_SPEED, 0.1 * (1.0 + d), speed)
    speed = np.where(np.isin(kind, (STATIONARY, TIE_GLITCH, SAME_T)), 0.0, speed)
    P["v"] = _unit(rng, m) * speed[:, None]
    acc = np.where(np.isin(kind, (ACCEL, LATE_ACCEL, VERY_LATE, FAR, DECEL)), rng.uniform(0.3, 3.0, m), 0.0)
    acc = np.where(kind == NEAR_ACCEL, 0.1 * (1.0 + d), acc)
    P["a"] = _unit(rng, m) * acc[:, None]
    # decelerating to a stop: a = -v / t_stop, then parked
    t_stop = rng.uniform(1.0, 20.0, m)
    P["t_stop"] = np.where(kind == DECEL, t_stop, np.inf)
    P["a"][kind == DECEL] = -P["v"][kind == DECEL] / t_stop[kind == DECEL, None]
    near = np.isin(kind, NEAR_KINDS)  # small timestamps and coarse steps: the rounding noise stays far below d
    P["step"][near] = 0.5
    P["t0"][near] = rng.uniform(0.0, 100.0, near.sum())
    P["step"][kind == SAME_T] = 0.0
    P["period"] = rng.choice([2, 3, 5], m)  # LATE_*: the last two arrivals of every period swap
    P["glitch"] = rng.uniform(0.3, 3.0, m) * rng.choice([-1.0, 1.0], m)
    return P


def _samples(P, ident, k):
    """(x, y, z, t) of the k-th arrival of vehicle `ident` (arrays that broadcast together) -> [..., 4] float64."""
    ident, k = np.asarray(ident, np.int64), np.asarray(k, np.int64)
    g = lambda name: P[name][ident]  # (gathered at the shape of ident, broadcast against k below)
    kind, per = g("kind"), g("period")
    tau = k  # time index of the arrival
    swap = np.isin(kind, (LATE_ACCEL, LATE_CRUISE))
    tau = np.where(swap & (k % per == per - 2), k + 1, tau)
    tau = np.where(swap & (k % per == per - 1), k - 1, tau)
    glitch = (kind == TIE_GLITCH) & (k % 5 == 4)  # a second report for an earlier time, elsewhere
    tau = np.where(glitch, k - 2, tau)
    very_late = (kind == VERY_LATE) & (k % 7 == 6)
    tau = np.where(very_late, k - 4, tau)
    tau = np.where(kind == REPEATED_T, k // 2, tau)
    tr = tau * g("step")
    te = np.minimum(tr, g("t_stop"))[..., None]
    pos = g("p0") + g("v") * te + 0.5 * g("a") * (te * te)
    pos[..., 0] += np.where(glitch, g("glitch"), 0.0)
    pos[..., 1] += np.where(very_late | ((kind == REPEATED_T) & (k % 2 == 1)), 0.05, 0.0)
    pos += np.where(kind == SAME_T, 0.5 * np.sin(k), 0.0)[..., None]  # one timestamp, positions that wander
    t = g("t0") + tr
    return np.concatenate([pos, np.broadcast_to(t[..., None], pos.shape[:-1] + (1,))], axis=-1)


def _speed_accel(hist, count):
    """Mean speed and mean acceleration magnitude of each history, sorted by timestamp (float64, the reference's
    order of operations): the distance of each case from the thresholds."""
    n, L = hist.shape[:2]
    valid = np.arange(L)[None, :] < count[:, None]
    t = np.where(valid, hist[..., 3], np.inf)
    h = np.take_along_axis(hist, np.argsort(t, axis=1, kind="stable")[..., None], 1)
    sv, sa = np.zeros((n, 3)), np.zeros((n, 3))
    nv, na = np.zeros(n), np.zeros(n)
    pv, pt = np.zeros((n, 3)), np.zeros(n)
    with np.errstate(all="ignore"):
        for k in range(1, L):
            dt = h[:, k, 3] - h[:, k - 1, 3]
            step = (k < count) & (dt > 0)
            v = (h[:, k, :3] - h[:, k - 1, :3]) / dt[:, None]
            dtv = h[:, k, 3] - pt
            acc = step & (nv > 0) & (dtv > 0)
            sa += np.where(acc[:, None], (v - pv) / dtv[:, None], 0.0)
            na += acc
            sv += np.where(step[:, None], v, 0.0)
            nv += step
            pv = np.where(step[:, None], v, pv)
            pt = np.where(step, h[:, k, 3], pt)
        speed = np.linalg.norm(sv / np.maximum(nv, 1)[:, None], axis=1)
        accel = np.linalg.norm(sa / np.maximum(na, 1)[:, None], axis=1)
    return speed, accel, nv


def _clear_of_thresholds(hist, count):
    """True where neither threshold decision is within a relative 1e-9 of 0.1."""
    speed, accel, nv = _speed_accel(hist, count)
    near = lambda x: np.abs(x - 0.1) < 1e-9 * 0.1
    return ~((nv > 0) & (near(speed) | ((speed >= 0.1) & near(accel))))


# ---- 1. the staged classifier ----------------------------------------------------------------------------------------
def test_staged_classifier_matches_the_oracle():
    from rcd_b200.host.engine import FrameEngine
    O = _O()
    rng = np.random.default_rng(1)
    lengths = list(range(13)) + [50, 99, 100]
    codes, near_sides, total = [], set(), 0
    with FrameEngine(1024, 1 << 16) as e:
        for L in lengths:
            m = 7000 if L <= 12 else 4000
            stride = L + int(rng.integers(1, 5))  # stride > count: the padding is NaN and must never be read
            P = _params(rng, m, range(13))
            hist = _samples(P, np.arange(m)[:, None], np.arange(L)[None, :]).reshape(m, L, 4)
            # this call takes histories already in timestamp order
            order = np.argsort(hist[..., 3], axis=1, kind="stable")
            hist = np.take_along_axis(hist, order[..., None], 1)
            count = np.full(m, L, np.uint32)
            keep = _clear_of_thresholds(hist, count) if L >= 2 else np.ones(m, bool)
            assert keep.mean() > 0.999
            hist, P_kind = hist[keep], P["kind"][keep]
            m = len(hist)
            staged = np.full((m, stride, 4), np.nan)
            staged[:, :L] = hist
            count = np.full(m, L, np.uint32)
            got = e.classify_patterns(staged, count)
            want = O.patterns(staged, count)
            bad = np.flatnonzero(got != want)
            assert len(bad) == 0, (L, len(bad), int(P_kind[bad[0]]), staged[bad[0], :count[bad[0]]].tolist(),
                                   int(got[bad[0]]), int(want[bad[0]]))
            if L >= 2:  # (two samples give no acceleration term)
                assert set(want.tolist()) == ({0, 1} if L == 2 else {0, 1, 2}), L
            else:
                assert set(want.tolist()) == {3}
            for kd, code in zip(P_kind[(count >= 3)], want[count >= 3]):
                if kd in NEAR_KINDS:
                    near_sides.add((int(kd), int(code)))
            codes.append(want)
            total += m
    assert total >= 100_000
    # the near-threshold cases fall on both sides of each threshold
    assert {(NEAR_SPEED, 0), (NEAR_SPEED, 1), (NEAR_ACCEL, 1), (NEAR_ACCEL, 2)} <= near_sides
    assert np.bincount(np.concatenate(codes), minlength=4).min() > 1000


# ---- 2. device rings through rcd_history_append / _reset / _move -----------------------------------------------------
class RingModel:
    """The oracle's model of the rings: slot s holds vehicle identity ident[s] and has received its arrivals
    0 .. count[s] - 1 (of _samples), in that order; the last H are kept.  Reset: a new identity, nothing received.
    Move: dst takes src's identity and count."""

    def __init__(self, P, n, H):
        self.P, self.H = P, H
        self.ident = np.arange(n, dtype=np.int64)
        self.count = np.zeros(n, np.int64)
        self.next_ident = n

    def arrivals(self, slots):
        return _samples(self.P, self.ident[slots], self.count[slots])

    def append(self, slots):
        self.count[slots] += 1

    def reset(self, slots):
        self.ident[slots] = np.arange(self.next_ident, self.next_ident + len(slots))
        self.next_ident += len(slots)
        self.count[slots] = 0

    def move(self, dst, src):
        self.ident[dst], self.count[dst] = self.ident[src], self.count[src]

    def histories(self, slots):
        """[len(slots), w, 4] arrival-ordered kept samples (w = the longest), and how many each slot has."""
        cnt = np.minimum(self.count[slots], self.H)
        w = max(1, int(cnt.max(initial=0)))
        k = (self.count[slots] - cnt)[:, None] + np.arange(w)[None, :]
        hist = _samples(self.P, self.ident[slots][:, None], np.minimum(k, self.count[slots][:, None]))
        return hist, cnt

    def codes(self, chunk=1 << 16):
        """Oracle codes of every slot, and which slots hold samples out of timestamp order."""
        n = len(self.count)
        codes, unordered = np.zeros(n, np.uint8), np.zeros(n, bool)
        by_len = np.argsort(self.count, kind="stable")  # (chunks of similar lengths)
        for a in range(0, n, chunk):
            sl = by_len[a: a + chunk]
            hist, cnt = self.histories(sl)
            codes[sl] = _O().patterns(hist, cnt)
            valid = np.arange(1, hist.shape[1])[None, :] < cnt[:, None]
            unordered[sl] = ((hist[:, 1:, 3] < hist[:, :-1, 3]) & valid).any(axis=1)
        return codes, unordered


def _ring_run(n, H, rounds, checkpoints, seed, resets=0, moves=0, kinds=range(10), busy=1.0):
    from rcd_b200.host import workloads as W
    from rcd_b200.host.engine import FrameEngine
    rng = np.random.default_rng(seed)
    P = _params(rng, n + resets * len(checkpoints) + 8, kinds)
    model = RingModel(P, n, H)
    rate = rng.uniform(0.0, busy, n)  # per-slot share of the rounds: counts span 0 .. rounds
    rate[: n // 16] = 1.0
    rate[-3:] = (0.0, 0.5 / rounds, 1.5 / rounds)  # and a few that stay (about) empty
    seen = []
    with FrameEngine(n, 1 << 16) as e:
        e.history_configure(H)
        e.upload(W.empty_frame(n))
        for r in range(1, rounds + 1):
            slots = np.flatnonzero(rng.random(n) < rate).astype(np.uint32)
            if len(slots):
                a = model.arrivals(slots)
                e.history_append(slots, a[:, 0], a[:, 1], a[:, 2], a[:, 3])
                model.append(slots)
            if r not in checkpoints:
                continue
            got, (want, unordered) = e.history_classify(), model.codes()
            bad = np.flatnonzero(got != want)
            assert len(bad) == 0, (H, r, len(bad), int(bad[0]), int(model.count[bad[0]]),
                                   int(P["kind"][model.ident[bad[0]]]), int(got[bad[0]]), int(want[bad[0]]))
            seen.append((want, unordered))
            wrapped = np.flatnonzero(model.count > H)
            for _ in range(moves if len(wrapped) else 0):  # copies of wrapped rings over other slots
                dst, src = int(rng.integers(0, n)), int(rng.choice(wrapped))
                e.history_move(dst, src)
                model.move(dst, src)
            if resets:
                gone = rng.choice(n, resets, replace=False).astype(np.uint32)
                e.history_reset(gone)
                model.reset(gone)
        got, (want, _) = e.history_classify(), model.codes()
        assert np.array_equal(got, want), (H, int((got != want).sum()))
    return model, seen


@pytest.mark.parametrize("H", [2, 3, 17, 100, 4096])
def test_device_rings_match_the_oracle(H):
    n = {2: 3000, 3: 3000, 17: 3000, 100: 2000, 4096: 96}[H]
    rounds = 3 * H
    checkpoints = {rounds // 5, rounds // 2, (4 * rounds) // 5, rounds}
    model, seen = _ring_run(n, H, rounds, checkpoints, seed=10 + H, resets=max(4, n // 50), moves=min(40, n // 4))
    wrapped = model.count[model.count > H]
    assert model.count.max() >= 2 * H and (model.count < 2).any()
    assert len(np.unique(wrapped % H)) >= min(H, n // 8)  # the oldest kept sample sits at many ring positions
    codes = np.concatenate([w for w, _ in seen])
    unordered = np.concatenate([u for _, u in seen])
    assert set(codes.tolist()) == ({0, 1, 3} if H == 2 else {0, 1, 2, 3})
    assert unordered.sum() >= min(50, len(unordered) // 10)  # late samples inside the kept window


def test_device_rings_at_a_million_slots():
    """Many blocks and the grid's tail: 2^20 + 77 slots, H = 100, every kind, late samples in many rings."""
    n = (1 << 20) + 77
    model, seen = _ring_run(n, 100, 110, {110}, seed=5, busy=0.2)
    assert model.count.max() > 100 and (model.count > 100).sum() >= n // 16
    assert seen[-1][1].sum() > 50_000


# ---- 3. rings through message ingest, and 4. the predict frame on them -----------------------------------------------
class StreamModel:
    """What the reference holds after the same messages: per slot the last H accepted samples in arrival order, and
    the state of the newest accepted message."""

    def __init__(self, H):
        self.H = H
        self.rings = {}
        self.state = {}

    def accept(self, slot, sample, state, history=True):
        if history:
            r = self.rings.setdefault(slot, [])
            r.append(sample)
            del r[: max(0, len(r) - self.H)]
        self.state[slot] = state

    def forget(self, slot):
        self.rings.pop(slot, None)
        self.state.pop(slot, None)

    def histories(self, n):
        hist = np.zeros((n, self.H, 4))
        cnt = np.zeros(n, np.uint32)
        for s, r in self.rings.items():
            hist[s, : len(r)] = r
            cnt[s] = len(r)
        return hist, cnt

    def codes(self, n):
        return _O().patterns(*self.histories(n))


def _arrival_order_code(samples):
    """The classification of a ring walked in arrival order, skipping steps back in time: what the rings gave
    before they were sorted.  Only used to show that the late samples here change emitted pairs."""
    if len(samples) < 2:
        return 3
    sv, sa = np.zeros(3), np.zeros(3)
    nv = na = 0
    pv, pt = np.zeros(3), 0.0
    last = samples[0]
    for cur in samples[1:]:
        dt = cur[3] - last[3]
        if dt > 0:
            v = (cur[:3] - last[:3]) / dt
            if nv > 0 and cur[3] - pt > 0:
                sa += (v - pv) / (cur[3] - pt)
                na += 1
            sv += v
            nv += 1
            pv, pt = v, cur[3]
        last = cur
    if nv == 0:
        return 0
    speed, accel = np.linalg.norm(sv / nv), np.linalg.norm(sa / max(na, 1))
    return 0 if speed < 0.1 else (1 if accel < 0.1 else 2)


def _batch(rng, P, ids, sent, counts, order_seed):
    """One buffer of messages: counts[v] messages of vehicle v (its arrivals sent[v], sent[v] + 1, ...), interleaved
    with the other vehicles' at random but in arrival order per vehicle.  Returns (text, [(vehicle, sample, row)])."""
    veh = np.repeat(np.arange(len(ids)), counts)
    np.random.default_rng(order_seed).shuffle(veh)
    occ = np.zeros(len(veh), np.int64)
    srt = np.argsort(veh, kind="stable")
    starts = np.concatenate([[0], np.cumsum(counts)[:-1]])
    occ[srt] = np.arange(len(veh)) - np.repeat(starts, counts)
    k = sent[veh] + occ
    smp = _samples(P, veh, k)
    rows = {"px": smp[:, 0], "py": smp[:, 1], "pz": smp[:, 2]}
    for c, name in enumerate(("vx", "vy", "vz")):
        rows[name] = P["v"][veh, c].astype(np.float32)
    for c, name in enumerate(("ax", "ay", "az")):
        rows[name] = P["a"][veh, c].astype(np.float32)
    rows["size"] = P["size"][veh]
    rows["heading"] = P["heading"][veh]
    rows["type"] = P["type"][veh]
    text = vehicle_messages(rows, [ids[v] for v in veh], smp[:, 3])
    sent += counts
    return text, veh, occ, smp, rows


def _state_row(rows, q):
    return tuple(float(np.float32(rows[f][q])) for f in ("px", "py", "pz", "vx", "vy", "vz", "ax", "ay", "az", "size",
                                                         "heading")) + (int(rows["type"][q]),)


def test_ingest_rings_and_the_predict_frame_match_the_oracle():
    from rcd_b200.host.ingest import VehiclePositionStream
    O = _O()
    rng = np.random.default_rng(3)
    H, n0, cap0 = 100, 2400, 2600
    total_ids = 3400
    kinds = (STATIONARY, CRUISE, ACCEL, DECEL, LATE_ACCEL, LATE_CRUISE, TIE_GLITCH, REPEATED_T, VERY_LATE)
    P = _params(rng, total_ids, kinds)
    P["kind"][:64] = np.where(np.arange(64) % 2, LATE_ACCEL, VERY_LATE)  # the heavy senders below
    # the vehicles that join after the reserve: accelerating, three messages whose second and third swap (the issue's
    # t = 3.5, 4.0, 3.6), inside one batch for even ones and across two batches for odd ones
    joiners = np.arange(n0 + 180, total_ids)
    P["kind"][joiners], P["period"][joiners] = LATE_ACCEL, 3
    late_accel = np.isin(P["kind"], (LATE_ACCEL, VERY_LATE))
    P["step"][:] = rng.choice([0.1, 0.5], total_ids)
    P["t0"][:] = np.where(rng.random(total_ids) < 0.6, EPOCH + rng.uniform(0, 1e5, total_ids), rng.uniform(0, 50, total_ids))
    # a dense square: accelerating vehicles with late messages have neighbours whose pairs depend on their pattern
    P["p0"][:] = np.column_stack([rng.uniform(0, 700, total_ids), rng.uniform(0, 700, total_ids),
                                  rng.uniform(0, 5, total_ids)])
    P["v"] *= 0.4
    P["size"] = rng.uniform(1.5, 5.0, total_ids).astype(np.float32)
    P["heading"] = rng.uniform(0, 6.28, total_ids).astype(np.float32)
    P["type"] = rng.integers(0, 5, total_ids)
    ids = [f"veh-{k}" for k in range(total_ids)]
    sent = np.zeros(total_ids, np.int64)
    active = np.zeros(total_ids, bool)
    active[:n0] = True
    model = StreamModel(H)
    heavy = {0: 255, 1: 256, 2: 300, 3: 254, 4: 120, 5: 101, 6: 100, 7: 99}  # messages in one batch
    rejected = 0
    with VehiclePositionStream(cap0, 1 << 21, max_history=H) as s:

        def check(tag):
            n = s.ingest.n_objects
            got, want = s.engine.history_classify(), model.codes(n)
            bad = np.flatnonzero(got != want)
            assert len(bad) == 0, (tag, len(bad), int(bad[0]), int(got[bad[0]]), int(want[bad[0]]))
            return want

        def send(b, history=True):
            nonlocal rejected
            counts = np.where(active, rng.choice([0, 1, 1, 1, 2, 3, 5], total_ids), 0)
            counts[active & (sent == 0)] = np.maximum(counts[active & (sent == 0)], 1)  # newcomers speak up
            if b in (1, 4, 6):
                for v, m in heavy.items():
                    counts[v + 8 * b] = m
            if b >= 5:
                counts[joiners[0::2]] = {5: 3, 6: 0, 7: 0}[b]
                counts[joiners[1::2]] = {5: 2, 6: 0, 7: 1}[b]
            text, veh, occ, smp, rows = _batch(rng, P, ids, sent, counts, 100 + b)
            if history:
                s.handle_messages(text)
            else:  # decoded and applied without touching the rings
                rec, ms = s.ingest.decode(text)
                s.engine.apply_records(rec, s.ingest.n_objects, ms, history=False)
            rejected += int(np.maximum(counts - 255, 0).sum())
            assert s.ingest.rejected == rejected, b
            for q in range(len(veh)):
                if occ[q] < 255:  # the 256th and later messages of a vehicle in one batch are dropped
                    model.accept(s.ingest.slot_of(ids[veh[q]]), tuple(smp[q]), _state_row(rows, q), history)

        for b in range(3):
            send(b)
        check("after three batches")
        # departures: the slots go to the next new vehicles, with fresh rings
        gone = rng.choice(np.flatnonzero(active[64:]) + 64, 150, replace=False)
        gone_slots = sorted(s.ingest.slot_of(ids[v]) for v in gone)
        assert sorted(s.remove_vehicles([ids[v] for v in gone])) == sorted(ids[v] for v in gone)
        for sl in gone_slots:
            model.forget(sl)
        active[gone] = False
        active[n0: n0 + 180] = True  # 150 recycled slots + 30 fresh ones
        send(3)
        assert sorted(s.ingest.slot_of(ids[v]) for v in range(n0, n0 + 180)) == gone_slots + list(range(n0, n0 + 30))
        check("recycled slots")
        send(4)
        # more vehicles than the frame holds: reserve keeps every ring and widens the row pitch
        s.reserve(max_objects=4096)
        active[n0 + 180:] = True
        send(5)
        check("after reserve")
        send(6, history=False)
        codes = check("records applied without history")
        send(7)
        codes = check("final")
        assert s.ingest.n_objects == total_ids - 150 and rejected == 3 * (1 + 45)
        # 4. the predict frame on these codes; the vehicle state is each vehicle's newest accepted message
        n = s.ingest.n_objects
        assert sorted(model.state) == list(range(n))
        st = np.array([model.state[sl] for sl in range(n)])
        frame = {f: st[:, c] for c, f in enumerate(("px", "py", "pz", "vx", "vy", "vz", "ax", "ay", "az", "size",
                                                    "heading"))}
        frame["type"] = st[:, 11].astype(np.int32)
        got = s.detect_all_vehicles(predict=True)
        ora = O.frame_A(frame, "predict", pattern_codes=codes)
        compare_pairs(got, ora["risks"], "predict")
        compare_counts(s.engine.counts(), None, ora, "predict", candidates=False)
        # the late messages matter: classified in arrival order, the rings would give other codes and other pairs
        hist, cnt = model.histories(n)
        slots = [s.ingest.slot_of(ids[v]) for v in np.flatnonzero(late_accel & active)]
        alt = codes.copy()
        for sl in slots:
            alt[sl] = _arrival_order_code(hist[sl, : cnt[sl]])
        assert (alt != codes).sum() >= 300
        other = O.frame_A(frame, "predict", pattern_codes=alt)["risks"]
        a = set(zip(ora["risks"]["i"].tolist(), ora["risks"]["j"].tolist()))
        b = set(zip(other["i"].tolist(), other["j"].tolist()))
        assert len(a ^ b) >= 200, len(a ^ b)
