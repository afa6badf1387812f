// Alert lifecycle on the device (SURVEY.md 8f rank 3).  The reference keeps one alert per
// (vehicle, other vehicle) in Python dicts and walks every risk of every frame through them:
//   AlertManager.process_collision_risks / update_alert / create_alert
//                                            src/collision/warning_system.py:259-285, 120-197
//   AlertManager._cleanup_expired_alerts     :488-517   (acknowledged, or older than 30 s)
//   AlertManager.acknowledge_alert           :199-213
// Here the table is an open-addressing hash table in HBM keyed by (i << 32 | j); a frame's emitted
// pairs are folded into it where they lie (the pair buffer never leaves the device) and only the
// CHANGES -- created alerts, priority changes, expiries -- are handed to the host.
//   entry = 48 bytes, 16-byte aligned: {key, state word} in the first 16 bytes, so ONE 16-byte load per probe answers
//   "is this the key" and "what is its alert number / priority / acknowledged bit" (a dependent second access -- a
//   second DRAM access for the quarter of the 40-byte entries of the first layout that straddled a line -- is gone);
//   then timestamp (float64 like time.time()), risk, ttc, distance.  The state word is read and written whole (an
//   update never needs a fence).
// Expiry and the purge of retired vehicles rebuild the table into its twin (no tombstones).
#pragma once
#include <cstddef>
#include "rcd_common.cuh"

namespace rcd {

struct alignas(16) AlertEntry {
    unsigned long long key;  // i << 32 | j; ALERT_EMPTY = free
    // the state word (offset 8): everything an update has to READ.  The creator of an entry writes it LAST, whole; the
    // table is initialised to 0xff.., so an unpublished entry reads alert_id = ALERT_ID_NONE
    u32 alert_id;
    int8_t priority;
    uint8_t acked;
    uint16_t pad;
    double ts;
    float risk, ttc, distance;
    u32 pad2;
};
static_assert(sizeof(AlertEntry) == 48 && offsetof(AlertEntry, alert_id) == 8 && offsetof(AlertEntry, ts) == 16,
              "AlertEntry: 48 bytes, {key, state word} in the first 16");
static_assert(sizeof(rcd_alert_event) == 40, "rcd_alert_event is 40 bytes");
constexpr unsigned long long ALERT_EMPTY = ~0ull;
constexpr u32 ALERT_ID_NONE = 0xffffffffu;  // an entry whose creator has not published it yet

__device__ __forceinline__ unsigned long long alert_state(u32 id, int priority, u32 acked) {
    return (unsigned long long)id | ((unsigned long long)(uint8_t)priority << 32) | ((unsigned long long)(acked & 0xffu) << 40);
}
// timestamp, risk, ttc in one 16-byte store (offset 16 of a 16-byte-aligned entry), distance in a second one
__device__ __forceinline__ void alert_store_values(AlertEntry *a, double now, float risk, float ttc, float distance) {
    const unsigned long long tb = (unsigned long long)__double_as_longlong(now);
    uint4 v;
    v.x = (u32)tb; v.y = (u32)(tb >> 32); v.z = __float_as_uint(risk); v.w = __float_as_uint(ttc);
    *reinterpret_cast<uint4 *>(&a->ts) = v;
    a->distance = distance;
}
__device__ __forceinline__ volatile unsigned long long *alert_state_ptr(AlertEntry *a) {
    return reinterpret_cast<volatile unsigned long long *>(&a->alert_id);
}

struct AlertCounters {
    unsigned long long n_events;     // events appended (may exceed the buffer; only the first cap are stored)
    unsigned long long n_created, n_changed, n_refreshed, n_expired, n_dropped;  // per call
    unsigned long long n_live;       // persists across calls, like next_id
    u32 next_id;
    u32 pad;
};

__device__ __forceinline__ unsigned long long alert_hash(unsigned long long k) {  // splitmix64 finaliser
    k ^= k >> 30; k *= 0xbf58476d1ce4e5b9ull;
    k ^= k >> 27; k *= 0x94d049bb133111ebull;
    k ^= k >> 31;
    return k;
}

// {key, state word} of a slot in one 16-byte access that bypasses L1 (other SMs publish state words during the pass)
__device__ __forceinline__ ulonglong2 alert_load_head(const AlertEntry *a) {
    return __ldcg(reinterpret_cast<const ulonglong2 *>(a));
}

// find the entry of `key`, or claim a free slot for it; nullptr when the table is full.  `state` is the entry's state
// word as the probe saw it (found entries), or the unpublished pattern (the caller re-reads it after a lost race)
__device__ __forceinline__ AlertEntry *alert_find_or_insert(AlertEntry *tab, unsigned long long mask, unsigned long long key,
                                                            bool &inserted, unsigned long long &state) {
    unsigned long long s = alert_hash(key) & mask;
    for (unsigned long long probes = 0; probes <= mask; ++probes, s = (s + 1) & mask) {
        const ulonglong2 head = alert_load_head(tab + s);
        unsigned long long prev = head.x;
        state = head.y;
        if (prev == ALERT_EMPTY) {
            prev = atomicCAS(&tab[s].key, ALERT_EMPTY, key);
            if (prev == key) state = *alert_state_ptr(tab + s);  // lost the race to another copy of the same key
        }
        if (prev == ALERT_EMPTY) { inserted = true; return tab + s; }
        if (prev == key) { inserted = false; return tab + s; }
    }
    return nullptr;
}
__device__ __forceinline__ AlertEntry *alert_find(AlertEntry *tab, unsigned long long mask, unsigned long long key) {
    unsigned long long s = alert_hash(key) & mask;
    for (unsigned long long probes = 0; probes <= mask; ++probes, s = (s + 1) & mask) {
        const unsigned long long k = tab[s].key;
        if (k == key) return tab + s;
        if (k == ALERT_EMPTY) return nullptr;
    }
    return nullptr;
}

// warp-aggregated append of one event per flagged lane
__device__ __forceinline__ void alert_emit(bool flag, const rcd_alert_event &e, rcd_alert_event *ev, unsigned long long cap,
                                           AlertCounters *c) {
    const u32 ballot = __ballot_sync(FULL_MASK, flag);
    if (ballot == 0) return;
    unsigned long long base = 0;
    const u32 leader = __ffs(ballot) - 1;
    if ((threadIdx.x & 31u) == leader) base = atomicAdd(&c->n_events, (unsigned long long)__popc(ballot));
    base = __shfl_sync(FULL_MASK, base, leader);
    if (!flag) return;
    const unsigned long long at = base + __popc(ballot & lanemask_lt());
    if (at < cap) ev[at] = e;
}

constexpr int ALERT_THREADS = 128;

// Fold pairs into the table: every pair with priority >= 0 (risk_level >= RISK_LEVEL_LOW, :273) whose
// `predicted` flag equals `pass` (a frame that ran detect AND predict can carry one risk of each kind for
// the same (i, j); two launches keep "the later risk wins" of the reference's loop deterministic;
// pass < 0 takes every pair).  n_dev (if not null) is the device-side pair count, clamped to n_max.
#ifndef RCD_ALERT_MIN_BLOCKS
#define RCD_ALERT_MIN_BLOCKS 12  // <= 40 registers: a block of the fold fits beside five resident blocks of k_pairs
#endif
__global__ void __launch_bounds__(ALERT_THREADS, RCD_ALERT_MIN_BLOCKS)
k_alert_update(const rcd_pair *__restrict__ pairs, unsigned long long n_max, const unsigned long long *n_dev, int pass,
               double now, AlertEntry *tab, unsigned long long mask, rcd_alert_event *ev, unsigned long long ev_cap,
               AlertCounters *c, int emit_refreshed) {
    const unsigned long long n = n_dev ? min(*n_dev, n_max) : n_max;
    const unsigned long long stride = (unsigned long long)gridDim.x * ALERT_THREADS;
    const unsigned long long rounds = (n + stride - 1) / stride;
    u32 created = 0, changed = 0, refreshed = 0, dropped = 0;
    // A key can occur twice in one pass (a vehicle without history owes the same risk as detect_collisions and as
    // the fall-back of predict_collisions): the thread that loses the insertion may arrive before the winner has
    // filled the entry in.  The winner publishes the entry by writing its state word LAST; a loser that finds it
    // unpublished counts a silent refresh (what the reference's loop does with the second copy: update_alert with
    // the same priority) and, if refreshes are reported, fetches the number after its other work.  Updates of
    // published entries read the state word whole and need no fence: the rest of the entry is only ever written here.
    constexpr int MAX_DEFERRED = 2;
    rcd_alert_event deferred[MAX_DEFERRED];
    volatile u32 *deferred_id[MAX_DEFERRED];
    int n_deferred = 0;
    for (unsigned long long r = 0; r < rounds; ++r) {  // uniform trip count: the emission is warp-wide
        const unsigned long long k = r * stride + (unsigned long long)blockIdx.x * ALERT_THREADS + threadIdx.x;
        bool emit = false;
        rcd_alert_event e;
        e.i = e.j = e.alert_id = 0; e.reserved = 0; e.risk = e.ttc = e.distance = 0.0f; e.priority = e.old_priority = -1; e.kind = 0; e.acknowledged = 0;
        e.timestamp = now;
        if (k < n) {
            const rcd_pair p = pairs[k];
            if (p.priority >= 0 && (pass < 0 || (int)p.predicted == pass)) {
                const unsigned long long key = ((unsigned long long)p.i << 32) | p.j;
                bool inserted = false;
                unsigned long long st = 0;
                AlertEntry *a = alert_find_or_insert(tab, mask, key, inserted, st);
                if (!a) {
                    ++dropped;
                } else {
                    e.i = p.i; e.j = p.j; e.risk = p.risk; e.ttc = p.ttc; e.distance = p.distance; e.priority = p.priority;
                    volatile unsigned long long *sp = alert_state_ptr(a);
                    volatile u32 *idp = &a->alert_id;
                    if (inserted) {  // create_alert (:120-160)
                        a->pad2 = 0;
                        alert_store_values(a, now, p.risk, p.ttc, p.distance);
                        e.alert_id = atomicAdd(&c->next_id, 1u);
                        __threadfence();
                        *sp = alert_state(e.alert_id, p.priority, 0u);  // publishes the entry
                        e.kind = RCD_ALERT_CREATED;
                        e.old_priority = -1;
                        ++created;
                        emit = true;
                    } else {
                        e.alert_id = (u32)st;
                        if (e.alert_id == ALERT_ID_NONE) {  // being created by another thread of this pass
                            e.kind = RCD_ALERT_REFRESHED;
                            e.old_priority = p.priority;
                            ++refreshed;
                            if (emit_refreshed) {
                                if (n_deferred < MAX_DEFERRED) { deferred[n_deferred] = e; deferred_id[n_deferred] = idp; ++n_deferred; }
                                else emit = true;
                            }
                        } else {     // update_alert (:162-197): the priority queue only hears of priority changes
                            const int old_priority = (int)(int8_t)((st >> 32) & 0xffu);
                            const u32 acked = (u32)((st >> 40) & 0xffu);
                            e.old_priority = (int8_t)old_priority;
                            e.acknowledged = (uint8_t)acked;
                            alert_store_values(a, now, p.risk, p.ttc, p.distance);
                            if (old_priority != (int)p.priority) {
                                *sp = alert_state(e.alert_id, p.priority, acked);
                                e.kind = RCD_ALERT_PRIORITY_CHANGED; ++changed; emit = true;
                            } else { e.kind = RCD_ALERT_REFRESHED; ++refreshed; emit = emit_refreshed != 0; }
                        }
                    }
                }
            }
        }
        alert_emit(emit, e, ev, ev_cap, c);
    }
    const int max_deferred = __reduce_max_sync(FULL_MASK, n_deferred);
    for (int d = 0; d < max_deferred; ++d) {
        rcd_alert_event e = deferred[d < n_deferred ? d : 0];
        if (d < n_deferred) e.alert_id = *deferred_id[d];
        alert_emit(d < n_deferred, e, ev, ev_cap, c);
    }
    unsigned long long v[4] = {created, changed, refreshed, dropped};
#pragma unroll
    for (int q = 0; q < 4; ++q) v[q] = warp_sum(v[q]);
    if ((threadIdx.x & 31u) == 0) {
        if (v[0]) { atomicAdd(&c->n_created, v[0]); atomicAdd(&c->n_live, v[0]); }
        if (v[1]) atomicAdd(&c->n_changed, v[1]);
        if (v[2]) atomicAdd(&c->n_refreshed, v[2]);
        if (v[3]) atomicAdd(&c->n_dropped, v[3]);
    }
}

// _cleanup_expired_alerts (:488-517): acknowledged or now - timestamp > max_age
struct AlertTooOld {
    double now, max_age;
    __device__ __forceinline__ bool operator()(const AlertEntry &a) const { return a.acked || __dsub_rn(now, a.ts) > max_age; }
};

// rcd_retire: i or j is the caller id of a retired slot.  ids: sorted, distinct (any u32 values: upload-built frames
// carry the caller's ids); a binary search per entry, retire batches being small next to the table.
struct AlertOfRetired {
    const u32 *ids;
    u32 n;
    __device__ __forceinline__ bool has(u32 v) const {
        u32 lo = 0, hi = n;
        while (lo < hi) {
            const u32 mid = (lo + hi) >> 1;
            if (__ldg(ids + mid) < v) lo = mid + 1; else hi = mid;
        }
        return lo < n && __ldg(ids + lo) == v;
    }
    __device__ __forceinline__ bool operator()(const AlertEntry &a) const {
        return has((u32)(a.key >> 32)) || has((u32)(a.key & 0xffffffffu));
    }
};

// rcd_alerts_reserve: every entry moves to a larger table of dst_mask + 1 slots
struct AlertKeep {
    unsigned long long dst_mask;
    __device__ __forceinline__ bool operator()(const AlertEntry &) const { return false; }
};
// The slot mask of the table a rebuild writes: the twin of the same size, unless the predicate brings its own.  (A
// compile-time choice: the expire and purge rebuilds keep the registers they had before rcd_alerts_reserve.)
template <typename Drop>
__device__ __forceinline__ unsigned long long rebuild_dst_mask(const Drop &, unsigned long long cap) { return cap - 1; }
__device__ __forceinline__ unsigned long long rebuild_dst_mask(const AlertKeep &k, unsigned long long) { return k.dst_mask; }

// Rebuild the table into an empty one (no tombstones): every entry `drop` selects -> EXPIRED event; everything else
// moves to dst.  Drop = AlertTooOld: rcd_alerts_expire; AlertOfRetired: the purge of rcd_retire (both into the twin);
// AlertKeep: rcd_alerts_reserve (into a larger table).
template <typename Drop>
__global__ void __launch_bounds__(ALERT_THREADS)
k_alert_rebuild(const AlertEntry *__restrict__ src, unsigned long long cap, Drop drop, AlertEntry *dst,
                rcd_alert_event *ev, unsigned long long ev_cap, AlertCounters *c) {
    const unsigned long long stride = (unsigned long long)gridDim.x * ALERT_THREADS;
    const unsigned long long rounds = (cap + stride - 1) / stride;
    u32 expired = 0, live = 0;
    for (unsigned long long r = 0; r < rounds; ++r) {
        const unsigned long long k = r * stride + (unsigned long long)blockIdx.x * ALERT_THREADS + threadIdx.x;
        bool emit = false;
        rcd_alert_event e;
        e.i = e.j = e.alert_id = 0; e.reserved = 0; e.risk = e.ttc = e.distance = 0.0f; e.priority = e.old_priority = -1; e.kind = RCD_ALERT_EXPIRED;
        e.acknowledged = 0; e.timestamp = 0.0;
        if (k < cap) {
            const AlertEntry a = src[k];
            if (a.key != ALERT_EMPTY) {
                if (drop(a)) {
                    e.i = (u32)(a.key >> 32); e.j = (u32)(a.key & 0xffffffffu); e.alert_id = a.alert_id;
                    e.risk = a.risk; e.ttc = a.ttc; e.distance = a.distance; e.priority = e.old_priority = a.priority; e.acknowledged = a.acked;
                    e.timestamp = a.ts;
                    emit = true;
                    ++expired;
                } else {
                    bool inserted = false;
                    unsigned long long st_unused = 0;
                    AlertEntry *d = alert_find_or_insert(dst, rebuild_dst_mask(drop, cap), a.key, inserted,
                                                         st_unused);  // at least as large: always fits
                    d->ts = a.ts; d->risk = a.risk; d->ttc = a.ttc; d->distance = a.distance; d->alert_id = a.alert_id;
                    d->priority = a.priority; d->acked = a.acked; d->pad = 0; d->pad2 = 0;
                    ++live;
                }
            }
        }
        alert_emit(emit, e, ev, ev_cap, c);
    }
    unsigned long long x = warp_sum((unsigned long long)expired), l = warp_sum((unsigned long long)live);
    if ((threadIdx.x & 31u) == 0) {
        if (x) atomicAdd(&c->n_expired, x);
        if (l) atomicAdd(&c->n_live, l);
    }
}

// acknowledge_alert (:199-213), addressed by (i, j)
__global__ void __launch_bounds__(ALERT_THREADS)
k_alert_ack(const u32 *__restrict__ i, const u32 *__restrict__ j, u32 n, AlertEntry *tab, unsigned long long mask, u32 *found) {
    const u32 k = blockIdx.x * ALERT_THREADS + threadIdx.x;
    if (k >= n) return;
    AlertEntry *a = alert_find(tab, mask, ((unsigned long long)i[k] << 32) | j[k]);
    if (a) { a->acked = 1; atomicAdd(found, 1u); }
}

// every live alert as an event record (kind = RCD_ALERT_REFRESHED), unordered
__global__ void __launch_bounds__(ALERT_THREADS)
k_alert_dump(const AlertEntry *__restrict__ tab, unsigned long long cap, rcd_alert_event *ev, unsigned long long ev_cap,
             AlertCounters *c) {
    const unsigned long long stride = (unsigned long long)gridDim.x * ALERT_THREADS;
    const unsigned long long rounds = (cap + stride - 1) / stride;
    for (unsigned long long r = 0; r < rounds; ++r) {
        const unsigned long long k = r * stride + (unsigned long long)blockIdx.x * ALERT_THREADS + threadIdx.x;
        bool emit = false;
        rcd_alert_event e;
        e.i = e.j = e.alert_id = 0; e.reserved = 0; e.risk = e.ttc = e.distance = 0.0f; e.priority = e.old_priority = -1; e.kind = RCD_ALERT_REFRESHED;
        e.acknowledged = 0; e.timestamp = 0.0;
        if (k < cap) {
            const AlertEntry a = tab[k];
            if (a.key != ALERT_EMPTY) {
                e.i = (u32)(a.key >> 32); e.j = (u32)(a.key & 0xffffffffu); e.alert_id = a.alert_id;
                e.risk = a.risk; e.ttc = a.ttc; e.distance = a.distance; e.priority = e.old_priority = a.priority; e.acknowledged = a.acked;
                e.timestamp = a.ts;
                emit = true;
            }
        }
        alert_emit(emit, e, ev, ev_cap, c);
    }
}

}  // namespace rcd
