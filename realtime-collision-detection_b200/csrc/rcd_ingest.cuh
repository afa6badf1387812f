// Device side of batched ingest: scatter decoded vehicle records (include/rcd.h, rcd_record) into the
// frame's SoA state and append their (x, y, z, t) float64 samples to the trajectory rings.  Replaces, per
// message, CollisionDetector.update_vehicle + CollisionPredictionModel.update_trajectory as called
// from EarlyWarningSystem._handle_vehicle_position (src/collision/warning_system.py:638-678,
// collision_detection.py:74-85, 553-570).
// Algorithmic bytes per record: 72 read + 58 written (state 50 + last_seen 8; + 32 into the ring + 4 ring counter r/w).
// Retirement (rcd_retire, rcd_retire_stale): k_stale_count / k_scan_tiles / k_stale_scatter select the slots whose
// newest record is too old, k_retire_slots turns slots into objects without a position.
#pragma once
#include "rcd_common.cuh"
#include "rcd_pairs.cuh"  // Sample64, MutableState

namespace rcd {

constexpr int APPLY_THREADS = 256;
constexpr int RECORD_WORDS = sizeof(rcd_record) / 8;  // 9 x 8 bytes

// A block stages its 256 records through shared memory with coalesced 8-byte loads (consecutive threads
// read consecutive words), then each thread takes one record.  Only records whose `seq` equals the
// launch's are applied: a batch with several messages for one vehicle is applied in `max_seq + 1`
// launches, which keeps "the last message wins" and the order of the ring samples deterministic.
__global__ void __launch_bounds__(APPLY_THREADS)
k_apply_records(u32 n, const unsigned long long *__restrict__ recs, u32 seq, u32 n_objects, MutableState st,
                Sample64 *__restrict__ hist, u32 *__restrict__ count, u32 cap, u32 H, double *__restrict__ last_seen) {
    __shared__ unsigned long long s_rec[APPLY_THREADS * RECORD_WORDS + APPLY_THREADS / 8];
    const u32 base = blockIdx.x * APPLY_THREADS;
    const u32 m = min((u32)APPLY_THREADS, n - base);
    const unsigned long long *src = recs + (size_t)base * RECORD_WORDS;
    for (u32 w = threadIdx.x; w < m * RECORD_WORDS; w += APPLY_THREADS) s_rec[w + w / 72] = __ldcs(src + w);
    __syncthreads();
    if (threadIdx.x >= m) return;
    // (one padding word per 8 records keeps the 9-word stride off the same banks)
    auto word = [&](u32 k) { const u32 w = threadIdx.x * RECORD_WORDS + k; return s_rec[w + w / 72]; };
    const unsigned long long tail = word(8);
    const u32 slot = (u32)(tail & 0xffffffffu);
    const u32 type = (u32)((tail >> 32) & 0xffu), rseq = (u32)((tail >> 40) & 0xffu);
    if (rseq != seq || slot >= n_objects) return;
    const double x = __longlong_as_double((long long)word(0)), y = __longlong_as_double((long long)word(1)),
                 z = __longlong_as_double((long long)word(2)), t = __longlong_as_double((long long)word(3));
    st.f[0][slot] = (float)x;
    st.f[1][slot] = (float)y;
    st.f[2][slot] = (float)z;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const unsigned long long w = word(4 + k);
        st.f[3 + 2 * k][slot] = __uint_as_float((u32)(w & 0xffffffffu));
        st.f[4 + 2 * k][slot] = __uint_as_float((u32)(w >> 32));
    }
    st.type[slot] = (uint8_t)type;
    last_seen[slot] = t;  // (the launch of the slot's last seq runs last: the newest message's time stays)
    if (hist) {
        const u32 c = count[slot];
        Sample64 v;
        v.x = x; v.y = y; v.z = z; v.t = t;
        hist[(size_t)(c % H) * cap + slot] = v;
        count[slot] = c + 1;
    }
}

// a slot without a record time: now - t > max_age is false for every now (NaN; also what a 0xff memset leaves)
__device__ __forceinline__ double no_record_time() { return __longlong_as_double(-1ll); }

// new slots: ids = slot index, default pattern, no record time
__global__ void __launch_bounds__(256) k_init_slots(u32 first, u32 n, u32 *__restrict__ id, uint8_t *__restrict__ pattern,
                                                    double *__restrict__ last_seen) {
    u32 i = first + blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        id[i] = i;
        pattern[i] = RCD_PAT_ACCELERATING;
        last_seen[i] = no_record_time();
    }
}

// ---- stale-slot selection: the slots s < n with now - last_seen[s] > max_age, in ascending order ----------------
// Two passes over last_seen (count per tile, then scatter at the tile's exclusive prefix) with a one-block scan of the
// tile counts between them.  Chosen over a single pass with a cross-block fix-up because the output order then falls
// out of the tile order with no inter-block protocol, and the second read is cheap: last_seen is 8 B/slot (80 MB at
// 10 M slots), so the scatter pass finds it in L2 after the count pass.  Each warp reads STALE_ITEMS coalesced 256-byte
// rows; a ballot per row keeps the order inside the warp, a scan over the warps the order inside the tile.
constexpr int STALE_THREADS = 256;
constexpr int STALE_ITEMS = 8;
constexpr u32 STALE_TILE = STALE_THREADS * STALE_ITEMS;  // 2048 slots

__device__ __forceinline__ bool is_stale(double t, double now, double max_age) { return __dsub_rn(now, t) > max_age; }

// stale-slot mask of row k of this warp's part of the tile (bit l: slot base + k * 32 + l)
__device__ __forceinline__ u32 stale_row(const double *__restrict__ last_seen, u32 n, u32 base, int k, double now,
                                         double max_age) {
    const u32 s = base + (u32)k * 32u + (threadIdx.x & 31u);
    return __ballot_sync(FULL_MASK, s < n && is_stale(__ldg(last_seen + s), now, max_age));  // (kept in L2 for the scatter)
}

__global__ void __launch_bounds__(STALE_THREADS)
k_stale_count(const double *__restrict__ last_seen, u32 n, double now, double max_age, u32 *__restrict__ tile_count) {
    __shared__ u32 s_warp[STALE_THREADS / 32];
    const u32 warp = threadIdx.x >> 5;
    const u32 base = blockIdx.x * STALE_TILE + warp * (STALE_ITEMS * 32);
    u32 c = 0;
#pragma unroll
    for (int k = 0; k < STALE_ITEMS; ++k) c += __popc(stale_row(last_seen, n, base, k, now, max_age));
    if ((threadIdx.x & 31u) == 0) s_warp[warp] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        u32 t = 0;
        for (int w = 0; w < STALE_THREADS / 32; ++w) t += s_warp[w];
        tile_count[blockIdx.x] = t;
    }
}

// exclusive scan of the tile counts in place (one block, any number of tiles); tile_count[tiles] = total
__global__ void __launch_bounds__(1024) k_scan_tiles(u32 *__restrict__ tile_count, u32 tiles) {
    __shared__ u32 s_warp[32];
    __shared__ u32 s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (u32 base = 0; base < tiles; base += 1024) {
        const u32 t = base + threadIdx.x;
        const u32 v = t < tiles ? tile_count[t] : 0u;
        u32 incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const u32 x = __shfl_up_sync(FULL_MASK, incl, o);
            if (lane_id() >= (u32)o) incl += x;
        }
        if (lane_id() == 31) s_warp[threadIdx.x >> 5] = incl;
        __syncthreads();
        u32 before = s_carry;
        for (u32 w = 0; w < (threadIdx.x >> 5); ++w) before += s_warp[w];
        if (t < tiles) tile_count[t] = before + incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = before + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) tile_count[tiles] = s_carry;
}

__global__ void __launch_bounds__(STALE_THREADS)
k_stale_scatter(const double *__restrict__ last_seen, u32 n, double now, double max_age, const u32 *__restrict__ tile_base,
                u32 *__restrict__ out) {
    __shared__ u32 s_warp[STALE_THREADS / 32];
    const u32 warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const u32 base = blockIdx.x * STALE_TILE + warp * (STALE_ITEMS * 32);
    u32 mask[STALE_ITEMS], c = 0;
#pragma unroll
    for (int k = 0; k < STALE_ITEMS; ++k) {
        mask[k] = stale_row(last_seen, n, base, k, now, max_age);
        c += __popc(mask[k]);
    }
    if (lane == 0) s_warp[warp] = c;
    __syncthreads();
    u32 at = tile_base[blockIdx.x];
    for (u32 w = 0; w < warp; ++w) at += s_warp[w];
#pragma unroll
    for (int k = 0; k < STALE_ITEMS; ++k) {
        if (mask[k] & (1u << lane)) out[at + __popc(mask[k] & lanemask_lt())] = base + (u32)k * 32u + lane;
        at += __popc(mask[k]);
    }
}

// Retire the listed slots: the ghost state of the halo exchange (every float field all bits set: no position), type 0,
// the default pattern, an empty trajectory ring, no record time.  The caller id stays (a later record brings the slot
// back under it); ids_out[k] receives the id of slots[k] for the alert purge.  Repeats write the same values.
// Bytes per slot: 4 (list) + 4 (id) read, 44 + 1 + 1 + 4 (ring count) + 8 (last_seen) + 4 (id out) written.
__global__ void __launch_bounds__(256)
k_retire_slots(const u32 *__restrict__ slots, u32 n, MutableState st, u32 *__restrict__ ring_count,
               double *__restrict__ last_seen, u32 *__restrict__ ids_out) {
    const u32 k = blockIdx.x * 256 + threadIdx.x;
    if (k >= n) return;
    const u32 s = slots[k];
#pragma unroll
    for (int f = 0; f < 11; ++f) st.f[f][s] = __uint_as_float(0xffffffffu);
    st.type[s] = 0;
    st.pattern[s] = RCD_PAT_ACCELERATING;
    if (ring_count) ring_count[s] = 0;
    if (last_seen) last_seen[s] = no_record_time();
    ids_out[k] = st.id[s];
}

}  // namespace rcd
