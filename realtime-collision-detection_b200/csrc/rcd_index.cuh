// Spatial index build: cell keys -> hand-written onesweep radix sort -> cell-ordered packed
// state + cell ranges.  Replaces the per-vehicle dict/set churn of SpatialIndex.insert_vehicle
// (src/collision/spatial_index.py:162-227) and compute_node.SpatialIndex.insert
// (src/compute/compute_node.py:55-96) with one whole-frame rebuild, which is also what the
// reference's perf harness times (src/test/performance_test.py:794-800: clear + N x insert).
#pragma once
#include "rcd_common.cuh"

namespace rcd {

constexpr int RADIX_BITS = 8;
constexpr int RADIX = 1 << RADIX_BITS;
constexpr int MAX_PASSES = 4;

// SoA input state as uploaded (device pointers)
struct InputState {
    const float *px, *py, *pz, *vx, *vy, *vz, *ax, *ay, *az, *size, *heading;
    const uint8_t *type;
    const uint8_t *pattern;
    const u32 *id;  // may be null -> identity
};

// -------------------------------------------------------------------------------------------------
// K1: one pass over the SoA state: cell keys + digit histograms of every sort pass, and the state
// packed into one 64-byte-aligned record per object in upload order
// ({x,y,z,size | vx,vy,vz,heading | ax,ay,az,meta | id,-,-,-}), so that the gather after the sort reads
// ONE aligned 64-byte block per object (the DRAM access granule) instead of thirteen scattered 4-byte
// fields.  The first sort pass needs no permutation array: its values are the positions themselves.
// Algorithmic bytes: 50 N read + 4 N (keys) + 52 N (records; 64 N with the padding) written = 106 N.
// -------------------------------------------------------------------------------------------------
constexpr int KEYS_THREADS = 256;

__device__ __forceinline__ u32 pack_meta(u32 type, u32 pattern, bool owned) {
    return type | ((pattern & 3u) << 8) | (owned ? META_OWNED : 0u);
}

__global__ void __launch_bounds__(KEYS_THREADS)
k_pack_keys(InputState in, u32 n, u32 n_owned, GridParams g, int passes, u32 *__restrict__ keys,
            u32 *__restrict__ hist /* [MAX_PASSES][RADIX] */,
            float4 *__restrict__ U /* [n][4]: one 64-byte record per object */) {
    __shared__ u32 s_hist[MAX_PASSES][RADIX];
    __shared__ float4 s_rec[KEYS_THREADS / 32][128];  // a warp's 32 records on their way to four dense 512-byte stores
    for (int k = threadIdx.x; k < MAX_PASSES * RADIX; k += KEYS_THREADS) (&s_hist[0][0])[k] = 0;
    __syncthreads();
    // one object per thread: every field load and the key store are fully coalesced 128-byte warp requests; the
    // records are turned through shared memory so that a warp stores its 2 KB span as four dense 512-byte requests
    // (16 full sectors each) instead of 4 x 32 half sectors
    const u32 stride = gridDim.x * KEYS_THREADS;
    const u32 lane = threadIdx.x & 31u;
    const u32 n_round = (n + 31u) & ~31u;  // whole warps run the loop: the staged stores are warp-wide
    for (u32 i = blockIdx.x * KEYS_THREADS + threadIdx.x; i < n_round; i += stride) {
        const bool live = i < n;
        const u32 il = live ? i : n - 1;
        const float x = __ldcs(in.px + il), y = __ldcs(in.py + il), z = __ldcs(in.pz + il);
        const float4 r0 = make_float4(x, y, z, __ldcs(in.size + il));
        const float4 r1 = make_float4(__ldcs(in.vx + il), __ldcs(in.vy + il), __ldcs(in.vz + il), __ldcs(in.heading + il));
        const u32 meta = pack_meta(__ldcs(in.type + il), __ldcs(in.pattern + il), il < n_owned);
        const float4 r2 = make_float4(__ldcs(in.ax + il), __ldcs(in.ay + il), __ldcs(in.az + il), __uint_as_float(meta));
        const float4 r3 = make_float4(__uint_as_float(__ldcs(in.id + il)), 0.0f, 0.0f, 0.0f);
        // objects without a position (NaN: ghost slots of the halo exchange, rcd_halo_pack_async) go to a cell of
        // their own behind the grid, which is under no query's box
        const u32 k = (x == x && y == y && z == z) ? cell_key(g, x, y, z) : g.ncells;
        if (live) keys[i] = k;
        {
            float4 *w = s_rec[threadIdx.x >> 5];
            // quarter q of record l sits at slot 4 l + (q ^ ((l >> 1) & 3)): both the per-object writes (64-byte stride)
            // and the dense reads below touch eight different 16-byte bank groups per quarter-warp
            const u32 sw = (lane >> 1) & 3u;
            w[4 * lane + (0u ^ sw)] = r0;
            w[4 * lane + (1u ^ sw)] = r1;
            w[4 * lane + (2u ^ sw)] = r2;
            w[4 * lane + (3u ^ sw)] = r3;
            __syncwarp();
            const u32 base = i - lane;  // first object of the warp
            float4 *dst = U + 4 * (size_t)base;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const u32 e = j * 32 + lane, o = e >> 2, q = e & 3u;
                if (base + o < n) dst[e] = w[4 * o + (q ^ ((o >> 1) & 3u))];
            }
            __syncwarp();
        }
        if (live)
            for (int p = 0; p < passes; ++p) atomicAdd(&s_hist[p][(k >> (p * RADIX_BITS)) & (RADIX - 1)], 1u);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < passes * RADIX; k += KEYS_THREADS) {
        u32 c = (&s_hist[0][0])[k];
        if (c) atomicAdd(&hist[k], c);
    }
}

// K2: exclusive scan of each pass's 256-bin histogram (one block, one warp per 32 bins).
__global__ void __launch_bounds__(RADIX) k_scan_hist(u32 *__restrict__ hist, int passes) {
    __shared__ u32 s_warp[RADIX / 32];
    for (int p = 0; p < passes; ++p) {
        u32 v = hist[p * RADIX + threadIdx.x];
        u32 incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            u32 t = __shfl_up_sync(FULL_MASK, incl, o);
            if (lane_id() >= (u32)o) incl += t;
        }
        if (lane_id() == 31) s_warp[threadIdx.x >> 5] = incl;
        __syncthreads();
        u32 base = 0;
        for (u32 w = 0; w < (threadIdx.x >> 5); ++w) base += s_warp[w];
        hist[p * RADIX + threadIdx.x] = base + incl - v;
        __syncthreads();
    }
}

// -------------------------------------------------------------------------------------------------
// K3: one onesweep pass (LSD, 8-bit digit): a single read and a single write of keys + values
// per pass.  Tiles take tickets from an atomic counter, so a tile only ever waits on tiles that
// are already running (decoupled look-back, forward progress guaranteed inside one launch).
// Ranking is stable: warp-striped loads, per-warp digit counters updated with match.any.
// IDENTITY (the first pass): the values are the positions, nothing is read for them.
// Algorithmic bytes per pass: 8 N read (4 N on the first pass) + 8 N written.
// -------------------------------------------------------------------------------------------------
#ifndef RCD_SORT_ITEMS
#define RCD_SORT_ITEMS 16
#endif
#ifndef RCD_SORT_CTAS
#define RCD_SORT_CTAS 3
#endif
#ifndef RCD_SORT_LOOKBACK
#define RCD_SORT_LOOKBACK 8
#endif
#ifndef RCD_SORT_ABLATE  // timing experiments only (WRONG RESULTS): 1 no global stores, 2 | 16 no look-back (16: stores bound-checked)
#define RCD_SORT_ABLATE 0
#endif
constexpr int SORT_THREADS = 256;
constexpr int SORT_WARPS = SORT_THREADS / 32;
constexpr int SORT_ITEMS = RCD_SORT_ITEMS;
constexpr int SORT_TILE = SORT_THREADS * SORT_ITEMS;  // 4096 keys
constexpr u32 STATUS_AGGREGATE = 1u << 30;
constexpr u32 STATUS_PREFIX = 2u << 30;
constexpr u32 STATUS_VALUE_MASK = (1u << 30) - 1u;

// look-back status words: gpu-scope relaxed accesses (the word carries its own flag, no fence needed)
__device__ __forceinline__ u32 ld_status(const u32 *p) {
    u32 v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_status(u32 *p, u32 v) {
    asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// lanes of the warp holding the same 8-bit digit: eight independent ballots pipeline far better
// than one MATCH.ANY (whose latency the ranking chain would pay once per item).  Written in PTX so that
// every bit costs four instructions (test, vote, select, and-xor) instead of the seven nvcc makes of the
// C++ form: peers &= vote ^ (bit ? 0 : ~0).
__device__ __forceinline__ u32 match_digit(u32 digit, u32 peers /* lanes that take part */) {
#pragma unroll
    for (int b = 0; b < RADIX_BITS; ++b) {
        u32 t;
        asm("{\n\t.reg .pred p;\n\t.reg .b32 v, m, a;\n\t"
            "and.b32 a, %1, %2;\n\t"
            "setp.ne.u32 p, a, 0;\n\t"
            "vote.sync.ballot.b32 v, p, 0xffffffff;\n\t"
            "selp.b32 m, 0, 0xffffffff, p;\n\t"
            "xor.b32 %0, v, m;\n\t}"
            : "=r"(t) : "r"(digit), "r"(1u << b));
        peers &= t;
    }
    return peers;
}

// One tile of one pass.  FULL: the tile holds SORT_TILE keys (every tile but the last): no bound checks.
template <bool FULL, bool IDENTITY>
__device__ __forceinline__ void onesweep_tile(const u32 *__restrict__ keys_in, const u32 *__restrict__ vals_in,
                                              u32 *__restrict__ keys_out, u32 *__restrict__ vals_out, u32 tile,
                                              u32 tile_count, int shift, const u32 *__restrict__ digit_base,
                                              u32 *tile_status, u32 (*s_warp_hist)[RADIX], u32 *s_digit_excl,
                                              u32 *s_global_base, u32 *s_scan, uint2 *s_kv) {
    const u32 tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const u32 tile_base = tile * SORT_TILE;
    // ---- load (warp-striped: item k of lane l is element warp*ITEMS*32 + k*32 + l) and rank ----
    u32 key[SORT_ITEMS], val[SORT_ITEMS], rank[SORT_ITEMS];
    const u32 warp_base = warp * (SORT_ITEMS * 32);
    const u32 *kin = keys_in + tile_base + warp_base + lane;
    const u32 *vin = vals_in + tile_base + warp_base + lane;
#pragma unroll
    for (int k = 0; k < SORT_ITEMS; ++k) {
        const bool valid = FULL || warp_base + k * 32 + lane < tile_count;
        key[k] = valid ? __ldcs(kin + k * 32) : 0xffffffffu;
        if (!IDENTITY) val[k] = valid ? __ldcs(vin + k * 32) : 0u;
    }
    const u32 lt = lanemask_lt();
    u32 *my_hist = s_warp_hist[warp];
#pragma unroll
    for (int k = 0; k < SORT_ITEMS; ++k) {
        const u32 digit = (key[k] >> shift) & (RADIX - 1);
        // invalid lanes are in nobody's group and do not touch the counters
        const bool valid = FULL || warp_base + k * 32 + lane < tile_count;
        const u32 group = match_digit(digit, FULL ? FULL_MASK : __ballot_sync(FULL_MASK, valid));
        // every lane of a group reads the counter (one broadcast per digit), the lowest lane advances it
        const u32 before = my_hist[digit];
        __syncwarp();
        if ((group & lt) == 0 && valid) my_hist[digit] = before + __popc(group);
        rank[k] = before + __popc(group & lt);
        __syncwarp();
    }
    __syncthreads();

    // ---- per digit (thread d): exclusive scan over warps, tile total ---------------------------
    u32 total = 0;
#pragma unroll
    for (int w = 0; w < SORT_WARPS; ++w) {
        u32 c = s_warp_hist[w][tid];
        s_warp_hist[w][tid] = total;
        total += c;
    }
    // publish this tile's digit count as early as possible
    if (tile == 0) {
        st_status(tile_status + tid, STATUS_PREFIX | total);
    } else {
        st_status(tile_status + (size_t)tile * RADIX + tid, STATUS_AGGREGATE | total);
    }
    // exclusive scan of the 256 digit totals -> start of each digit inside the sorted tile
    {
        u32 incl = total;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            u32 t = __shfl_up_sync(FULL_MASK, incl, o);
            if (lane >= (u32)o) incl += t;
        }
        if (lane == 31) s_scan[warp] = incl;
        __syncthreads();
        u32 base = 0;
        for (u32 w = 0; w < warp; ++w) base += s_scan[w];
        s_digit_excl[tid] = base + incl - total;
    }
    __syncthreads();
    // ---- scatter (key, value) into shared memory in sorted order.  Done BEFORE the look-back: it needs
    // only tile-local offsets, and the predecessors' prefixes have that much longer to arrive.
#pragma unroll
    for (int k = 0; k < SORT_ITEMS; ++k) {
        if (FULL || warp_base + k * 32 + lane < tile_count) {
            const u32 digit = (key[k] >> shift) & (RADIX - 1);
            const u32 pos = s_digit_excl[digit] + my_hist[digit] + rank[k];
            s_kv[pos] = make_uint2(key[k], IDENTITY ? tile_base + warp_base + k * 32 + lane : val[k]);
        }
    }
    // ---- decoupled look-back for digit `tid` ----------------------------------------------------
    // Up to LOOKBACK predecessors are fetched with independent loads and then consumed in order, so a
    // long run of AGGREGATE tiles costs one memory latency per batch instead of one per tile.
    u32 excl = 0;
    if (tile > 0 && !(RCD_SORT_ABLATE & 2)) {
        constexpr int LOOKBACK = RCD_SORT_LOOKBACK;
        int t = (int)tile - 1;
        bool done = false;
        while (!done) {
            u32 st[LOOKBACK];
#pragma unroll
            for (int k = 0; k < LOOKBACK; ++k)
                st[k] = (t - k >= 0) ? ld_status(tile_status + (size_t)(t - k) * RADIX + tid) : STATUS_PREFIX;
#pragma unroll
            for (int k = 0; k < LOOKBACK; ++k) {
                if (done) break;
                const u32 flag = st[k] & ~STATUS_VALUE_MASK;
                if (flag == 0) break;  // that predecessor holds a ticket, so it is running: fetch again from it
                excl += st[k] & STATUS_VALUE_MASK;
                --t;
                if (flag == STATUS_PREFIX) done = true;
            }
        }
        st_status(tile_status + (size_t)tile * RADIX + tid, STATUS_PREFIX | (excl + total));
    }
    s_global_base[tid] = digit_base[tid] + excl - s_digit_excl[tid];
    __syncthreads();

    // ---- write the sorted tile's runs to global ------------------------------------------------
#pragma unroll
    for (int k = 0; k < SORT_ITEMS; ++k) {
        const u32 idx = k * SORT_THREADS + tid;
        if (FULL || idx < tile_count) {
            const uint2 kv = s_kv[idx];
            const u32 out = s_global_base[(kv.x >> shift) & (RADIX - 1)] + idx;
#if RCD_SORT_ABLATE & 1
            if (kv.x == 0xdeadbeefu && kv.y == 0x12345678u && out == 0x0badf00du)
#elif RCD_SORT_ABLATE & 16
            if (out < (gridDim.x - 1u) * SORT_TILE)
#endif
            {
                keys_out[out] = kv.x;
                vals_out[out] = kv.y;
            }
        }
    }
}

template <bool IDENTITY>
__global__ void __launch_bounds__(SORT_THREADS, RCD_SORT_CTAS)
k_onesweep_pass(const u32 *__restrict__ keys_in, const u32 *__restrict__ vals_in,
                u32 *__restrict__ keys_out, u32 *__restrict__ vals_out, u32 n, int shift,
                const u32 *__restrict__ digit_base /* [RADIX] exclusive, this pass */,
                u32 *tile_status /* [tiles][RADIX], zeroed */, u32 *tile_counter) {
    __shared__ u32 s_warp_hist[SORT_WARPS][RADIX];
    __shared__ u32 s_digit_excl[RADIX];
    __shared__ u32 s_global_base[RADIX];
    __shared__ u32 s_scan[SORT_WARPS];
    __shared__ uint2 s_kv[SORT_TILE];
    __shared__ u32 s_tile;

    const u32 tid = threadIdx.x;
    if (tid == 0) s_tile = atomicAdd(tile_counter, 1u);
    for (int k = tid; k < SORT_WARPS * RADIX; k += SORT_THREADS) (&s_warp_hist[0][0])[k] = 0;
    __syncthreads();
    const u32 tile = s_tile;
    const u32 tile_count = min((u32)SORT_TILE, n - tile * SORT_TILE);
    if (tile_count == SORT_TILE)
        onesweep_tile<true, IDENTITY>(keys_in, vals_in, keys_out, vals_out, tile, tile_count, shift, digit_base, tile_status,
                                      s_warp_hist, s_digit_excl, s_global_base, s_scan, s_kv);
    else
        onesweep_tile<false, IDENTITY>(keys_in, vals_in, keys_out, vals_out, tile, tile_count, shift, digit_base, tile_status,
                                       s_warp_hist, s_digit_excl, s_global_base, s_scan, s_kv);
}

// all passes of one sort: (keys[0], identity) -> (keys[cur], vals[cur]); returns cur.
// identity = false: the values start in vals[0].
inline int launch_onesweep(u32 *const keys[2], u32 *const vals[2], u32 n, int passes, const u32 *hist, u32 *tile_status,
                           u32 *tile_counter, cudaStream_t stream, bool identity = true) {
    const u32 tiles = (n + SORT_TILE - 1) / SORT_TILE;
    int cur = 0;
    for (int p = 0; p < passes; ++p) {
        if (p == 0 && identity)
            k_onesweep_pass<true><<<tiles, SORT_THREADS, 0, stream>>>(keys[0], nullptr, keys[1], vals[1], n, 0, hist, tile_status,
                                                                    tile_counter);
        else
            k_onesweep_pass<false><<<tiles, SORT_THREADS, 0, stream>>>(
                keys[cur], vals[cur], keys[cur ^ 1], vals[cur ^ 1], n, p * RADIX_BITS, hist + p * RADIX,
                tile_status + (size_t)p * tiles * RADIX, tile_counter + p);
        cur ^= 1;
    }
    return cur;
}

// -------------------------------------------------------------------------------------------------
// K4: gather the packed records into the three planes in cell order.
// Algorithmic bytes: 4 N (perm) + 52 N gathered (record with the caller id) + 56 N written = 112 N;
// a record is one aligned 64-byte block, so DRAM traffic is 124 N.
// -------------------------------------------------------------------------------------------------
constexpr int REORDER_THREADS = 256;
// four lanes per object: one 16-byte load each, so a warp request covers 8 whole records (16 full sectors) and every
// store instruction writes whole 128-byte runs of the planes
__global__ void __launch_bounds__(REORDER_THREADS)
k_reorder(const u32 *__restrict__ perm, u32 n, const float4 *__restrict__ U,
          float4 *__restrict__ P0, float4 *__restrict__ P1, float4 *__restrict__ P2, u32 *__restrict__ sorted_slot,
          u32 *__restrict__ sorted_id) {
    const u32 lane = threadIdx.x & 31u;
    const u32 base = (blockIdx.x * REORDER_THREADS + threadIdx.x) - lane;  // first position of the warp
    if (base >= n) return;
    const u32 s_own = base + lane;
    u32 src_own = s_own < n ? __ldcs(perm + s_own) : 0u;
#if RCD_SORT_ABLATE
    src_own = min(src_own, n - 1);
#endif
    if (s_own < n) sorted_slot[s_own] = src_own;
    const u32 q = lane & 3u;
    float4 *const plane = q == 0 ? P0 : q == 1 ? P1 : P2;
    float4 v[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const u32 o = r * 8 + (lane >> 2);
        const u32 src = __shfl_sync(FULL_MASK, src_own, o);
        v[r] = __ldg(U + 4 * (size_t)src + q);  // (positions past n read record 0: harmless, never stored)
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const u32 s = base + r * 8 + (lane >> 2);
        if (s < n) {
            if (q < 3) plane[s] = v[r];
            else sorted_id[s] = __float_as_uint(v[r].x);
        }
    }
}

// lower bound in the sorted key array
__device__ __forceinline__ u32 lower_bound_keys(const u32 *__restrict__ keys, u32 n, u32 key) {
    u32 lo = 0, hi = n;
    while (lo < hi) {
        u32 mid = (lo + hi) >> 1;
        if (keys[mid] < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// -------------------------------------------------------------------------------------------------
// K5: dense cell table.  cell_begin[c] = position in cell order of the first object whose cell is
// >= c, for every c in [0, ncells]; the objects of the cell run [c0, c1] of one grid row are then
// cell_begin[c0] .. cell_begin[c1 + 1] -- two loads, whatever the cell size.  One block owns
// CT_CELLS consecutive cells: two binary searches give its slice of the sorted keys, the first
// object of every occupied cell is marked in shared memory, a suffix-minimum fills the empty cells.
// Every entry is written every frame (no memset).  Bytes: 4 N read + 4 C written.
// -------------------------------------------------------------------------------------------------
constexpr int CT_THREADS = 256;
constexpr int CT_PER_THREAD = 4;
constexpr int CT_CELLS = CT_THREADS * CT_PER_THREAD;

__global__ void __launch_bounds__(CT_THREADS)
k_cell_table(const u32 *__restrict__ keys, u32 n, u32 ncells, u32 *__restrict__ cell_begin) {
    __shared__ u32 s_first[CT_CELLS];
    __shared__ u32 s_warp_min[CT_THREADS / 32];
    __shared__ u32 s_range[2];
    const u32 c0 = blockIdx.x * CT_CELLS;
    const u32 c1 = min(c0 + (u32)CT_CELLS, ncells);  // exclusive
    if (threadIdx.x < 2) s_range[threadIdx.x] = lower_bound_keys(keys, n, threadIdx.x == 0 ? c0 : c1);
#pragma unroll
    for (int k = 0; k < CT_PER_THREAD; ++k) s_first[threadIdx.x + k * CT_THREADS] = 0xffffffffu;
    __syncthreads();
    const u32 s0 = s_range[0], s1 = s_range[1];
    for (u32 s = s0 + threadIdx.x; s < s1; s += CT_THREADS) {
        const u32 key = keys[s];
#if RCD_SORT_ABLATE
        if (key - c0 >= (u32)CT_CELLS) continue;
#endif
        if (s == s0 || keys[s - 1] != key) s_first[key - c0] = s;
    }
    __syncthreads();
    // suffix minimum over the block's cells, seeded with s1 (= first object of any later cell)
    u32 v[CT_PER_THREAD];
    u32 run = 0xffffffffu;
#pragma unroll
    for (int k = CT_PER_THREAD - 1; k >= 0; --k) {
        run = min(run, s_first[threadIdx.x * CT_PER_THREAD + k]);
        v[k] = run;
    }
    u32 suf = run;  // inclusive suffix minimum over the threads of the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u32 t = __shfl_down_sync(FULL_MASK, suf, o);
        if (lane_id() + o < 32) suf = min(suf, t);
    }
    if (lane_id() == 0) s_warp_min[threadIdx.x >> 5] = suf;
    __syncthreads();
    u32 later = s1;  // minimum over everything after this thread
    for (u32 w = (threadIdx.x >> 5) + 1; w < CT_THREADS / 32; ++w) later = min(later, s_warp_min[w]);
    const u32 next = __shfl_down_sync(FULL_MASK, suf, 1);
    if (lane_id() < 31) later = min(later, next);
#pragma unroll
    for (int k = 0; k < CT_PER_THREAD; ++k) {
        const u32 c = c0 + threadIdx.x * CT_PER_THREAD + k;
        if (c < c1) cell_begin[c] = min(v[k], later);
    }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) cell_begin[ncells] = n;
}

// -------------------------------------------------------------------------------------------------
// K6: query order.  The pair kernel walks the cell rows under the bounding box of a tile's 32 query
// volumes, so a tile should hold queries whose volumes overlap: objects are keyed by the 2-D Morton
// code of the centre of their volume -- the object itself for radius queries, the middle of the chord
// of the predicted centre path (collision_detection.py:728-741) for predict queries -- and sorted;
// consecutive 32 objects are then a compact tile at any density.  Halo copies (not queried) get the
// top key and end up behind the last tile.  Owned objects without a position come just before them.  Bytes: 48 N read + 4 N written, then the sort passes.
// -------------------------------------------------------------------------------------------------
constexpr int QKEY_BITS = 23;                       // both axes together, split so that the key lattice is (nearly) square
constexpr u32 QKEY_NO_POSITION = 1u << QKEY_BITS;   // an owned object without a position (retired): behind every live query
constexpr u32 QKEY_NOT_QUERIED = QKEY_NO_POSITION + 1u;  // halo copies: behind everything
constexpr int QKEY_PASSES = 3;                      // 24 bits

__device__ __forceinline__ u32 spread_bits_2d(u32 v) {  // 16 bits -> every other bit
    v &= 0xffffu;
    v = (v | (v << 8)) & 0x00ff00ffu;
    v = (v | (v << 4)) & 0x0f0f0f0fu;
    v = (v | (v << 2)) & 0x33333333u;
    v = (v | (v << 1)) & 0x55555555u;
    return v;
}

struct QueryKeyParams {
    float ox, oy;          // origin of the key lattice
    float inv_res_x, inv_res_y;
    float max_x, max_y;    // 2^bits_x - 1, 2^bits_y - 1
    int bits_lo;           // min(bits_x, bits_y): that many bits of each axis are interleaved; the longer axis keeps
    int x_longer;          // its remaining high bits on top (a slab is 8 times as long as it is wide: 10 + 13 bits)
    int capsule;           // 1: predict queries are keyed by the middle of their chord
};

// Morton key of the query volume of the object at cell position s (p0 = P0[s], p2 = P2[s]; P1[s] is read only for
// capsules).  Shared by k_query_keys and k_query_keys_list, so a listed query lands in the same key as unlisted.
// An object without a position (a retired slot, rcd_retire) gets QKEY_NO_POSITION: such queries form the trailing
// tiles of the query order, which k_tile_plan leaves empty, and the live queries are tiled exactly as in a frame
// without them (the sort is stable and their cell positions come first).
__device__ __forceinline__ u32 query_key(const float4 &p0, const float4 &p2, const float4 *__restrict__ P1, u32 s,
                                         const QueryKeyParams &q) {
    if (p0.x != p0.x) return QKEY_NO_POSITION;
    float x = p0.x, y = p0.y;
    const u32 pattern = meta_pattern(__float_as_uint(p2.w));
    if (q.capsule && pattern != RCD_PAT_NO_HISTORY) {
        const float4 p1 = P1[s];
        const float fv = (pattern >= RCD_PAT_CONSTANT_VELOCITY) ? 4.75f : 0.0f;
        const float fa = (pattern == RCD_PAT_ACCELERATING) ? 22.5625f : 0.0f;
        const float mx = x + p1.x * fv + p2.x * fa, my = y + p1.y * fv + p2.y * fa;
        if (fabsf(mx) < 1.0e30f && fabsf(my) < 1.0e30f) { x = mx; y = my; }
    }
    const u32 ix = (u32)fminf(fmaxf((x - q.ox) * q.inv_res_x, 0.0f), q.max_x);  // NaN -> 0
    const u32 iy = (u32)fminf(fmaxf((y - q.oy) * q.inv_res_y, 0.0f), q.max_y);
    const u32 lo_mask = (1u << q.bits_lo) - 1u;
    return spread_bits_2d(ix & lo_mask) | (spread_bits_2d(iy & lo_mask) << 1) |
           (((q.x_longer ? ix : iy) >> q.bits_lo) << (2 * q.bits_lo));
}

__global__ void __launch_bounds__(KEYS_THREADS)
k_query_keys(const float4 *__restrict__ P0, const float4 *__restrict__ P1, const float4 *__restrict__ P2, u32 n,
             QueryKeyParams q, u32 *__restrict__ keys, u32 *__restrict__ hist) {
    __shared__ u32 s_hist[QKEY_PASSES][RADIX];
    for (int k = threadIdx.x; k < QKEY_PASSES * RADIX; k += KEYS_THREADS) (&s_hist[0][0])[k] = 0;
    __syncthreads();
    const u32 stride = gridDim.x * KEYS_THREADS;
    for (u32 s = blockIdx.x * KEYS_THREADS + threadIdx.x; s < n; s += stride) {
        const float4 p0 = P0[s];
        const float4 p2 = P2[s];
        const u32 meta = __float_as_uint(p2.w);
        u32 key = QKEY_NOT_QUERIED;
        if (meta & META_OWNED) key = query_key(p0, p2, P1, s, q);
        keys[s] = key;
#pragma unroll
        for (int p = 0; p < QKEY_PASSES; ++p) atomicAdd(&s_hist[p][(key >> (p * RADIX_BITS)) & (RADIX - 1)], 1u);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < QKEY_PASSES * RADIX; k += KEYS_THREADS) {
        u32 c = (&s_hist[0][0])[k];
        if (c) atomicAdd(&hist[k], c);
    }
}

// -------------------------------------------------------------------------------------------------
// K6 for a listed query set (rcd_set_queries): keys of the k listed objects only, with their cell positions as
// the values of the sort (every onesweep pass then reads them, none is the identity pass).  The list holds upload
// slots; slot_pos (k_slot_pos, once per index build) turns them into cell positions.  Bytes: 8 k + 48 k read
// (gathers) + 8 k written.
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(KEYS_THREADS)
k_query_keys_list(const float4 *__restrict__ P0, const float4 *__restrict__ P1, const float4 *__restrict__ P2,
                  const u32 *__restrict__ list, const u32 *__restrict__ slot_pos, u32 k, QueryKeyParams q,
                  u32 *__restrict__ keys, u32 *__restrict__ vals, u32 *__restrict__ hist) {
    __shared__ u32 s_hist[QKEY_PASSES][RADIX];
    for (int t = threadIdx.x; t < QKEY_PASSES * RADIX; t += KEYS_THREADS) (&s_hist[0][0])[t] = 0;
    __syncthreads();
    const u32 stride = gridDim.x * KEYS_THREADS;
    for (u32 t = blockIdx.x * KEYS_THREADS + threadIdx.x; t < k; t += stride) {
        const u32 s = slot_pos[list[t]];
        const u32 key = query_key(P0[s], P2[s], P1, s, q);
        keys[t] = key;
        vals[t] = s;
#pragma unroll
        for (int p = 0; p < QKEY_PASSES; ++p) atomicAdd(&s_hist[p][(key >> (p * RADIX_BITS)) & (RADIX - 1)], 1u);
    }
    __syncthreads();
    for (int t = threadIdx.x; t < QKEY_PASSES * RADIX; t += KEYS_THREADS) {
        u32 c = (&s_hist[0][0])[t];
        if (c) atomicAdd(&hist[t], c);
    }
}

// upload slot -> position in cell order: the inverse of sorted_slot (k_reorder)
__global__ void __launch_bounds__(256)
k_slot_pos(const u32 *__restrict__ sorted_slot, u32 n, u32 *__restrict__ slot_pos) {
    const u32 s = blockIdx.x * 256 + threadIdx.x;
    if (s < n) slot_pos[sorted_slot[s]] = s;
}

// Checks a query list in device memory: err |= 1 for a slot >= n_owned, |= 2 for a slot listed twice.
// seen: a zeroed bitmap of n_owned bits.
__global__ void __launch_bounds__(256)
k_check_queries(const u32 *__restrict__ list, u32 k, u32 n_owned, u32 *__restrict__ seen, u32 *__restrict__ err) {
    for (u32 t = blockIdx.x * 256 + threadIdx.x; t < k; t += gridDim.x * 256) {
        const u32 s = list[t];
        if (s >= n_owned) {
            atomicOr(err, 1u);
            continue;
        }
        const u32 bit = 1u << (s & 31u);
        if (atomicOr(&seen[s >> 5], bit) & bit) atomicOr(err, 2u);
    }
}

// bounding box of the positions (auto grid): ordered-int atomics
__device__ __forceinline__ int float_ordered(float f) {
    int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__host__ __device__ __forceinline__ float ordered_float(int i) {
    int j = i >= 0 ? i : i ^ 0x7fffffff;
#ifdef __CUDA_ARCH__
    return __int_as_float(j);
#else
    float f;
    memcpy(&f, &j, 4);
    return f;
#endif
}

__global__ void __launch_bounds__(256)
k_bbox(const float *__restrict__ px, const float *__restrict__ py, const float *__restrict__ pz, u32 n,
       int *__restrict__ bbox /* min x,y,z, max x,y,z (ordered ints) */) {
    float lo[3] = {3.0e38f, 3.0e38f, 3.0e38f}, hi[3] = {-3.0e38f, -3.0e38f, -3.0e38f};
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float p[3] = {px[i], py[i], pz[i]};
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            if (p[d] == p[d] && fabsf(p[d]) < 1.0e30f) {  // ignore non-finite coordinates
                lo[d] = fminf(lo[d], p[d]);
                hi[d] = fmaxf(hi[d], p[d]);
            }
        }
    }
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        for (int o = 16; o > 0; o >>= 1) {
            lo[d] = fminf(lo[d], __shfl_xor_sync(FULL_MASK, lo[d], o));
            hi[d] = fmaxf(hi[d], __shfl_xor_sync(FULL_MASK, hi[d], o));
        }
        if (lane_id() == 0) {
            atomicMin(&bbox[d], float_ordered(lo[d]));
            atomicMax(&bbox[3 + d], float_ordered(hi[d]));
        }
    }
}

}  // namespace rcd
