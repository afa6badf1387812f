// Pair enumeration + narrow phase + classification.
//
// Three kernels per frame, connected by compact queues in global memory, so that every stage runs
// with full warps and each kernel's hot loop stays small:
//
//   k_tile_plan: one warp per tile of 32 queries in *query order* (Morton order of the centres of the query
//              volumes, rcd_index.cuh).  Every query has a volume a neighbour must lie in to matter -- a ball
//              of radius R, or (predict) the capsule of radius 100 m about the chord of the predicted centre
//              path.  The plan stores the cell box of the tile's volumes, an x range for every cell row of the
//              box (what some volume reaches inside the row's y band: the corners of the box are empty), and
//              cuts the tile into work items of about equal numbers of 32-neighbour chunks.
//   k_pairs  : persistent, the S1 filter only.  A warp takes work items from an atomic counter; lane = query.
//              It streams the cell rows of its tile through its own slice of shared memory
//              (cp.async one chunk of 32 neighbours ahead, re-laid two neighbours side by side).  For
//              every (query, neighbour) the lane takes, in packed fp32 (FADD2 / FFMA2, two neighbours
//              per instruction):
//                * the radius test |p_j - p_i| <= R where the mode has one (candidate counts; pairs inside
//                  the fp32 guard band of the radius are flagged for the exact stage), and
//                * T1: can the relative trajectory come close at all?  The trajectory of the pair is
//                  expanded about the middle tm of the time window, g(tm + u) = g0 + g1 u + ca u^2 / 2 with
//                  g0 = centre_i(tm) - pos_j(tm) and g1 the relative velocity at tm -- differences of
//                  per-object quantities, so the neighbour's half is computed once when it is staged --
//                  and the linear part must come within  L = A_i + B_j + kq |ca|  for some u in [-D, D + 0.9]:
//                  A_i, B_j bound the safe distance and the rounding, kq |ca| the curvature |ca| D^2 / 2 and the
//                  part of the 10 samples' motion that is not along g1 (the samples of an offset move with the
//                  pair's CURRENT relative velocity rv = g1 + delta for tau <= 0.9 s: the part along g1 only
//                  stretches the window by 0.9 s, |delta| <= |v_i - uv_i| + tm |ca| goes into the bound).
//              The outcome of a test is the sign bit of a packed subtraction, shifted into per-lane bit masks
//              (one funnel shift per test; no compare, no store); the pass rule is applied once per chunk.
//              Survivors (about 1 in 29) are appended to the pair queue QA, which warps fill in private
//              256-entry blocks (one global atomic per block, not per push).
//   k_narrow : QA -> Q3.  A warp takes 32 queued pairs (lane = pair): detect narrow phase (temporal
//              filter + closest approach) and, for predict queries, the offsets whose 10 samples can reach
//              the safe distance at all (all 20 offsets in packed fp32) -> offset mask; then the per-offset
//              work in three more phases with different lane assignments ((pair, offset) / surviving item /
//              pair): radius test, the 10 samples, the max-risk merge.
//   k_exact  : lane = pair; the decision is taken in fp64 in the reference's operation order
//              (rcd_exact.cuh), merged over offsets, emitted through one 64-bit atomic cursor and
//              classified (alert priority).
// The fp32 stages only ever *reject*, with guard bands that dominate the rounding error.
//
// Replaces the reference's per-vehicle Python loops:
//   detect : CollisionDetector.detect_collisions      src/collision/collision_detection.py:110-191
//   predict: CollisionPredictionModel.predict_collisions                                  :572-865
//   compute-node: SpatialIndex.query_nearby + CollisionDetector.detect_collisions
//                                                       src/compute/compute_node.py:98-119, 229-321
//   alert class: AlertManager.process_collision_risks/_get_priority
//                                                       src/collision/warning_system.py:259-311
#pragma once
#include "rcd_common.cuh"
#include "rcd_index.cuh"
#include "rcd_exact.cuh"

namespace rcd {

constexpr int TQ = 32;            // queries per tile = one warp
constexpr int PAIR_WARPS = 4;     // warps (independent tiles) per block
constexpr int PAIR_THREADS = PAIR_WARPS * 32;
constexpr int CH = 32;            // neighbours staged per chunk (1 per lane)
constexpr int QA_BLOCK = 256;     // entries of the pair queue a warp reserves at a time
constexpr u32 QA_INR = 1u << 30;  // entry flag: certainly within the radius (and counted as a candidate)
constexpr u32 QA_UND = 1u << 31;  // entry flag: inside the fp32 guard band of the radius: k_exact decides and counts
constexpr u32 QA_SI_MASK = (1u << 30) - 1u;
constexpr u32 QA_NO_BLOCK = 0xffffffffu;

// one queued pair between k_narrow and k_exact: positions in cell order + offset mask (predict)
struct QEntry {
    u32 si, sj, mask;
};

struct PairParams {
    u32 n;                   // objects (owned + halo)
    u32 n_owned;             // queries
    u32 ntiles;
    u32 item_chunks;         // smallest work item of k_pairs, in chunks (k_tile_plan)
    uint4 *items;            // work items of k_pairs
    u32 items_cap;
    int4 *tile_box;          // [2 * ntiles] cell box of every tile: {x0, x1, y0, y1}, {z0, z1, -, -}
    uint2 *tile_rowx;        // [TILE_ROWS * ntiles] x cell range of the first TILE_ROWS cell rows of every tile's box
    GridParams g;
    const float4 *P0, *P1, *P2;
    const u32 *qorder;       // query order -> position in cell order
    const u32 *sorted_slot;  // cell order -> upload slot
    const u32 *sorted_id;    // cell order -> caller id
    const u32 *cell_begin;   // [ncells + 1]
    float R, T;              // search radius / time window (detect)
    int steps;               // int(T / 0.1)
    float pt, threshold;     // compute-node: prediction_time, risk_threshold
    // T1: middle and half width of the time window, on/off
    float tm, D;
    int use_t1;
    rcd_pair *out;
    unsigned long long out_cap;
    Counters *counters;
    u32 *tile_counter;
    u32 *cand_count;         // per upload slot
    u32 *risk_count;         // per upload slot: risks emitted for the object as the querying vehicle
    uint2 *qa;               // pair queue k_pairs -> k_narrow: {si | flags, sj}
    u32 *qa_fill;            // entries used in every QA block
    u32 qa_blocks_cap;
    uint4 *ovf;              // work of k_pairs left to its overflow pass: {work item, row batch, chunk, -}
    u32 ovf_cap;
    QEntry *q3;              // k_narrow -> k_exact
    u32 qcap;
    u32 q3_split;            // detect entries: [0, q3_split); predict entries: [q3_split, qcap)
};

// relative guard band of the fp32 radius test (fp32 error of d2 is < 1e-6 relative)
constexpr float BAND_R2 = 2.0e-5f;

// shared-memory state of one warp of k_pairs
struct StagePacked {      // a chunk of 32 neighbours, two side by side per entry (operands of the packed filter)
    float4 xy[CH / 2];    // {x0, x1, y0, y1}                      current position
    float4 zb[CH / 2];    // {z0, z1, B0, B1}                      ... and the neighbour's half of the T1 bound
    float4 nxy[CH / 2];   // {-Nx0, -Nx1, -Ny0, -Ny1}              N = position at tm, negated
    float4 nzv[CH / 2];   // {-Nz0, -Nz1, -NVx0, -NVx1}            NV = velocity at tm, negated
    float4 nvyz[CH / 2];  // {-NVy0, -NVy1, -NVz0, -NVz1}
    float4 naxy[CH / 2];  // {-ax0, -ax1, -ay0, -ay1}              acceleration, negated
    float2 naz[CH / 2];   // {-az0, -az1}
    u32 pos[CH];          // position in cell order of the staged object
};
struct WarpShared {
    float4 r0[CH], r1[CH], r2[CH];  // landing zone of the cp.async copies (the chunk after the one being filtered)
    StagePacked buf[2];
    u32 row_lo[TQ];
    u32 row_prefix[TQ + 1];
};

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
    unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

// packed fp32 pairs (Blackwell FADD2 / FMUL2 / FFMA2: two lanes of fp32 per instruction; a float2 built
// from one scalar becomes the broadcast operand form)
__device__ __forceinline__ unsigned long long f2_bits(float2 v) { return *reinterpret_cast<unsigned long long *>(&v); }
__device__ __forceinline__ float2 bits_f2(unsigned long long v) { return *reinterpret_cast<float2 *>(&v); }
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
    unsigned long long d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(f2_bits(a)), "l"(f2_bits(b)));
    return bits_f2(d);
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b) {
    unsigned long long d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(f2_bits(a)), "l"(f2_bits(b)));
    return bits_f2(d);
}
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(f2_bits(a)), "l"(f2_bits(b)), "l"(f2_bits(c)));
    return bits_f2(d);
}
__device__ __forceinline__ float2 splat2(float v) { return make_float2(v, v); }
// mask = mask << 1 | sign bit of t: one funnel shift per test instead of compare + select + or (the difference itself
// comes out of a packed add on the FMA pipe; NaN results are canonical, sign clear)
__device__ __forceinline__ u32 shift_in_sign(u32 mask, float t) {
    u32 r;
    asm("shf.l.wrap.b32 %0, %1, %2, 1;" : "=r"(r) : "r"(__float_as_uint(t)), "r"(mask));
    return r;
}
// keeps a loop-invariant value in its register (the compiler would otherwise re-derive it inside the hot loop)
__device__ __forceinline__ float pin_reg(float v) {
    asm volatile("" : "+f"(v));
    return v;
}

// sqrt(x) rounded up a little: only ever used for conservative bounds (MUFU.SQRT, ~1 ulp)
__device__ __forceinline__ float sqrt_ub(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r * (1.0f + 4.0e-6f);
}
// 1/x to ~1 ulp (MUFU.RCP); callers cover the error with their slack terms
__device__ __forceinline__ float rcp_fast(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// result of the exact stage for one queued pair
struct EmitRec {
    u32 si, sj;
    float ttc, dist, rs, risk, cx, cy, cz, tcl, dcl;
    int prio, offset;
    bool hit, predicted, high;  // high: risk > 0.7 decided in fp64 (stats["high_risk_collisions"])
    bool twice;                 // emit (and count) the record twice (ENTRY_TWICE)
    u32 potential;              // detect: the pair passed stage 2 (stats["potential_collisions"])
};

__device__ __forceinline__ EmitRec make_rec(u32 si, u32 sj, double ttc, double dist, double rs, double risk,
                                            double mx, double my, double mz, double tcl, double dcl, int prio,
                                            int offset, bool predicted) {
    EmitRec r;
    r.si = si; r.sj = sj;
    r.ttc = (float)ttc; r.dist = (float)dist; r.rs = (float)rs; r.risk = (float)risk;
    r.cx = (float)mx; r.cy = (float)my; r.cz = (float)mz;
    r.tcl = (float)tcl; r.dcl = (float)dcl;
    r.prio = prio; r.offset = offset;
    r.hit = true; r.predicted = predicted; r.high = risk > 0.7;
    r.twice = false;
    r.potential = 0;
    return r;
}
__device__ __forceinline__ EmitRec no_rec() {
    EmitRec r;
    r.si = r.sj = 0;
    r.ttc = r.dist = r.rs = r.risk = r.cx = r.cy = r.cz = r.tcl = r.dcl = 0.0f;
    r.prio = -1; r.offset = 255;
    r.hit = false; r.predicted = false; r.high = false;
    r.twice = false;
    r.potential = 0;
    return r;
}

// store one pair at `pos` (three 16-byte stores; rcd_pair is 48 bytes)
__device__ __forceinline__ void store_pair(const PairParams &P, unsigned long long pos, const EmitRec &e) {
    atomicAdd(&P.risk_count[P.sorted_slot[e.si]], 1u);
    if (pos >= P.out_cap) return;
    rcd_pair r;
    r.i = P.sorted_id[e.si];
    r.j = P.sorted_id[e.sj];
    r.ttc = e.ttc; r.distance = e.dist; r.rel_speed = e.rs; r.risk = e.risk;
    r.cx = e.cx; r.cy = e.cy; r.cz = e.cz;
    r.t_closest = e.tcl; r.d_closest = e.dcl;
    r.priority = (int8_t)e.prio;
    r.offset = (uint8_t)e.offset;
    r.predicted = e.predicted ? 1 : 0;
    r.reserved = 0;
    uint4 *dst = reinterpret_cast<uint4 *>(P.out + pos);
    const uint4 *src = reinterpret_cast<const uint4 *>(&r);
    dst[0] = src[0]; dst[1] = src[1]; dst[2] = src[2];
}

// per-thread emission (queue-overflow fallbacks only; the exact stage aggregates per warp)
__device__ __noinline__ void thread_emit(const PairParams &P, const EmitRec &e) {
    if (!e.hit) return;
    const unsigned long long copies = e.twice ? 2ULL : 1ULL;
    unsigned long long pos = atomicAdd(&P.counters->n_pairs, copies);
    if (e.high) atomicAdd(&P.counters->n_high_risk, copies);
    if (e.prio >= 0) atomicAdd(&P.counters->n_alerts[e.prio], copies);
    store_pair(P, pos, e);
    if (e.twice) store_pair(P, pos + 1, e);
}

// ---- fp64 decisions (rare) ---------------------------------------------------------------------------
__device__ __noinline__ bool exact_within_radius(float ax, float ay, float az, float bx, float by, float bz, float R) {
    return within_radius_d(ax, ay, az, bx, by, bz, (double)R);
}

// detect: stages 2-4 in fp64 for the pair (si, sj)
__device__ __noinline__ EmitRec exact_detect(const PairParams &P, u32 si, u32 sj, float T, int steps) {
    ObjD A = widen(P.P0[si], P.P1[si], P.P2[si]), B = widen(P.P0[sj], P.P1[sj], P.P2[sj]);
    DetectResultD r = detect_pair_d(A, B, (double)T, steps);
    EmitRec e = r.hit ? make_rec(si, sj, r.ttc, r.dist, r.rs, r.risk, r.mx, r.my, r.mz, r.tc, r.cd, r.priority, 255, false)
                      : no_rec();
    e.potential = r.potential ? 1u : 0u;
    return e;
}

__device__ __noinline__ bool exact_predict_radius(const PairParams &P, u32 si, u32 sj, u32 pattern, int m) {
    ObjD A = widen(P.P0[si], P.P1[si], P.P2[si]);
    const float4 b0 = P.P0[sj];
    double cx, cy, cz;
    predict_centre_d(A, pattern, 0.5 * (double)m, cx, cy, cz);
    return within_radius_d(cx, cy, cz, b0.x, b0.y, b0.z, (double)PREDICT_RADIUS);
}

// predict: every offset in `mask` in fp64, max-risk merge (strict >, offsets ascending, :848-865)
__device__ __noinline__ EmitRec exact_predict(const PairParams &P, u32 si, u32 sj, u32 pattern, u32 mask) {
    ObjD A = widen(P.P0[si], P.P1[si], P.P2[si]), B = widen(P.P0[sj], P.P1[sj], P.P2[sj]);
    double best_risk = -1.0;
    PredictResultD best;
    int best_m = -1;
    while (mask) {
        int m = __ffs(mask) - 1;
        mask &= mask - 1;
        PredictResultD r = predict_pair_d(A, B, pattern, m);
        if (r.hit && r.risk > best_risk) { best_risk = r.risk; best = r; best_m = m; }
    }
    if (best_m < 0) return no_rec();
    return make_rec(si, sj, best.ttc, best.dist, best.rs, best.risk, best.mx, best.my, best.mz, 0.5 * (double)best_m,
                    0.0, priority_d(best.risk, best.ttc), best_m, true);
}

// Queue entries whose winning offset m and first hit sample k were already settled in fp32 with
// every margin wide open carry RESOLVED | m | k << 8: one fp64 evaluation yields the emitted values.
constexpr u32 RESOLVED = 1u << 31;
// Queue entries of radius queries whose fp32 distance lies inside the guard band of the radius carry
// RADIUS_UNDECIDED: the exact stage takes the radius test (spatial_index.py:268) before anything else
// and counts the candidate.  k_pairs itself never evaluates fp64.
constexpr u32 RADIUS_UNDECIDED = 1u << 30;
// Internal frame mode of rcd_step(RCD_MODE_PREDICT | RCD_STEP_WITH_DETECT): the predict pass also runs
// detect_collisions(100.0, 10.0) for every object on the pairs it streams anyway (the ball of radius 100
// about an object lies inside its predict capsule).  Objects without history (pattern 3) then owe the same
// risk twice -- once as detect_collisions, once as the fall-back of predict_collisions (:590-592) -- which
// their queue entries carry as ENTRY_TWICE.
constexpr int MODE_PREDICT_WITH_DETECT = 3;
constexpr u32 ENTRY_TWICE = 1u << 29;
__host__ __device__ constexpr bool is_predict(int mode) { return mode == RCD_MODE_PREDICT || mode == MODE_PREDICT_WITH_DETECT; }

// predict, full fallback: every offset, radius test included (collision_detection.py:789-865)
__device__ __noinline__ EmitRec exact_predict_all(const PairParams &P, u32 si, u32 sj, u32 pattern) {
    u32 mask = 0;
    for (int m = 0; m < PREDICT_OFFSETS; ++m)
        if (exact_predict_radius(P, si, sj, pattern, m)) mask |= 1u << m;
    return mask ? exact_predict(P, si, sj, pattern, mask) : no_rec();
}

__device__ __forceinline__ EmitRec exact_predict_resolved_body(const PairParams &P, u32 si, u32 sj, u32 pattern, int m, int k) {
    ObjD A = widen(P.P0[si], P.P1[si], P.P2[si]), B = widen(P.P0[sj], P.P1[sj], P.P2[sj]);
    const double t = dmul(0.5, (double)m);
    double cx, cy, cz;
    predict_centre_d(A, pattern, t, cx, cy, cz);
    const double qx = pos1_d(B.px, B.vx, B.ax, t), qy = pos1_d(B.py, B.vy, B.ay, t), qz = pos1_d(B.pz, B.vz, B.az, t);
    const double safe = safe_d(A.size, B.size);
    const double tau = dmul((double)k, 0.1);
    const double xi = pos1_d(cx, A.vx, A.ax, tau), yi = pos1_d(cy, A.vy, A.ay, tau), zi = pos1_d(cz, A.vz, A.az, tau);
    const double xj = pos1_d(qx, B.vx, B.ax, tau), yj = pos1_d(qy, B.vy, B.ay, tau), zj = pos1_d(qz, B.vz, B.az, tau);
    const double d = dist3_d(xi, yi, zi, xj, yj, zj);
    if (!(d <= safe)) {  // cannot happen while the guard bands hold; stay exact if it ever does
        atomicAdd(&P.counters->n_fallback, 1ULL);
        return exact_predict_all(P, si, sj, pattern);
    }
    const double rs = mag3_d(dsub(A.vx, B.vx), dsub(A.vy, B.vy), dsub(A.vz, B.vz));
    const double risk = risk_level_d(A.heading, B.heading, A.type, B.type, tau, d, safe, rs);
    const double ttc = dadd(tau, t);
    return make_rec(si, sj, ttc, d, rs, risk, half_d(dadd(xi, xj)), half_d(dadd(yi, yj)),
                    half_d(dadd(zi, zj)), t, 0.0, priority_d(risk, ttc), m, true);
}

__device__ __noinline__ EmitRec exact_predict_resolved(const PairParams &P, u32 si, u32 sj, u32 pattern, int m, int k) {
    return exact_predict_resolved_body(P, si, sj, pattern, m, k);
}

__device__ __noinline__ EmitRec exact_compute_node(const PairParams &P, u32 si, u32 sj) {
    // predict_position needs >= 2 samples of both vehicles (compute_node.py:202-203, 269-270): pairs that came here
    // for the radius decision have not passed the fp32 narrow phase, which checks this
    if (meta_pattern(__float_as_uint(P.P2[si].w)) == 0u || meta_pattern(__float_as_uint(P.P2[sj].w)) == 0u) return no_rec();
    ObjD A = widen(P.P0[si], P.P1[si], P.P2[si]), B = widen(P.P0[sj], P.P1[sj], P.P2[sj]);
    ComputeNodeResultD r = compute_node_pair_d(A, B, (double)P.pt, (double)P.threshold);
    if (!r.hit) return no_rec();
    return make_rec(si, sj, r.ttc, r.fut, r.rs, r.risk, r.mx, r.my, r.mz, 0.0, 0.0, -1, 255, false);
}

// the exact stage for one queue entry
template <int MODE>
__device__ __forceinline__ EmitRec exact_entry(const PairParams &P, u32 si, u32 sj, u32 mask) {
    const bool twice = (mask & ENTRY_TWICE) != 0;
    mask &= ~ENTRY_TWICE;
    if (mask & RADIUS_UNDECIDED) {
        const float4 a0 = P.P0[si], b0 = P.P0[sj];
        const float R = is_predict(MODE) ? PREDICT_RADIUS : P.R;
        if (!exact_within_radius(a0.x, a0.y, a0.z, b0.x, b0.y, b0.z, R)) return no_rec();
        atomicAdd(&P.counters->n_candidates, twice ? 2ULL : 1ULL);
        if (P.cand_count) atomicAdd(&P.cand_count[P.sorted_slot[si]], twice ? 2u : 1u);
        if (MODE == RCD_MODE_COMPUTE_NODE && si == sj) return no_rec();  // the index returns self (quirk Q8)
        mask = 0;
    }
    EmitRec e;
    if (MODE == RCD_MODE_DETECT) e = exact_detect(P, si, sj, P.T, P.steps);
    else if (MODE == RCD_MODE_COMPUTE_NODE) e = exact_compute_node(P, si, sj);
    else if (mask == 0) e = exact_detect(P, si, sj, 10.0f, 100);  // pattern 3 / fused detect: the defaults (:592)
    else {
        const u32 pattern = meta_pattern(__float_as_uint(P.P2[si].w));
        e = (mask & RESOLVED) ? exact_predict_resolved(P, si, sj, pattern, (int)(mask & 31u), (int)((mask >> 8) & 15u))
                              : exact_predict(P, si, sj, pattern, mask);
    }
    if (twice) { e.twice = true; e.potential *= 2u; }
    return e;
}

// queue-full fallback: decide and emit the pair in place (correct, slower, out of line)
template <int MODE>
__device__ __noinline__ u32 finish_entry_inline(const PairParams &P, u32 si, u32 sj, u32 mask) {
    const EmitRec e = exact_entry<MODE>(P, si, sj, mask);
    thread_emit(P, e);
    return e.potential;
}

// ---- narrow phase, detect: temporal filter + closest approach in fp32 (collision_detection.py:244-292) ------
// returns true when the pair must be decided in fp64.  The radius test was taken by the S1 filter (QA_INR /
// QA_UND): pairs inside the guard band of the radius go to the exact stage without passing through here.
__device__ __forceinline__ bool narrow_detect(const float4 &a0, const float4 &a1, const float4 &a2, const float4 &b0,
                                              const float4 &b1, const float4 &b2, float T) {
    float dx = b0.x - a0.x, dy = b0.y - a0.y, dz = b0.z - a0.z;  // rel_position = other - self
    float d2 = dx * dx + dy * dy + dz * dz;
    float rvx = a1.x - b1.x, rvy = a1.y - b1.y, rvz = a1.z - b1.z;  // rel_velocity = self - other
    float rs2 = rvx * rvx + rvy * rvy + rvz * rvz;
    if (rs2 < 0.0099f) return false;  // rel_speed < 0.1 with margin (0.1^2 = 0.01)
    float dot = dx * rvx + dy * rvy + dz * rvz;
    float edot = 4.0e-6f * sqrt_ub(d2 * rs2) + 1.0e-20f;  // (bounds only need upper estimates: MUFU sqrt / rcp)
    // dot > 0: either (dot > 0 and cur > 5) or time_to_closest < 0 rejects the pair (:273, :280)
    if (dot > edot) return false;
    if (-dot > T * rs2 * (1.0f + 1.0e-5f) + edot) return false;  // time_to_closest > time_window
    const float inv_rs2 = rcp_fast(rs2);
    float tc = fmaxf(-dot, 0.0f) * inv_rs2;
    float rax = a2.x - b2.x, ray = a2.y - b2.y, raz = a2.z - b2.z;
    float h = 0.5f * tc * tc;
    float ex = rvx * tc + rax * h - dx, ey = rvy * tc + ray * h - dy, ez = rvz * tc + raz * h - dz;
    float cd2 = ex * ex + ey * ey + ez * ez;
    float safe = (a0.w + b0.w) * 0.5f + 5.0f;
    float tcerr = edot * inv_rs2 * (1.0f + 1.0e-6f) + 4.0e-6f * tc;  // 4e-6 tc also covers the rcp (1 ulp)
    float band = 2.0e-3f + 2.0f * (sqrt_ub(rs2) + sqrt_ub(rax * rax + ray * ray + raz * raz) * tc) * tcerr;
    float thr = safe + band;
    return cd2 <= thr * thr;
}

// coefficients of one predict pair: g(t) = centre_i(t) - predicted_j(t) = -d + cv t + ca t^2/2 (:814),
// e(t) = centre_i(t) - p_j = -d + uv t + ua t^2/2 (:801-803); the samples move with rv, ra (:326-327)
struct PredictCoef {
    float dx, dy, dz;
    float uvx, uvy, uvz, uax, uay, uaz;
    float cvx, cvy, cvz, cax, cay, caz;
    float rvx, rvy, rvz, inv_rv2, lim2;  // sample motion: relative velocity, 1/|rv|^2, (safe_b + 0.405 |ra|)^2
    float safe_b2, hr, hr2;
    float safe, safe_b;                  // safe distance, and with its guard band
};
__device__ __forceinline__ PredictCoef predict_coef(const float4 &a0, const float4 &a1, const float4 &a2,
                                                    const float4 &b0, const float4 &b1, const float4 &b2,
                                                    u32 pattern) {
    PredictCoef c;
    const float fv = (pattern >= RCD_PAT_CONSTANT_VELOCITY) ? 1.0f : 0.0f;
    const float fa = (pattern == RCD_PAT_ACCELERATING) ? 1.0f : 0.0f;
    c.uvx = a1.x * fv; c.uvy = a1.y * fv; c.uvz = a1.z * fv;
    c.uax = a2.x * fa; c.uay = a2.y * fa; c.uaz = a2.z * fa;
    c.dx = b0.x - a0.x; c.dy = b0.y - a0.y; c.dz = b0.z - a0.z;
    c.cvx = c.uvx - b1.x; c.cvy = c.uvy - b1.y; c.cvz = c.uvz - b1.z;
    c.cax = c.uax - b2.x; c.cay = c.uay - b2.y; c.caz = c.uaz - b2.z;
    float rvx = a1.x - b1.x, rvy = a1.y - b1.y, rvz = a1.z - b1.z;
    float rax = a2.x - b2.x, ray = a2.y - b2.y, raz = a2.z - b2.z;
    float rvn = sqrt_ub(rvx * rvx + rvy * rvy + rvz * rvz);
    float ran = sqrt_ub(rax * rax + ray * ray + raz * raz);
    float d2 = c.dx * c.dx + c.dy * c.dy + c.dz * c.dz;
    float safe = (a0.w + b0.w) * 0.5f + 5.0f;
    float safe_b = safe + 2.0e-3f + 1.0e-6f * sqrt_ub(d2);
    c.safe = safe;
    c.safe_b = safe_b;
    c.safe_b2 = safe_b * safe_b;
    // the 10 samples move the pair by at most |rv|*0.9 + |ra|*0.405 from the offset state
    c.hr = safe_b + rvn * 0.9f + ran * 0.405f;
    c.hr2 = c.hr * c.hr;
    c.rvx = rvx; c.rvy = rvy; c.rvz = rvz;
    const float rv2 = rvx * rvx + rvy * rvy + rvz * rvz;
    c.inv_rv2 = rv2 > 1.0e-12f ? rcp_fast(rv2) : 0.0f;
    const float lim = (safe_b + ran * 0.405f) * (1.0f + 1.0e-5f) + 1.0e-3f;
    c.lim2 = lim * lim;
    return c;
}
// Can one of the 10 samples after offset time t come within the safe distance?  The samples move
// along g + rv tau + ra tau^2/2, tau in [0, 0.9]: |.| >= min_tau |g + rv tau| - 0.405 |ra|.
__device__ __forceinline__ bool offset_may_hit(const PredictCoef &c, float t) {
    const float h = 0.5f * t * t;
    const float gx = c.cvx * t + c.cax * h - c.dx, gy = c.cvy * t + c.cay * h - c.dy, gz = c.cvz * t + c.caz * h - c.dz;
    if (gx * gx + gy * gy + gz * gz > c.hr2) return false;
    const float tau = fminf(fmaxf(-(gx * c.rvx + gy * c.rvy + gz * c.rvz) * c.inv_rv2, 0.0f), 0.9f);
    const float ex = gx + c.rvx * tau, ey = gy + c.rvy * tau, ez = gz + c.rvz * tau;
    return ex * ex + ey * ey + ez * ez <= c.lim2;
}
__device__ __forceinline__ float g2_at(const PredictCoef &c, float t) {
    float h = 0.5f * t * t;
    float gx = c.cvx * t + c.cax * h - c.dx, gy = c.cvy * t + c.cay * h - c.dy, gz = c.cvz * t + c.caz * h - c.dz;
    return gx * gx + gy * gy + gz * gz;
}

// ---- S2a / S2b, predict: when can the relative trajectory come close at all? ---------------------------
// g(t) = -d + cv t + ca t^2/2 is the offset state of the pair (centre_i(t) - predicted_j(t)); an offset
// at time t can only be hit if |g(t)| <= hr (the 10 samples move the pair by at most hr - safe).
struct WindowCoef {
    float dx, dy, dz, cvx, cvy, cvz, cax, cay, caz;
    float hr;   // safe + band + 0.9 |rv| + 0.405 |ra|, rounded up
    float can;  // |ca|, rounded up
    float d2, eps;
};
__device__ __forceinline__ WindowCoef window_coef(const float4 &a0, const float4 &a1, const float4 &a2,
                                                  const float4 &b0, const float4 &b1, const float4 &b2, u32 pattern) {
    WindowCoef c;
    const float fv = (pattern >= RCD_PAT_CONSTANT_VELOCITY) ? 1.0f : 0.0f;
    const float fa = (pattern == RCD_PAT_ACCELERATING) ? 1.0f : 0.0f;
    c.dx = b0.x - a0.x; c.dy = b0.y - a0.y; c.dz = b0.z - a0.z;
    c.cvx = a1.x * fv - b1.x; c.cvy = a1.y * fv - b1.y; c.cvz = a1.z * fv - b1.z;
    c.cax = a2.x * fa - b2.x; c.cay = a2.y * fa - b2.y; c.caz = a2.z * fa - b2.z;
    const float rvx = a1.x - b1.x, rvy = a1.y - b1.y, rvz = a1.z - b1.z;
    const float rax = a2.x - b2.x, ray = a2.y - b2.y, raz = a2.z - b2.z;
    const float rvn = sqrt_ub(rvx * rvx + rvy * rvy + rvz * rvz);
    const float ran = sqrt_ub(rax * rax + ray * ray + raz * raz);
    c.can = sqrt_ub(c.cax * c.cax + c.cay * c.cay + c.caz * c.caz);
    c.d2 = c.dx * c.dx + c.dy * c.dy + c.dz * c.dz;
    const float dn = sqrt_ub(c.d2);
    const float safe = (a0.w + b0.w) * 0.5f + 5.0f;
    c.hr = safe + 2.0e-3f + 1.0e-6f * dn + rvn * 0.9f + ran * 0.405f;  // = PredictCoef::hr
    c.eps = 1.0e-2f + 1.0e-5f * dn;
    return c;
}
// S2a: |g(t)| >= |-d + cv t| - |ca| t^2/2 on [0, 9.5]; the linear part is minimal at ts = d.cv / |cv|^2.
// False when no offset can be hit.  (Cheap: this runs on every pair the S1 filter lets through.)
__device__ __forceinline__ bool window_reject_linear(const WindowCoef &c) {
    const float L = (c.hr + 45.125f * c.can) * (1.0f + 1.0e-4f) + c.eps;
    const float cv2 = c.cvx * c.cvx + c.cvy * c.cvy + c.cvz * c.cvz;
    if (!(cv2 > 1.0e-8f)) return c.d2 <= L * L;  // (almost) no relative drift: every offset looks the same
    const float ts = (c.dx * c.cvx + c.dy * c.cvy + c.dz * c.cvz) * rcp_fast(cv2);
    const float tc = fminf(fmaxf(ts, 0.0f), 9.5f);
    const float lx = c.cvx * tc - c.dx, ly = c.cvy * tc - c.dy, lz = c.cvz * tc - c.dz;
    return lx * lx + ly * ly + lz * lz <= L * L;
}
// S2b: the time window [t_lo, t_hi] that can hold a hit, as offsets [m_lo, m_hi].  First the window of
// the linear part with the whole acceleration term as slack; then, twice, the trajectory is expanded
// about the middle tm of the current window, g(tm + u) = g0 + g1 u + ca u^2/2 (exact for a quadratic),
// so only |ca| D^2/2 (D = half width) is left as slack and the window tightens quadratically.
__device__ __forceinline__ bool predict_window(const WindowCoef &c, int &m_lo, int &m_hi) {
    const float L = (c.hr + 45.125f * c.can) * (1.0f + 1.0e-4f) + c.eps;
    const float L2 = L * L;
    const float cv2 = c.cvx * c.cvx + c.cvy * c.cvy + c.cvz * c.cvz;
    m_lo = 0;
    m_hi = PREDICT_OFFSETS - 1;
    float t_lo = 0.0f, t_hi = 9.5f;
    if (cv2 > 1.0e-8f) {
        const float inv = rcp_fast(cv2);
        const float dcv = c.dx * c.cvx + c.dy * c.cvy + c.dz * c.cvz;
        const float ts = dcv * inv;
        const float tc = fminf(fmaxf(ts, 0.0f), 9.5f);
        const float lx = c.cvx * tc - c.dx, ly = c.cvy * tc - c.dy, lz = c.cvz * tc - c.dz;
        if (lx * lx + ly * ly + lz * lz > L2) return false;
        // |-d + cv t|^2 = dg2 + cv2 (t - ts)^2 with dg2 the global minimum: t must lie within w of ts.
        // The cancellation in dg2 (a few ulp of d2) moves w by up to ~2e-3 sqrt(d2 / cv2): covered twice over.
        const float dg2 = fmaxf(c.d2 - dcv * ts, 0.0f);
        const float w = sqrt_ub(fmaxf(L2 - dg2, 0.0f) * inv) + 1.0e-3f + 4.0e-3f * sqrt_ub(c.d2 * inv);
        t_lo = fmaxf(ts - w, 0.0f);
        t_hi = fminf(ts + w, 9.5f);
        if (t_lo > t_hi) return false;
    } else if (!(c.d2 <= L2)) {
        return false;
    }
#pragma unroll
    for (int it = 0; it < 2; ++it) {
        const float tm = 0.5f * (t_lo + t_hi);
        const float D = 0.5f * (t_hi - t_lo) + 1.0e-5f;
        const float hh = 0.5f * tm * tm;
        const float g0x = c.cvx * tm + c.cax * hh - c.dx, g0y = c.cvy * tm + c.cay * hh - c.dy,
                    g0z = c.cvz * tm + c.caz * hh - c.dz;
        const float g1x = c.cvx + c.cax * tm, g1y = c.cvy + c.cay * tm, g1z = c.cvz + c.caz * tm;
        const float g12 = g1x * g1x + g1y * g1y + g1z * g1z;
        const float Lr = (c.hr + 0.5f * c.can * D * D) * (1.0f + 1.0e-4f) + c.eps;
        const float Lr2 = Lr * Lr;
        const float g02 = g0x * g0x + g0y * g0y + g0z * g0z;
        if (!(g12 > 1.0e-8f)) {  // no relative drift at tm: |g| >= |g0| - slack over the whole window
            if (g02 > Lr2) return false;
            continue;
        }
        const float inv1 = rcp_fast(g12);
        const float us = -(g0x * g1x + g0y * g1y + g0z * g1z) * inv1;  // minimum of the linear part, relative to tm
        const float uc = fminf(fmaxf(us, -D), D);
        const float ex = g0x + g1x * uc, ey = g0y + g1y * uc, ez = g0z + g1z * uc;
        if (ex * ex + ey * ey + ez * ez > Lr2) return false;
        const float mx = g0x + g1x * us, my = g0y + g1y * us, mz = g0z + g1z * us;  // global minimum, no cancellation
        const float dgg = mx * mx + my * my + mz * mz;
        const float w = sqrt_ub(fmaxf(Lr2 - dgg, 0.0f) * inv1) + 1.0e-3f + 4.0e-3f * sqrt_ub(g02 * inv1);
        t_lo = fmaxf(t_lo, tm + us - w);
        t_hi = fminf(t_hi, tm + us + w);
        if (t_lo > t_hi) return false;
    }
    // the offsets are the times 0.5 m inside the window (2e-3: fp32 rounding of 2 t, and then some)
    m_lo = max((int)ceilf(2.0f * t_lo - 2.0e-3f), 0);
    m_hi = min((int)floorf(2.0f * t_hi + 2.0e-3f), PREDICT_OFFSETS - 1);
    return m_lo <= m_hi;
}

// ---- diagnostic variant (RCD_STEP_COUNT_CANDIDATES): every offset takes the radius test in k_pairs so that
// candidates can be counted per query; bit m set <=> offset m is a candidate that may be hit
__device__ __forceinline__ u32 predict_scan(const PairParams &P, const PredictCoef &c, u32 si, u32 sj, u32 pattern,
                                            int m_lo, int m_hi, u32 &n_exact) {
    u32 mask = 0;
    const float R2 = PREDICT_RADIUS * PREDICT_RADIUS;
    u32 ncand = 0;
#pragma unroll 1
    for (int m = 0; m < PREDICT_OFFSETS; ++m) {
        float t = 0.5f * (float)m, h = 0.5f * t * t;
        float ex = c.uvx * t + c.uax * h - c.dx, ey = c.uvy * t + c.uay * h - c.dy, ez = c.uvz * t + c.uaz * h - c.dz;
        float c2 = ex * ex + ey * ey + ez * ez;
        if (c2 > R2 * (1.0f + BAND_R2)) continue;
        if (c2 >= R2 * (1.0f - BAND_R2)) {
            ++n_exact;
            if (!exact_predict_radius(P, si, sj, pattern, m)) continue;
        }
        ++ncand;
        if (m >= m_lo && m <= m_hi && offset_may_hit(c, t)) mask |= 1u << m;
    }
    if (ncand) {
        atomicAdd(&P.counters->n_candidates, (unsigned long long)ncand);
        if (P.cand_count) atomicAdd(&P.cand_count[P.sorted_slot[si]], ncand);
    }
    return mask;
}

// ---- k_sample body: radius test + the 10 samples in fp32 for every offset in `mask` -----------------
// Returns the queue word for the exact stage: 0 (no offset can hit), RESOLVED | m | k << 8 when the
// winner of the max-risk merge and its first hit sample are beyond doubt in fp32, else the mask of
// the offsets the exact stage has to evaluate.
template <bool COUNT_CAND>
__device__ __forceinline__ u32 sample_predict(const PairParams &P, u32 si, u32 sj, u32 mask, u32 &n_exact) {
    const float4 a0 = P.P0[si], a1 = P.P1[si], a2 = P.P2[si];
    const float4 b0 = P.P0[sj], b1 = P.P1[sj], b2 = P.P2[sj];
    const u32 pattern = meta_pattern(__float_as_uint(a2.w));
    const PredictCoef c = predict_coef(a0, a1, a2, b0, b1, b2, pattern);
    const float rvx = a1.x - b1.x, rvy = a1.y - b1.y, rvz = a1.z - b1.z;
    const float rax = a2.x - b2.x, ray = a2.y - b2.y, raz = a2.z - b2.z;
    const float R2 = PREDICT_RADIUS * PREDICT_RADIUS;
    const float safe = (a0.w + b0.w) * 0.5f + 5.0f;
    const float band = sqrtf(c.safe_b2) - safe;                 // the guard band of predict_coef
    const float safe_in = fmaxf(safe - band, 0.0f), safe_in2 = safe_in * safe_in;
    const float inv_safe = 1.0f / safe;
    u32 maybe_mask = 0;      // offsets with a sample inside safe + band
    bool doubt = false;      // some decisive sample lies inside the band
    float best = -1.0f, second = -1.0f;
    int best_m = -1, best_k = 0;
    while (mask) {
        const int m = __ffs(mask) - 1;
        mask &= mask - 1;
        const float t = 0.5f * (float)m, h = 0.5f * t * t;
        if (!COUNT_CAND) {  // with COUNT_CAND both tests were already taken in k_pairs
            if (!offset_may_hit(c, t)) continue;  // none of the 10 samples can come within the safe distance
            float ex = c.uvx * t + c.uax * h - c.dx, ey = c.uvy * t + c.uay * h - c.dy, ez = c.uvz * t + c.uaz * h - c.dz;
            float c2 = ex * ex + ey * ey + ez * ez;
            if (c2 > R2 * (1.0f + BAND_R2)) continue;
            if (c2 >= R2 * (1.0f - BAND_R2)) {
                ++n_exact;
                if (!exact_predict_radius(P, si, sj, pattern, m)) continue;
            }
        }
        const float gx = c.cvx * t + c.cax * h - c.dx, gy = c.cvy * t + c.cay * h - c.dy, gz = c.cvz * t + c.caz * h - c.dz;
        int first = -1;
        float r2first = 0.0f;
#pragma unroll
        for (int k = PREDICT_STEPS - 1; k >= 0; --k) {  // descending: the last assignment is the first sample
            const float tau = 0.1f * (float)k, hh = 0.5f * tau * tau;
            float rx = gx + rvx * tau + rax * hh, ry = gy + rvy * tau + ray * hh, rz = gz + rvz * tau + raz * hh;
            float r2 = rx * rx + ry * ry + rz * rz;
            if (r2 <= c.safe_b2) { first = k; r2first = r2; }
        }
        if (first < 0) continue;  // no sample within safe + band: certainly no hit at this offset
        maybe_mask |= 1u << m;
        if (r2first > safe_in2) { doubt = true; continue; }  // the first candidate sample is inside the band
        // certain hit at sample `first`, and every earlier sample is certainly outside: the parts of the
        // risk that differ between offsets (collision_detection.py:371-374) decide the merge
        const float part = 0.3f * (1.0f - sqrtf(r2first) * inv_safe) + 0.3f * (1.0f - 0.01f * (float)first);
        if (part > best) { second = best; best = part; best_m = m; best_k = first; }
        else if (part > second) second = part;
    }
    if (maybe_mask == 0) return 0;
    // a runner-up within 1e-4 (fp32 error of `part` is ~1e-5) or any sample in the band: fp64 decides
    if (doubt || best_m < 0 || best - second <= 1.0e-4f) return maybe_mask;
    return RESOLVED | (u32)best_m | ((u32)best_k << 8);
}

// ---- S2, compute-node pair function in fp32 (compute_node.py:258-292) --------------------------------
__device__ __forceinline__ bool narrow_compute_node(const PairParams &P, const float4 &a0, const float4 &a1,
                                                    const float4 &a2, const float4 &b0, const float4 &b1,
                                                    const float4 &b2, bool self, bool undecided) {
    float dx = b0.x - a0.x, dy = b0.y - a0.y, dz = b0.z - a0.z;
    float d2 = dx * dx + dy * dy + dz * dz;
    if (undecided) return true;  // fp32 could not decide the radius test (compute_node.py:113-116)
    if (self) return false;                              // compute_node.py:251-252
    if (d2 > 2500.0f * (1.0f + BAND_R2)) return false;   // current_distance > 50
    if (meta_pattern(__float_as_uint(a2.w)) == 0u || meta_pattern(__float_as_uint(b2.w)) == 0u)
        return false;                                    // predict_position needs >= 2 samples (:202-203)
    float rvx = a1.x - b1.x, rvy = a1.y - b1.y, rvz = a1.z - b1.z;
    float fx = dx - rvx * P.pt, fy = dy - rvy * P.pt, fz = dz - rvz * P.pt;  // future_j - future_i
    float fut2 = fx * fx + fy * fy + fz * fz;
    float rs2 = rvx * rvx + rvy * rvy + rvz * rvz;
    if (fut2 > d2 * (1.0f + 1.0e-4f) + 1.0e-6f && d2 > 16.0f * (1.0f + 1.0e-4f)) return false;  // moving apart
    float fut = fmaxf(sqrtf(fut2), 0.1f);
    return !(0.4f * sqrtf(rs2) < P.threshold * fut * (1.0f - 1.0e-4f));  // risk >= threshold (maybe)
}

// queue-full fallback of the predict path: finish the pair in place (correct, slower, out of line)
template <bool COUNT_CAND>
__device__ __noinline__ void finish_predict_pair(const PairParams &P, u32 si, u32 sj, u32 mask) {
    u32 dummy = 0;
    const u32 m2 = sample_predict<COUNT_CAND>(P, si, sj, mask, dummy);
    if (m2) finish_entry_inline<RCD_MODE_PREDICT>(P, si, sj, m2);
}

// warp-aggregated append to a global queue; returns false for the lanes whose entry did not fit
__device__ __forceinline__ bool global_push(QEntry *q, u32 cap, unsigned long long *count, bool flag, u32 si, u32 sj,
                                            u32 mask) {
    const u32 ballot = __ballot_sync(FULL_MASK, flag);
    if (ballot == 0) return true;
    unsigned long long base = 0;
    const u32 leader = __ffs(ballot) - 1;
    if ((threadIdx.x & 31u) == leader) base = atomicAdd(count, (unsigned long long)__popc(ballot));
    base = __shfl_sync(FULL_MASK, base, leader);
    if (!flag) return true;
    const unsigned long long at = base + __popc(ballot & lanemask_lt());
    if (at >= cap) return false;
    QEntry e;
    e.si = si; e.sj = sj; e.mask = mask;
    q[at] = e;
    return true;
}
// predict: the offsets of the pair (si, sj) the later phases have to look at (0: none)
template <bool COUNT_CAND>
__device__ __forceinline__ u32 predict_mask(const PairParams &P, const float4 &a0, const float4 &a1, const float4 &a2,
                                            const float4 &b0, const float4 &b1, const float4 &b2, u32 si, u32 sj,
                                            u32 pat, u32 &n_exact) {
    int m_lo = 0, m_hi = PREDICT_OFFSETS - 1;
    if (COUNT_CAND) {  // diagnostic: every offset takes the radius test here so that candidates can be counted
        const bool in = predict_window(window_coef(a0, a1, a2, b0, b1, b2, pat), m_lo, m_hi);
        if (!in) { m_lo = 1; m_hi = 0; }
        const PredictCoef c = predict_coef(a0, a1, a2, b0, b1, b2, pat);
        return predict_scan(P, c, si, sj, pat, m_lo, m_hi, n_exact);
    }
    if (predict_window(window_coef(a0, a1, a2, b0, b1, b2, pat), m_lo, m_hi))
        return (2u << m_hi) - (1u << m_lo);  // offsets m_lo..m_hi; the per-offset phases test each of them
    return 0u;
}

// pair-queue-full fallback of k_pairs: everything k_narrow and k_exact would do for one pair, in place
// (correct, slower, out of line)
template <int MODE, bool COUNT_CAND>
__device__ __noinline__ u32 narrow_entry_inline(const PairParams &P, u32 si_flags, u32 sj) {
    const u32 si = si_flags & QA_SI_MASK;
    const bool inr = (si_flags & QA_INR) != 0, und = (si_flags & QA_UND) != 0;
    if (si == sj && MODE != RCD_MODE_COMPUTE_NODE) return 0u;  // _spatial_filtering strips self (:224-225)
    const float4 a0 = P.P0[si], a1 = P.P1[si], a2 = P.P2[si];
    const float4 b0 = P.P0[sj], b1 = P.P1[sj], b2 = P.P2[sj];
    u32 n_pot = 0;
    if (MODE == RCD_MODE_DETECT) {
        if (und || narrow_detect(a0, a1, a2, b0, b1, b2, P.T))
            n_pot += finish_entry_inline<MODE>(P, si, sj, und ? RADIUS_UNDECIDED : 0u);
    } else if (MODE == RCD_MODE_COMPUTE_NODE) {
        if (narrow_compute_node(P, a0, a1, a2, b0, b1, b2, si == sj, und))
            finish_entry_inline<MODE>(P, si, sj, und ? RADIUS_UNDECIDED : 0u);
    } else {
        const u32 pat = meta_pattern(__float_as_uint(a2.w));
        const bool nohist = pat == RCD_PAT_NO_HISTORY;
        if ((nohist || MODE == MODE_PREDICT_WITH_DETECT) && (inr || und)) {
            const bool twice = nohist && MODE == MODE_PREDICT_WITH_DETECT;
            if (und || narrow_detect(a0, a1, a2, b0, b1, b2, 10.0f))
                n_pot += finish_entry_inline<MODE>(P, si, sj, (und ? RADIUS_UNDECIDED : 0u) | (twice ? ENTRY_TWICE : 0u));
        }
        if (!nohist) {
            u32 dummy = 0;
            const u32 mask = predict_mask<COUNT_CAND>(P, a0, a1, a2, b0, b1, b2, si, sj, pat, dummy);
            if (mask) finish_predict_pair<COUNT_CAND>(P, si, sj, mask);
        }
    }
    return n_pot;
}

__device__ __forceinline__ float abs3(float x, float y, float z) { return fabsf(x) + fabsf(y) + fabsf(z); }
__device__ __forceinline__ float rsqrt_fast(float x) {
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// Volume a neighbour must lie in to matter for one query: a ball of radius Rq for radius queries; for
// predict queries the capsule of radius 100 (+ slack) about the chord of the centre path
// c(t) = uv t + ua t^2/2, t in [0, 9.5] (:728-741): the path leaves its chord by at most |ua| 9.5^2 / 8.
// w is the chord, rad the radius.
struct QueryVolume {
    float wx, wy, wz, inv_w2, rad;
    float fv, fa;  // which parts of the motion the centre path follows (radius queries: all of it)
    float an;      // |a_i|, rounded up
    bool radius_query;
};
template <int MODE>
__device__ __forceinline__ QueryVolume query_volume(const float4 &p1, const float4 &p2, u32 pattern, float Rq) {
    QueryVolume v;
    // queries that take the radius-R test (detect-like); the others are predict queries
    v.radius_query = !is_predict(MODE) || pattern == RCD_PAT_NO_HISTORY;
    v.fv = v.radius_query ? 1.0f : ((pattern >= RCD_PAT_CONSTANT_VELOCITY) ? 1.0f : 0.0f);
    v.fa = v.radius_query ? 1.0f : ((pattern == RCD_PAT_ACCELERATING) ? 1.0f : 0.0f);
    v.an = sqrt_ub(p2.x * p2.x + p2.y * p2.y + p2.z * p2.z);
    v.wx = v.wy = v.wz = v.inv_w2 = 0.0f;
    if (!v.radius_query) {
        v.wx = p1.x * v.fv * 9.5f + p2.x * v.fa * 45.125f;
        v.wy = p1.y * v.fv * 9.5f + p2.y * v.fa * 45.125f;
        v.wz = p1.z * v.fv * 9.5f + p2.z * v.fa * 45.125f;
        float w2 = v.wx * v.wx + v.wy * v.wy + v.wz * v.wz;
        v.rad = (PREDICT_RADIUS + 11.28125f * v.an * v.fa) * (1.0f + 1.0e-5f) + 2.0e-2f + 1.0e-5f * sqrtf(w2);
        if (!(w2 < 1.0e30f) || !(v.rad < 1.0e30f)) {  // non-finite motion: scan everything
            v.wx = v.wy = v.wz = w2 = 0.0f;
            v.rad = 1.0e18f;
        }
        v.inv_w2 = w2 > 1.0e-12f ? 1.0f / w2 : 0.0f;
    } else {
        v.rad = Rq * (1.0f + 1.0e-5f) + 1.0e-3f;
    }
    return v;
}

// objects of the cell row `rr` of a tile's box: position of the first one in cell order, and how many.  The first
// TILE_ROWS rows of a box carry their own x range (k_tile_plan: the box is the bounding box of 32 query volumes --
// capsules pointing in all directions -- and its corners are empty; a row only spans the cells some volume reaches).
constexpr int TILE_ROWS = 64;
struct TileBox { int x0, x1, y0, y1, z0, z1; };
__device__ __forceinline__ void row_span(const PairParams &P, const TileBox &b, u32 tile, int rr, u32 &lo, u32 &cnt) {
    const int ny_span = b.y1 - b.y0 + 1;
    const int yy = b.y0 + rr % ny_span, zz = b.z0 + rr / ny_span;
    int x0 = b.x0, x1 = b.x1;
    if (rr < TILE_ROWS) {
        const uint2 rx = P.tile_rowx[(size_t)tile * TILE_ROWS + rr];
        x0 = (int)rx.x;
        x1 = (int)rx.y;
    }
    lo = 0;
    cnt = 0;
    if (x0 > x1) return;  // no query volume reaches this row
    const u32 c0 = (u32)((zz * P.g.ny + yy) * P.g.nx + x0);
    const u32 first = P.cell_begin[c0], last = P.cell_begin[c0 + (u32)(x1 - x0) + 1u];
    lo = first;
    cnt = last - first;
}

// work items of k_pairs: {tile, row batch | flags, first chunk in that batch, number of chunks}: a run of
// chunks in the tile's sequence of (row batch, chunk), which may continue into the following row batches
constexpr u32 ITEM_FIRST = 1u << 30;  // the item that subtracts the query's hit on itself from the candidate count
constexpr u32 ITEM_RBASE_MASK = (1u << 30) - 1u;
constexpr int PLAN_ITEMS_PER_TILE = 32;
constexpr int ITEMS_PER_TILE_CAP = PLAN_ITEMS_PER_TILE;

// -------------------------------------------------------------------------------------------------
// k_tile_plan: one warp per tile.  The cost of a tile is the number of objects under its box, which spans
// four orders of magnitude on clustered frames (hotspot density ~ 1/r): the plan cuts every tile into work
// items of about the same size -- a run of chunks of one row batch -- so that the persistent warps of k_pairs
// stay busy to the end.  Also stores the tile's cell box (computed once, here).
// -------------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(128) k_tile_plan(PairParams P) {
    const u32 lane = threadIdx.x & 31u;
    const GridParams g = P.g;
    const float Rq = is_predict(MODE) ? PREDICT_RADIUS : P.R;
    const u32 nwarps = gridDim.x * (blockDim.x >> 5);
    for (u32 tile = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); tile < P.ntiles; tile += nwarps) {
        const u32 qi = tile * TQ + lane;
        float4 p0 = make_float4(0.f, 0.f, 0.f, 0.f), p1 = p0, p2 = p0;
        if (qi < P.n_owned) {
            const u32 s = P.qorder[qi];
            p0 = P.P0[s];
            p1 = P.P1[s];
            p2 = P.P2[s];
        }
        // a query without a position (retired slot, NaN) is a lane past the queries: it widens no box.  A tile of them
        // only (the trailing tiles of the query order, query_key) gets an empty box -- no rows, no work items; the
        // clamped box of "no lane" would be inverted, {nx-1..0, ny-1..0, nz-1..0}, with (2-ny)(2-nz) rows
        const bool valid = qi < P.n_owned && p0.x == p0.x;
        if (!__any_sync(FULL_MASK, valid)) {
            if (lane == 0) {
                P.tile_box[2 * (size_t)tile] = make_int4(1, 0, 1, 0);
                P.tile_box[2 * (size_t)tile + 1] = make_int4(1, 0, 0, 0);
            }
            continue;
        }
        const QueryVolume v = query_volume<MODE>(p1, p2, meta_pattern(__float_as_uint(p2.w)), Rq);
        // cells of the bounding box of the tile's query volumes (cell_coord is monotone, so a
        // neighbour inside the box in space is inside it in cells; 0.05 m + 1 ulp covers the fp32 sums)
        const float big = 3.0e38f;
        const float lox = warp_minf(valid ? fminf(p0.x, p0.x + v.wx) - v.rad : big);
        const float hix = warp_maxf(valid ? fmaxf(p0.x, p0.x + v.wx) + v.rad : -big);
        const float loy = warp_minf(valid ? fminf(p0.y, p0.y + v.wy) - v.rad : big);
        const float hiy = warp_maxf(valid ? fmaxf(p0.y, p0.y + v.wy) + v.rad : -big);
        const float loz = warp_minf(valid ? fminf(p0.z, p0.z + v.wz) - v.rad : big);
        const float hiz = warp_maxf(valid ? fmaxf(p0.z, p0.z + v.wz) + v.rad : -big);
        TileBox b;
        b.x0 = cell_coord(lox - (0.05f + 4.0e-7f * fabsf(lox)), g.ox, g.inv_cell, g.nx);
        b.x1 = cell_coord(hix + (0.05f + 4.0e-7f * fabsf(hix)), g.ox, g.inv_cell, g.nx);
        b.y0 = cell_coord(loy - (0.05f + 4.0e-7f * fabsf(loy)), g.oy, g.inv_cell, g.ny);
        b.y1 = cell_coord(hiy + (0.05f + 4.0e-7f * fabsf(hiy)), g.oy, g.inv_cell, g.ny);
        b.z0 = cell_coord(loz - (0.05f + 4.0e-7f * fabsf(loz)), g.oz, g.inv_cell_z, g.nz);
        b.z1 = cell_coord(hiz + (0.05f + 4.0e-7f * fabsf(hiz)), g.oz, g.inv_cell_z, g.nz);
        if (lane == 0) {
            P.tile_box[2 * (size_t)tile] = make_int4(b.x0, b.x1, b.y0, b.y1);
            P.tile_box[2 * (size_t)tile + 1] = make_int4(b.z0, b.z1, 0, 0);
        }
        const int nrows = (b.y1 - b.y0 + 1) * (b.z1 - b.z0 + 1);
        const int nbatches = (nrows + TQ - 1) / TQ;
        // x range of every cell row: union over the tile's queries (lane = query) of what their volume reaches inside
        // the row's y band, reduced over the warp with two integer REDUX per row.  A capsule (chord w, radius rad) is
        // covered by 5 discs about the chord points k/4 with radius sqrt(rad^2 + (|w|/8)^2); everything in the x-y
        // projection (conservative for the 3-D volume).  Row rr's range is kept by lane rr % 32 and stored per batch.
        {
            const int ny_span = b.y1 - b.y0 + 1;
            float r2q = v.rad * v.rad + (v.wx * v.wx + v.wy * v.wy) * (1.0f / 64.0f);
            const bool everything = valid && !(r2q < 1.0e30f);  // non-finite motion
            if (!valid || everything) r2q = -1.0f;              // (no disc of this lane reaches any row)
            const bool any_everything = __any_sync(FULL_MASK, everything);
            float dcx[5], dcy[5];
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                dcx[k] = fmaf(v.wx, 0.25f * (float)k, p0.x);
                dcy[k] = fmaf(v.wy, 0.25f * (float)k, p0.y);
            }
            const int nr = min(nrows, TILE_ROWS);
            int keep_lo = 0x7fffffff, keep_hi = (int)0x80000000;  // ordered-int encodings of this lane's row range
            for (int rr = 0; rr < nr; ++rr) {
                const int yy = b.y0 + rr % ny_span;
                // the row holds the objects with floor((y - oy) / cell) == yy (border rows also what lies beyond the grid)
                const float eps = 0.01f * g.cell + 2.0e-6f * (fabsf(g.oy) + fabsf((float)(yy + 1) * g.cell));
                const float ya = (yy <= 0) ? -big : g.oy + (float)yy * g.cell - eps;
                const float yb = (yy >= g.ny - 1) ? big : g.oy + (float)(yy + 1) * g.cell + eps;
                float xmin = big, xmax = -big;
#pragma unroll
                for (int k = 0; k < 5; ++k) {
                    const float dy = fmaxf(fmaxf(ya - dcy[k], dcy[k] - yb), 0.0f);
                    const float h2 = r2q - dy * dy;
                    if (h2 >= 0.0f) {
                        const float hx = sqrt_ub(h2);
                        xmin = fminf(xmin, dcx[k] - hx);
                        xmax = fmaxf(xmax, dcx[k] + hx);
                    }
                }
                if (any_everything) { xmin = -big; xmax = big; }
                const int lo_all = __reduce_min_sync(FULL_MASK, float_ordered(xmin));
                const int hi_all = __reduce_max_sync(FULL_MASK, float_ordered(xmax));
                if ((int)lane == (rr & 31)) { keep_lo = lo_all; keep_hi = hi_all; }
                if ((rr & 31) == 31 || rr == nr - 1) {  // a batch of rows is complete: lane l stores row (rr & ~31) + l
                    const int row = (rr & ~31) + (int)lane;
                    if (row <= rr) {
                        const float fx0 = ordered_float(keep_lo), fx1 = ordered_float(keep_hi);
                        uint2 rx = make_uint2(1u, 0u);  // empty
                        if (fx0 <= fx1) {
                            const int cx0 = cell_coord(fx0 - (0.05f + 4.0e-7f * fabsf(fx0)), g.ox, g.inv_cell, g.nx);
                            const int cx1 = cell_coord(fx1 + (0.05f + 4.0e-7f * fabsf(fx1)), g.ox, g.inv_cell, g.nx);
                            rx = make_uint2((u32)max(cx0, b.x0), (u32)min(cx1, b.x1));
                        }
                        P.tile_rowx[(size_t)tile * TILE_ROWS + row] = rx;  // (read back below by the same lane)
                    }
                    keep_lo = 0x7fffffff;
                    keep_hi = (int)0x80000000;
                }
            }
        }
        u32 tot_chunks = 0;
        for (int bt = 0; bt < nbatches; ++bt) {
            u32 lo = 0, cnt = 0;
            const int rr = bt * TQ + (int)lane;
            if (rr < nrows) row_span(P, b, tile, rr, lo, cnt);
            tot_chunks += (warp_sum(cnt) + CH - 1) / CH;
        }
        if (tot_chunks == 0) continue;
        // at most PLAN_ITEMS_PER_TILE items of K chunks each; item j starts at chunk j K of the tile's sequence
        const u32 K = max(P.item_chunks, (tot_chunks + PLAN_ITEMS_PER_TILE - 1) / PLAN_ITEMS_PER_TILE);
        const u32 n_it = (tot_chunks + K - 1) / K;
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(&P.counters->n_items, (unsigned long long)n_it);
        base = __shfl_sync(FULL_MASK, base, 0);
        u32 cum = 0;
        for (int bt = 0; bt < nbatches; ++bt) {
            u32 lo = 0, cnt = 0;
            const int rr = bt * TQ + (int)lane;
            if (rr < nrows) row_span(P, b, tile, rr, lo, cnt);
            const u32 nch = (warp_sum(cnt) + CH - 1) / CH;
            // the items that start inside this batch's chunks [cum, cum + nch)
            const u32 j0 = (cum + K - 1) / K, j1 = min((cum + nch + K - 1) / K, n_it);
            for (u32 j = j0 + lane; j < j1; j += 32)
                if (base + j < P.items_cap)
                    P.items[base + j] = make_uint4(tile, (u32)(bt * TQ) | (j == 0 ? ITEM_FIRST : 0u), j * K - cum, min(K, tot_chunks - j * K));
            cum += nch;
        }
    }
}

// -------------------------------------------------------------------------------------------------
// k_pairs: the S1 filter (see the head of this file).
// -------------------------------------------------------------------------------------------------
// SLOW: the overflow pass.  A warp of the regular pass that finds the pair queue full records where it stopped
// (work item, row batch, chunk) and moves on; the overflow pass redoes exactly those parts and finishes every
// surviving pair in place (narrow phase, fp64 decision, emission -- out of line, one pair per thread).  It is
// launched after every regular pass and returns at once when nothing was recorded, so the regular pass carries
// no call in its loops.
template <int MODE, bool COUNT_CAND, bool SLOW>
#ifndef RCD_PAIR_MIN_BLOCKS
#define RCD_PAIR_MIN_BLOCKS 5
#endif
__global__ void __launch_bounds__(PAIR_THREADS, SLOW ? 4 : RCD_PAIR_MIN_BLOCKS) k_pairs(PairParams P) {
    __shared__ WarpShared shared[PAIR_WARPS];
    WarpShared &ws = shared[threadIdx.x >> 5];
    const u32 lane = threadIdx.x & 31u;
    const GridParams g = P.g;
    constexpr bool PRED = is_predict(MODE);
    constexpr bool FUSED = MODE == MODE_PREDICT_WITH_DETECT;
    constexpr bool USE_CAPSULE = PRED && COUNT_CAND;  // diagnostic variant: every neighbour inside the capsule goes on
    constexpr bool t1_on = MODE != RCD_MODE_COMPUTE_NODE && !USE_CAPSULE;
    const float tm = P.tm, D = P.D, h2 = 0.5f * tm * tm;
    const float Rq = PRED ? PREDICT_RADIUS : P.R;
    const float R2_hi = Rq * Rq * (1.0f + BAND_R2), R2_lo = Rq * Rq * (1.0f - BAND_R2);
    const float FAR = 3.0e38f;
    u32 n_pot = 0;                                // per-lane statistics, flushed once at the end
    unsigned long long n_chunks = 0;              // (uniform) chunks of 32 neighbours this warp filtered
    u32 qa_block = QA_NO_BLOCK, qa_used = 0;      // this warp's block of the pair queue (uniform)
    bool qa_full = false;                         // (uniform) the pair queue has no block left

    const u32 n_work = SLOW ? (u32)min(P.counters->n_overflow, (unsigned long long)P.ovf_cap)
                            : (u32)min(P.counters->n_items, (unsigned long long)P.items_cap);

    for (;;) {
        u32 idx = 0;
        if (lane == 0) idx = atomicAdd(P.tile_counter + (SLOW ? 1 : 0), 1u);
        idx = __shfl_sync(FULL_MASK, idx, 0);
        if (idx >= n_work) break;
        // a work item: chunks [c_lo, c_hi) of one row batch of one tile (k_tile_plan), or -- overflow pass --
        // what the regular pass left of an item when the pair queue ran out
        const uint4 it = SLOW ? P.ovf[idx] : P.items[idx];
        const u32 tile = it.x;
        const int rbase0 = (int)(it.y & ITEM_RBASE_MASK);
        const bool first_item = (it.y & ITEM_FIRST) != 0;
        u32 remaining = it.w;  // chunks left to do

        const u32 qi = tile * TQ + lane;
        const bool valid = qi < P.n_owned;
        u32 s = 0;
        float4 p0 = make_float4(0.f, 0.f, 0.f, 0.f), p1 = p0, p2 = p0;
        if (valid) {
            s = P.qorder[qi];
            p0 = P.P0[s];
            p1 = P.P1[s];
            p2 = P.P2[s];
        }
        const u32 pattern = meta_pattern(__float_as_uint(p2.w));
        const QueryVolume vol = query_volume<MODE>(p1, p2, pattern, Rq);
        const bool radius_query = vol.radius_query;
        const bool counts = valid && (radius_query || FUSED);  // in-radius neighbours are candidates of this query
        const float wx = vol.wx, wy = vol.wy, wz = vol.wz, inv_w2 = vol.inv_w2, rad = vol.rad;
        const float fv = vol.fv, fa = vol.fa, an = vol.an;
        // T1: this query's half.  Radius queries follow their true motion (the detect trajectory, :229-294),
        // predict queries the motion of their pattern (:728-741): M = centre at tm, MV = its velocity there.
        const float uvx = p1.x * fv, uvy = p1.y * fv, uvz = p1.z * fv;
        const float uax = p2.x * fa, uay = p2.y * fa, uaz = p2.z * fa;
        const float Mx = fmaf(uax, h2, fmaf(uvx, tm, p0.x)), My = fmaf(uay, h2, fmaf(uvy, tm, p0.y)),
                    Mz = fmaf(uaz, h2, fmaf(uvz, tm, p0.z));
        const float MVx = fmaf(uax, tm, uvx), MVy = fmaf(uay, tm, uvy), MVz = fmaf(uaz, tm, uvz);
        // The linear part of the relative trajectory must come within  L = A_i + B_j + kq |Ua_i - a_j|  of zero for
        // some u in [-D, Dhi].  Predict queries: a hit at offset t_m = tm + u, sample tau is
        //   |g(t_m) + rv tau + ra tau^2 / 2| <= safe,   g(tm + u) = g0 + g1 u + ca u^2 / 2  (exact),
        // and with rv = g1 + delta, delta = (v_i - uv_i) - ca tm, this is
        //   |g0 + g1 (u + tau)| <= safe + 0.405 |ra| + 0.9 |delta| + |ca| D^2 / 2,   u + tau in [-D, D + 0.9]:
        // the motion of the samples along g1 only stretches the window (Dhi = D + 0.9); what is left of it,
        // 0.9 |delta| <= 0.9 |v_i - uv_i| + 0.9 tm |ca|, and |ra| <= |ca| + |a_i - Ua_i| go into A and kq
        // (ca = Ua_i - a_j: the acceleration the query's centre path follows, minus the neighbour's).  The detect
        // part of the fused frame follows the same g for accelerating patterns: its samples g(0.1 k), k < 100, lie
        // inside the stretched window and the curvature up to there, |ca| (D + 0.4)^2 / 2, is below kq |ca|.
        // Radius queries have no sample motion: Dhi = D, kq = D^2 / 2.  err: fp32 rounding of M, MV (x4).
        float A, kq, Dhi;
        {
            Dhi = radius_query ? D : D + 0.9f;
            const float err = 5.0e-7f * (abs3(p0.x, p0.y, p0.z) + tm * abs3(uvx, uvy, uvz) + h2 * abs3(uax, uay, uaz)) +
                              5.0e-7f * (D + 0.9f) * (abs3(uvx, uvy, uvz) + tm * abs3(uax, uay, uaz));
            if (radius_query) {
                A = 0.5f * p0.w + 5.0f + 2.0e-2f + err;
                kq = 0.5f * D * D * (1.0f + 1.2e-4f);
            } else {
                const float dvx = p1.x - uvx, dvy = p1.y - uvy, dvz = p1.z - uvz;
                const float dvn = sqrt_ub(dvx * dvx + dvy * dvy + dvz * dvz);
                A = 0.5f * p0.w + 5.0f + 2.0e-2f + 0.405f * an * (1.0f - fa) + 0.9f * dvn + err;
                kq = (0.405f + 0.9f * tm + 0.5f * D * D) * (1.0f + 1.2e-4f);
            }
            A *= 1.0f + 1.0e-4f;
        }
        // the clamp of the minimiser to [-D, Dhi] as a saturating FMA: uc = -D + span * sat((u + D) / span)
        const float span = pin_reg(D + Dhi), inv_span = pin_reg(1.0f / (D + Dhi)), off_span = pin_reg(D / (D + Dhi));
        // The filter keeps four bit masks per lane and chunk (bit = staged neighbour): im = inside the radius for
        // certain, nm = inside radius + guard band, tm = passed T1 (or the capsule test), bm = within the compute-node
        // distance bound.  What passes, per lane:  (tm & useT & (im | ~andI)) | (im & orI) | (bm & orB) | (nm & ~im):
        //   radius query, T1 on  : in the radius and T1            radius query, T1 off : in the radius
        //   predict query        : T1 (+ everything in the radius where the fused detect part follows another trajectory)
        //   compute-node         : within min(radius, 50 m)
        // (the masks are built from sign bits: d2 - R2lo < 0, d2 - next(R2hi) < 0, bound - value < 0)
        float R2lo_l = -1.0f, R2hi_n = -1.0f, dmaxB = -1.0f;
        u32 useT = 0u, andI = 0u, orI = 0u, orB = 0u;
        if (counts) { R2lo_l = R2_lo; R2hi_n = __uint_as_float(__float_as_uint(R2_hi) + 1u); }
        if (valid) {
            if (MODE == RCD_MODE_COMPUTE_NODE) { dmaxB = fminf(R2_lo, 2500.0f * (1.0f + 2.0f * BAND_R2)); orB = ~0u; }  // current_distance <= 50
            else if (radius_query) { if (t1_on) { useT = ~0u; andI = ~0u; } else orI = ~0u; }
            else {
                useT = ~0u;
                if (FUSED && pattern != RCD_PAT_ACCELERATING) orI = ~0u;  // detect follows another trajectory: all of them
            }
        }
        const float rad2 = rad * rad;
        u32 ncand = 0;  // candidates decided by the filter itself

        // the tile's cell box (k_tile_plan)
        TileBox box;
        {
            const int4 bxy = P.tile_box[2 * (size_t)tile], bz = P.tile_box[2 * (size_t)tile + 1];
            box.x0 = bxy.x; box.x1 = bxy.y; box.y0 = bxy.z; box.y1 = bxy.w; box.z0 = bz.x; box.z1 = bz.y;
        }
        const int nrows = (box.y1 - box.y0 + 1) * (box.z1 - box.z0 + 1);

        bool stopped = false;  // (uniform) regular pass: the pair queue ran out in this item
        if (!SLOW && qa_full) {  // nothing can be queued any more: hand the whole item to the overflow pass
            if (lane == 0) {
                const unsigned long long k = atomicAdd(&P.counters->n_overflow, 1ULL);
                if (k < P.ovf_cap) P.ovf[k] = make_uint4(tile, it.y & ~ITEM_FIRST, it.z, it.w);
            }
            stopped = true;
        }
        for (int rbase = rbase0; rbase < nrows && remaining && !stopped; rbase += TQ) {
            // ---- span of one cell row per lane: two loads from the dense cell table ------------------
            u32 lo = 0, rcnt = 0;
            if ((int)lane + rbase < nrows) row_span(P, box, tile, rbase + (int)lane, lo, rcnt);
            u32 incl = rcnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                u32 t = __shfl_up_sync(FULL_MASK, incl, o);
                if (lane >= (u32)o) incl += t;
            }
            __syncwarp();  // previous batch's readers of row_* are done
            ws.row_lo[lane] = lo;
            ws.row_prefix[lane] = incl - rcnt;
            if (lane == 31) ws.row_prefix[TQ] = incl;
            __syncwarp();
            const u32 total = ws.row_prefix[TQ];
            const u32 nchunks = (total + CH - 1) / CH;

            // chunk c of the flattened spans: cp.async of the lane's own object into the landing zone
            auto stage = [&](u32 c, StagePacked &b) {
                const u32 f = c * CH + lane;
                if (f < total) {
                    int a = 0, z = TQ - 1;  // last row r with prefix[r] <= f
                    while (a < z) {
                        int mid = (a + z + 1) >> 1;
                        if (ws.row_prefix[mid] <= f) a = mid; else z = mid - 1;
                    }
                    const u32 src = ws.row_lo[a] + (f - ws.row_prefix[a]);
                    cp_async16(&ws.r0[lane], P.P0 + src);
                    cp_async16(&ws.r1[lane], P.P1 + src);
                    cp_async16(&ws.r2[lane], P.P2 + src);
                    b.pos[lane] = src;
                }
                cp_async_commit();
            };
            // ... and, once it has landed, the lane's object as operands of the packed filter: the position, and
            // the neighbour's half of T1 (N = position at tm, NV = velocity at tm, B = its share of the bound).
            // The last chunk is padded with an object no query can reach instead of bound checks per test.
            auto relayout = [&](u32 c, StagePacked &b) {
                const u32 f = c * CH + lane;
                float x = 1.0e30f, y = 1.0e30f, z = 1.0e30f, B = 0.0f;
                float nx = -1.0e18f, ny = -1.0e18f, nz = -1.0e18f, nvx = 0.0f, nvy = 0.0f, nvz = 0.0f, nax = 0.0f, nay = 0.0f, naz = 0.0f;
                if (f < total) {
                    const float4 q0 = ws.r0[lane], q1 = ws.r1[lane], q2 = ws.r2[lane];
                    x = q0.x; y = q0.y; z = q0.z;
                    if (t1_on) {
                        nx = -fmaf(q2.x, h2, fmaf(q1.x, tm, q0.x));
                        ny = -fmaf(q2.y, h2, fmaf(q1.y, tm, q0.y));
                        nz = -fmaf(q2.z, h2, fmaf(q1.z, tm, q0.z));
                        nvx = -fmaf(q2.x, tm, q1.x);
                        nvy = -fmaf(q2.y, tm, q1.y);
                        nvz = -fmaf(q2.z, tm, q1.z);
                        const float err = 5.0e-7f * (abs3(q0.x, q0.y, q0.z) + tm * abs3(q1.x, q1.y, q1.z) + h2 * abs3(q2.x, q2.y, q2.z)) +
                                          5.0e-7f * (D + 0.9f) * (abs3(q1.x, q1.y, q1.z) + tm * abs3(q2.x, q2.y, q2.z));
                        B = (0.5f * q0.w + err) * (1.0f + 1.0e-4f);
                        nax = -q2.x; nay = -q2.y; naz = -q2.z;
                    }
                }
                const u32 e = lane >> 1, h = lane & 1u;
                float *xy = reinterpret_cast<float *>(&b.xy[e]);
                xy[h] = x; xy[2u + h] = y;
                float *zb = reinterpret_cast<float *>(&b.zb[e]);
                zb[h] = z; zb[2u + h] = B;
                if (t1_on) {
                    float *nxy = reinterpret_cast<float *>(&b.nxy[e]);
                    nxy[h] = nx; nxy[2u + h] = ny;
                    float *nzv = reinterpret_cast<float *>(&b.nzv[e]);
                    nzv[h] = nz; nzv[2u + h] = nvx;
                    float *nvyz = reinterpret_cast<float *>(&b.nvyz[e]);
                    nvyz[h] = nvy; nvyz[2u + h] = nvz;
                    float *naxy = reinterpret_cast<float *>(&b.naxy[e]);
                    naxy[h] = nax; naxy[2u + h] = nay;
                    reinterpret_cast<float *>(&b.naz[e])[h] = naz;
                }
            };

            u32 kbuf = 0;
            const u32 c_begin = min(nchunks, (rbase == rbase0) ? it.z : 0u);
            const u32 c_end = c_begin + min(nchunks - c_begin, remaining);
            if (c_begin < c_end) {
                stage(c_begin, ws.buf[0]);
                cp_async_wait<0>();
                relayout(c_begin, ws.buf[0]);
            }
            __syncwarp();
            for (u32 c = c_begin; c < c_end; ++c, kbuf ^= 1u) {
                StagePacked &b = ws.buf[kbuf];
                const bool more = c + 1u < c_end;
                if (more) stage(c + 1u, ws.buf[kbuf ^ 1u]);  // in flight while this chunk is filtered
                const u32 m = min((u32)CH, total - c * CH);
                // ---- S1: one query per lane against every staged neighbour, two per packed instruction -----
                // Each lane keeps what passes as bit masks over the staged chunk (no warp vote, no store per test).
                u32 im = 0, nm = 0, fm = 0, bm = 0;
                const u32 npair = (m + 1u) >> 1;
                for (u32 u = 0; u < npair; ++u) {
                    const float4 xy = b.xy[u];
                    const float4 zb = b.zb[u];
                    const float2 dx = add2(make_float2(xy.x, xy.y), splat2(-p0.x));  // p_j - p_i
                    const float2 dy = add2(make_float2(xy.z, xy.w), splat2(-p0.y));
                    const float2 dz = add2(make_float2(zb.x, zb.y), splat2(-p0.z));
                    const float2 d2 = fma2(dz, dz, fma2(dy, dy, mul2(dx, dx)));
                    float2 tf = make_float2(0.0f, 0.0f);  // sign set: the test failed
                    if (USE_CAPSULE) {  // distance to the chord (w = 0 for radius queries)
                        const float2 dot = fma2(dz, splat2(wz), fma2(dy, splat2(wy), mul2(dx, splat2(wx))));
                        const float2 sc = make_float2(__saturatef(dot.x * inv_w2), __saturatef(dot.y * inv_w2));
                        const float2 ex = fma2(sc, splat2(-wx), dx), ey = fma2(sc, splat2(-wy), dy), ez = fma2(sc, splat2(-wz), dz);
                        const float2 e2 = fma2(ez, ez, fma2(ey, ey, mul2(ex, ex)));
                        tf = fma2(e2, splat2(-1.0f), splat2(rad2));  // < 0 <=> outside the capsule
                    } else if (t1_on) {
                        const float4 nxy = b.nxy[u], nzv = b.nzv[u], nvyz = b.nvyz[u];
                        const float2 gx = add2(make_float2(nxy.x, nxy.y), splat2(Mx));   // g0 = M_i - N_j
                        const float2 gy = add2(make_float2(nxy.z, nxy.w), splat2(My));
                        const float2 gz = add2(make_float2(nzv.x, nzv.y), splat2(Mz));
                        const float2 hx = add2(make_float2(nzv.z, nzv.w), splat2(MVx));  // g1 = MV_i - NV_j
                        const float2 hy = add2(make_float2(nvyz.x, nvyz.y), splat2(MVy));
                        const float2 hz = add2(make_float2(nvyz.z, nvyz.w), splat2(MVz));
                        const float2 g12c = fma2(hz, hz, fma2(hy, hy, fma2(hx, hx, splat2(1.0e-12f))));  // |g1|^2 (+ a floor)
                        const float2 dot = fma2(gz, hz, fma2(gy, hy, mul2(gx, hx)));
                        const float2 um = mul2(dot, make_float2(rcp_fast(g12c.x), rcp_fast(g12c.y)));  // -(minimum of the linear part, relative to tm)
                        const float2 sc = make_float2(__saturatef(fmaf(-um.x, inv_span, off_span)), __saturatef(fmaf(-um.y, inv_span, off_span)));
                        const float2 uc = fma2(sc, splat2(span), splat2(-D));
                        const float2 lx = fma2(hx, uc, gx), ly = fma2(hy, uc, gy), lz = fma2(hz, uc, gz);
                        const float2 l2 = fma2(lz, lz, fma2(ly, ly, mul2(lx, lx)));
                        const float4 naxy = b.naxy[u];
                        const float2 naz = b.naz[u];
                        const float2 qx = add2(make_float2(naxy.x, naxy.y), splat2(uax));  // Ua_i - a_j
                        const float2 qy = add2(make_float2(naxy.z, naxy.w), splat2(uay));
                        const float2 qz = add2(naz, splat2(uaz));
                        const float2 q2c = fma2(qz, qz, fma2(qy, qy, fma2(qx, qx, splat2(1.0e-12f))));  // |ca|^2 (+ the same floor)
                        const float2 qn = mul2(q2c, make_float2(rsqrt_fast(q2c.x), rsqrt_fast(q2c.y)));
                        const float2 L = fma2(splat2(kq), qn, add2(make_float2(zb.z, zb.w), splat2(A)));
                        const float2 L2 = mul2(L, L);
                        tf = fma2(l2, splat2(-1.0f), L2);  // < 0 <=> the linear part stays farther away than L
                    }
                    // the masks grow by one sign bit per test (the first test of the chunk ends up in the highest bit)
                    const float2 ti = add2(d2, splat2(-R2lo_l)), tn = add2(d2, splat2(-R2hi_n));
                    im = shift_in_sign(shift_in_sign(im, ti.x), ti.y);
                    nm = shift_in_sign(shift_in_sign(nm, tn.x), tn.y);
                    if (USE_CAPSULE || t1_on) fm = shift_in_sign(shift_in_sign(fm, tf.x), tf.y);
                    if (MODE == RCD_MODE_COMPUTE_NODE) {
                        const float2 tb2 = add2(d2, splat2(-dmaxB));
                        bm = shift_in_sign(shift_in_sign(bm, tb2.x), tb2.y);
                    }
                }
                // test k of the chunk (neighbour k) sits in bit nbits - 1 - k; the padding of an odd chunk is masked out
                const u32 nbits = 2u * npair;
                const u32 vm = (nbits >= 32u ? ~0u : ((1u << nbits) - 1u)) & ~((1u << (nbits - m)) - 1u);
                const u32 tm = (USE_CAPSULE || t1_on) ? ~fm : ~0u;
                im &= vm;
                const u32 um = nm & ~im & vm;   // inside the guard band of the radius: the exact stage decides (and counts)
                const u32 pm = ((tm & useT & (im | ~andI)) | (im & orI) | (bm & orB) | um) & vm;
                const u32 nc = (u32)__popc(im);
                const u32 cnt = (u32)__popc(pm);
                // ---- survivors -> pair queue (the warp's private block; a new one when this one is full) -------
                u32 off = cnt;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    u32 t = __shfl_up_sync(FULL_MASK, off, o);
                    if (lane >= (u32)o) off += t;
                }
                const u32 total_pairs = __shfl_sync(FULL_MASK, off, 31);
                off -= cnt;
                if (SLOW) {  // overflow pass: finish every survivor here
                    for (u32 rest = pm; rest; rest &= rest - 1u) {
                        const u32 bt = (u32)__ffs(rest) - 1u;
                        n_pot += narrow_entry_inline<MODE, COUNT_CAND>(
                            P, s | (((im >> bt) & 1u) ? QA_INR : 0u) | (((um >> bt) & 1u) ? QA_UND : 0u), b.pos[nbits - 1u - bt]);
                    }
                } else if (total_pairs) {
                    // room left in the warp's block; what does not fit goes to new blocks, taken with ONE atomic so that
                    // they are adjacent: the survivors of a chunk stay one contiguous run of the queue
                    const u32 room = qa_block == QA_NO_BLOCK ? 0u : (u32)QA_BLOCK - qa_used;
                    u32 nnew = 0, nb = 0;
                    if (total_pairs > room) {
                        nnew = (total_pairs - room + QA_BLOCK - 1) / QA_BLOCK;
                        if (lane == 0) nb = (u32)min(atomicAdd(&P.counters->n_qa_blocks, (unsigned long long)nnew), 0xf0000000ULL);
                        nb = __shfl_sync(FULL_MASK, nb, 0);
                        if (nb + nnew > P.qa_blocks_cap) {  // queue full: the overflow pass redoes the item from this chunk on
                            if (lane == 0) {
                                const unsigned long long k = atomicAdd(&P.counters->n_overflow, 1ULL);
                                if (k < P.ovf_cap)
                                    P.ovf[k] = make_uint4(tile, (u32)rbase, c, remaining - (c - c_begin));
                            }
                            for (u32 k = nb + lane; k < min(nb + nnew, P.qa_blocks_cap); k += 32) P.qa_fill[k] = 0u;  // taken, unused
                            qa_full = true;
                            stopped = true;
                            if (more) cp_async_wait<0>();
                            __syncwarp();
                            break;
                        }
                    }
                    uint2 *dst_cur = P.qa + ((size_t)(qa_block == QA_NO_BLOCK ? 0u : qa_block) * QA_BLOCK + qa_used);
                    uint2 *dst_new = P.qa + (size_t)nb * QA_BLOCK;
                    u32 at = off;
                    for (u32 rest = pm; __any_sync(FULL_MASK, rest != 0u); rest &= rest - 1u, ++at) {
                        if (rest) {
                            const u32 bt = (u32)__ffs(rest) - 1u;
                            const uint2 e = make_uint2(s | (((im >> bt) & 1u) ? QA_INR : 0u) | (((um >> bt) & 1u) ? QA_UND : 0u),
                                                       b.pos[nbits - 1u - bt]);
                            if (at < room) dst_cur[at] = e; else dst_new[at - room] = e;
                        }
                    }
                    if (nnew) {  // the old block and all new ones but the last are full now
                        const u32 rest = total_pairs - room - (nnew - 1u) * QA_BLOCK;  // 1 .. QA_BLOCK
                        if (lane == 0 && qa_block != QA_NO_BLOCK) P.qa_fill[qa_block] = QA_BLOCK;
                        for (u32 k = lane; k + 1u < nnew; k += 32) P.qa_fill[nb + k] = QA_BLOCK;
                        qa_block = nb + nnew - 1u;
                        qa_used = rest;
                    } else {
                        qa_used += total_pairs;
                    }
                }
                ncand += nc;  // (a chunk handed to the overflow pass is counted there)
                if (more) {
                    cp_async_wait<0>();
                    relayout(c + 1u, ws.buf[kbuf ^ 1u]);
                }
                __syncwarp();
            }
            remaining -= c_end - c_begin;
            n_chunks += c_end - c_begin;
        }
        // ---- end of tile ------------------------------------------------------------------------------
        // the filter counted the query itself (distance 0); only the compute-node index returns self (quirk Q8).
        // (the hit is seen by one of the tile's items, so the first one subtracts it and the partial counts are
        // combined with wrapping adds).  Objects without history owe every candidate twice in the
        // fused frame: once as detect_collisions, once as the fall-back of predict_collisions (:590-592).
        const bool self_seen = (p0.x - p0.x) == 0.0f && (p0.y - p0.y) == 0.0f && (p0.z - p0.z) == 0.0f;  // finite position
        if (!SLOW && MODE != RCD_MODE_COMPUTE_NODE && counts && first_item && self_seen) ncand -= 1u;
        if (FUSED && pattern == RCD_PAT_NO_HISTORY) ncand *= 2u;
        if (counts && P.cand_count && ncand) atomicAdd(&P.cand_count[P.sorted_slot[s]], ncand);
        long long csum = warp_sum((long long)(counts ? (int)ncand : 0));
        if (lane == 0 && csum) atomicAdd(&P.counters->n_candidates, (unsigned long long)csum);
    }
    if (!SLOW && lane == 0 && qa_block < P.qa_blocks_cap) P.qa_fill[qa_block] = qa_used;
    unsigned long long p = warp_sum((unsigned long long)n_pot);
    if (lane == 0 && p) atomicAdd(&P.counters->n_potential, p);
    if (lane == 0 && n_chunks) atomicAdd(&P.counters->n_tests, n_chunks * (unsigned long long)(CH * TQ));
}

// -------------------------------------------------------------------------------------------------
// k_narrow: QA -> Q3.  A warp takes 32 queued pairs at a time and works through them in phases with
// different lane assignments, so that every phase runs with (almost) full warps although the pairs
// carry different numbers of offsets.  Phase 1 runs on every batch.  Only some of a batch's pairs have
// offsets to look at, so those wait in a warp-private ring in shared memory, and phases 2-4 run on groups
// of 32 of them (on what is left once more after the warp's last batch):
//   1. lane = pair            : gather both objects; detect narrow phase (-> Q3); predict: the offsets whose
//                               samples can reach the safe distance -> (si, sj, offset mask) into the ring
//   group start, lane = pair  : gather the pair again (an L1 / L2 hit) and rebuild its coefficients -> shared memory
//   2. lane = (pair, offset)  : is the neighbour within 100 m of the predicted centre (:801-803)?  survivors ->
//                               item list
//   3. lane = surviving item  : the 10 samples of the offset (:322-342) in fp32 -> first sample inside
//                               safe + band and its squared distance -> shared memory
//   4. lane = pair            : merge over the offsets (max risk, earliest offset on ties, :848-865)
//                               -> 0 / RESOLVED | m | k << 8 / mask of the offsets fp64 must decide
// The ring holds 12 bytes per pair and the coefficients are rebuilt: keeping them in the ring instead would
// cost 6.4 KB more per warp, and the kernel would lose its 8 blocks per SM.
// sample_predict() above is the decision of phases 2-4 for one pair on one thread (queue-overflow fallback).
// -------------------------------------------------------------------------------------------------
constexpr int STAGE_THREADS = 128;
constexpr int STAGE_WARPS = STAGE_THREADS / 32;
constexpr int SC = 25;  // coefficients per pair (odd stride: conflict-free)
enum { SC_D = 0, SC_CV = 3, SC_CA = 6, SC_RV = 9, SC_RA = 12, SC_UV = 15, SC_UA = 18, SC_SAFEB2 = 21, SC_SAFEIN2 = 22,
       SC_INVSAFE = 23 };
constexpr u32 NARROW_RING = 64;  // pending predict pairs of a warp: fewer than 32 left over + one batch
struct SampleShared {
    float coef[32][SC];                        // of the group's pairs
    float part[32][PREDICT_OFFSETS];           // offset-dependent part of the risk of a certain hit (< 0: undecided in
                                               // fp32), with the index of the first sample in the 4 lowest mantissa bits
    u32 hit_mask[32];                          // offsets with a sample within safe + band
    QEntry ring[NARROW_RING];                  // predict pairs waiting for phases 2-4: {si, sj, offset mask}
    unsigned short items[64];                  // pair of the group | offset << 5
};
constexpr int QA_BATCHES_PER_BLOCK = QA_BLOCK / 32;
constexpr u32 SAMPLE_ITEMS = 32u;  // items per pass of the sample phase (two lanes per item, 5 samples each, measured slower)

__device__ __forceinline__ float sqrt_approx(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// Q3 holds three kinds of entries, kept apart so that the warps of k_exact run one code path: detect entries grow
// from the front; predict entries fill [q3_split, qcap) (the predict modes; other modes: q3_split = qcap), the RESOLVED
// ones (one fp64 evaluation each) from q3_split on, those whose offsets fp64 has to scan in the last quarter of the region.
__device__ __forceinline__ u32 q3_unresolved_begin(const PairParams &P) { return P.qcap - (P.qcap - P.q3_split) / 4u; }
__device__ __forceinline__ bool push_detect(const PairParams &P, bool flag, u32 si, u32 sj, u32 word) {
    return global_push(P.q3, P.q3_split, &P.counters->n_q3, flag, si, sj, word);
}
__device__ __forceinline__ bool push_predict(const PairParams &P, bool flag, u32 si, u32 sj, u32 word) {
    const u32 ub = q3_unresolved_begin(P);
    const bool res = (word & RESOLVED) != 0;
    const bool ok_r = global_push(P.q3 + P.q3_split, ub - P.q3_split, &P.counters->n_q3p, flag && res, si, sj, word);
    const bool ok_u = global_push(P.q3 + ub, P.qcap - ub, &P.counters->n_q3u, flag && !res, si, sj, word);
    return ok_r && ok_u;
}

template <int MODE, bool COUNT_CAND>
#ifndef RCD_NARROW_MIN_BLOCKS
#define RCD_NARROW_MIN_BLOCKS 8
#endif
__global__ void __launch_bounds__(STAGE_THREADS, RCD_NARROW_MIN_BLOCKS) k_narrow(PairParams P) {
    __shared__ SampleShared shared[STAGE_WARPS];
    SampleShared &sh = shared[threadIdx.x >> 5];
    constexpr bool PRED = is_predict(MODE);
    constexpr bool FUSED = MODE == MODE_PREDICT_WITH_DETECT;
    const u32 lane = threadIdx.x & 31u;
    const unsigned long long nblocks = min(P.counters->n_qa_blocks, (unsigned long long)P.qa_blocks_cap);
    const unsigned long long nbatch = nblocks * QA_BATCHES_PER_BLOCK;
    const unsigned long long wstride = (unsigned long long)gridDim.x * STAGE_WARPS;
    const float R2 = PREDICT_RADIUS * PREDICT_RADIUS;
    u32 n_exact = 0, n_pot = 0;
    u32 head = 0, n_pend = 0;  // (warp-uniform) the pending pairs are sh.ring[(head + k) % NARROW_RING], k < n_pend
    // the queue entry of a batch (loaded one batch ahead of its use); x = 0xffffffff: none
    auto fetch = [&](unsigned long long batch) {
        uint2 e = make_uint2(0xffffffffu, 0u);
        if (batch < nbatch) {
            const u32 blk = (u32)(batch / QA_BATCHES_PER_BLOCK), within = (u32)(batch % QA_BATCHES_PER_BLOCK) * 32u;
            if (within + lane < P.qa_fill[blk]) e = __ldcs(P.qa + (size_t)blk * QA_BLOCK + within + lane);
        }
        return e;
    };

    // ---- phases 2-4 on the first ng (<= 32) pending pairs: lane (and pr below) = position in the group ------
    auto run_group = [&](u32 ng) {
        u32 si = 0, sj = 0, mask = 0;
        if (lane < ng) {
            const QEntry q = sh.ring[(head + lane) % NARROW_RING];
            si = q.si; sj = q.sj; mask = q.mask;
            const float4 a0 = P.P0[si], a1 = P.P1[si], a2 = P.P2[si];
            const float4 b0 = P.P0[sj], b1 = P.P1[sj], b2 = P.P2[sj];
            const PredictCoef c = predict_coef(a0, a1, a2, b0, b1, b2, meta_pattern(__float_as_uint(a2.w)));
            float *o = sh.coef[lane];
            o[SC_D] = c.dx; o[SC_D + 1] = c.dy; o[SC_D + 2] = c.dz;
            o[SC_CV] = c.cvx; o[SC_CV + 1] = c.cvy; o[SC_CV + 2] = c.cvz;
            o[SC_CA] = c.cax; o[SC_CA + 1] = c.cay; o[SC_CA + 2] = c.caz;
            o[SC_RV] = c.rvx; o[SC_RV + 1] = c.rvy; o[SC_RV + 2] = c.rvz;
            o[SC_RA] = a2.x - b2.x; o[SC_RA + 1] = a2.y - b2.y; o[SC_RA + 2] = a2.z - b2.z;
            o[SC_UV] = c.uvx; o[SC_UV + 1] = c.uvy; o[SC_UV + 2] = c.uvz;
            o[SC_UA] = c.uax; o[SC_UA + 1] = c.uay; o[SC_UA + 2] = c.uaz;
            o[SC_SAFEB2] = c.safe_b2;
            const float safe_in = fmaxf(c.safe - (c.safe_b - c.safe), 0.0f);  // safe minus the guard band
            o[SC_SAFEIN2] = safe_in * safe_in;
            o[SC_INVSAFE] = rcp_fast(c.safe);  // (feeds the fp32 merge key only: ~1e-7 relative)
        }
        sh.hit_mask[lane] = 0;
        const u32 cnt = (u32)__popc(mask);
        u32 off = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            u32 t = __shfl_up_sync(FULL_MASK, off, o);
            if (lane >= (u32)o) off += t;
        }
        const u32 total = __shfl_sync(FULL_MASK, off, 31);
        off -= cnt;
        __syncwarp();

        // ---- 3. lane = item: the 10 samples of one offset of one pair ---------------------------------
        u32 n_items = 0;  // warp-uniform length of the item list
        auto run_samples = [&](u32 take) {
            if (lane < take) {
                const u32 it = sh.items[n_items - take + lane];
                const u32 pr = it & 31u, m = it >> 5;
                const float *c = sh.coef[pr];
                const float t = 0.5f * (float)m, h = 0.5f * t * t;
                const float gx = c[SC_CV] * t + c[SC_CA] * h - c[SC_D], gy = c[SC_CV + 1] * t + c[SC_CA + 1] * h - c[SC_D + 1],
                            gz = c[SC_CV + 2] * t + c[SC_CA + 2] * h - c[SC_D + 2];
                const float rvx = c[SC_RV], rvy = c[SC_RV + 1], rvz = c[SC_RV + 2];
                const float rax = c[SC_RA], ray = c[SC_RA + 1], raz = c[SC_RA + 2];
                const float safe_b2 = c[SC_SAFEB2];
                int first = -1;
                float r2first = 0.0f;
#pragma unroll
                for (int kk = PREDICT_STEPS - 1; kk >= 0; --kk) {  // descending: the last assignment is the first sample
                    const float tau = 0.1f * (float)kk, hh = 0.5f * tau * tau;
                    const float rx = gx + rvx * tau + rax * hh, ry = gy + rvy * tau + ray * hh, rz = gz + rvz * tau + raz * hh;
                    const float r2 = rx * rx + ry * ry + rz * rz;
                    if (r2 <= safe_b2) { first = kk; r2first = r2; }
                }
                if (first >= 0) {
                    // a first sample inside the guard band: fp64 decides (-1).  Otherwise a certain hit at sample `first`,
                    // every earlier sample certainly outside: the parts of the risk that differ between the offsets of
                    // a pair (collision_detection.py:371-374) decide the merge (fp32 error of `part` ~1e-5)
                    float part = -1.0f;
                    if (r2first <= c[SC_SAFEIN2])
                        part = 0.3f * (1.0f - sqrt_approx(r2first) * c[SC_INVSAFE]) + 0.3f * (1.0f - 0.01f * (float)first);
                    sh.part[pr][m] = __uint_as_float((__float_as_uint(part) & ~15u) | (u32)first);  // (15 ulp << 1e-4)
                    atomicOr(&sh.hit_mask[pr], 1u << m);
                }
            }
            n_items -= take;
            __syncwarp();
        };

        // ---- 2. lane = (pair, offset) ---------------------------------------------------------------------
        for (u32 fbase = 0; fbase < total; fbase += 32) {
            const u32 f = fbase + lane;
            u32 pr = 0;
#pragma unroll
            for (int step = 16; step > 0; step >>= 1) {
                const u32 cand = pr + step;
                const u32 v = __shfl_sync(FULL_MASK, off, cand & 31u);
                if (cand < 32u && v <= f) pr = cand;
            }
            const u32 pr_off = __shfl_sync(FULL_MASK, off, pr);
            const u32 pr_mask = __shfl_sync(FULL_MASK, mask, pr);
            bool pass = false;
            u32 m = 0;
            if (f < total) {
                m = __fns(pr_mask, 0u, (int)(f - pr_off) + 1);  // (f - pr_off)-th offset of the pair's mask
                pass = true;
                if (!COUNT_CAND) {  // with COUNT_CAND both tests were already taken in phase 1
                    const float *c = sh.coef[pr];
                    const float t = 0.5f * (float)m, h = 0.5f * t * t;
                    const float dx = c[SC_D], dy = c[SC_D + 1], dz = c[SC_D + 2];
                    // (that the samples of this offset can reach the safe distance was established in phase 1)
                    {   // neighbour within 100 m of the predicted centre?
                        const float ux = c[SC_UV] * t + c[SC_UA] * h - dx, uy = c[SC_UV + 1] * t + c[SC_UA + 1] * h - dy,
                                    uz = c[SC_UV + 2] * t + c[SC_UA + 2] * h - dz;
                        const float c2 = ux * ux + uy * uy + uz * uz;
                        pass = c2 <= R2 * (1.0f + BAND_R2);
                        if (pass && c2 >= R2 * (1.0f - BAND_R2)) {
                            ++n_exact;
                            const QEntry q = sh.ring[(head + pr) % NARROW_RING];
                            pass = exact_predict_radius(P, q.si, q.sj, meta_pattern(__float_as_uint(P.P2[q.si].w)), (int)m);
                        }
                    }
                }
            }
            const u32 bal = __ballot_sync(FULL_MASK, pass);
            if (bal) {
                if (pass) sh.items[n_items + __popc(bal & lanemask_lt())] = (unsigned short)(pr | (m << 5));
                n_items += __popc(bal);
                __syncwarp();
                while (n_items >= SAMPLE_ITEMS) run_samples(SAMPLE_ITEMS);
            }
        }
        while (n_items) run_samples(min(n_items, SAMPLE_ITEMS));
        __syncwarp();

        // ---- 4. lane = pair: merge over the offsets ------------------------------------------------------
        const u32 maybe_mask = sh.hit_mask[lane];  // the other offsets have no sample within safe + band: certainly no hit
        bool doubt = false;      // some decisive sample lies inside the band
        float best = -1.0f, second = -1.0f;
        int best_m = -1;
        u32 rest = maybe_mask;
        while (rest) {
            const int m = __ffs(rest) - 1;
            rest &= rest - 1;
            const float part = sh.part[lane][m];
            doubt = doubt || part < 0.0f;
            if (part > best) { second = best; best = part; best_m = m; }
            else if (part > second) second = part;
        }
        u32 word = 0;
        if (maybe_mask) {
            // a runner-up within 1e-4 or any sample in the band: fp64 decides
            word = (doubt || best_m < 0 || best - second <= 1.0e-4f)
                       ? maybe_mask : (RESOLVED | (u32)best_m | ((__float_as_uint(best) & 15u) << 8));
        }
        if (!push_predict(P, word != 0, si, sj, word))
            finish_entry_inline<RCD_MODE_PREDICT>(P, si, sj, word);
        __syncwarp();  // the next group overwrites this warp's shared memory (and the next batch these ring slots)
    };

    unsigned long long batch = (unsigned long long)blockIdx.x * STAGE_WARPS + (threadIdx.x >> 5);
    uint2 e_next = fetch(batch);
    for (;; batch += wstride) {
        const bool more = batch < nbatch;  // false: one more pass, for the pairs still in the ring
        const uint2 e = e_next;
        if (more) e_next = fetch(batch + wstride);
        // (no entry in the batch: the warp that owned the block stopped before it)
        if (more && __any_sync(FULL_MASK, e.x != 0xffffffffu)) {
            // ---- 1. lane = pair ------------------------------------------------------------------------
            u32 si = 0, sj = 0, mask = 0, det_word = 0;
            bool det_keep = false;
            if (e.x != 0xffffffffu) {
                si = e.x & QA_SI_MASK;
                sj = e.y;
                const bool inr = (e.x & QA_INR) != 0, und = (e.x & QA_UND) != 0;
                if (si != sj || MODE == RCD_MODE_COMPUTE_NODE) {  // _spatial_filtering strips self (:224-225)
                    const float4 a0 = P.P0[si], a1 = P.P1[si], a2 = P.P2[si];
                    const float4 b0 = P.P0[sj], b1 = P.P1[sj], b2 = P.P2[sj];
                    if (MODE == RCD_MODE_DETECT) {
                        det_keep = und || narrow_detect(a0, a1, a2, b0, b1, b2, P.T);
                        det_word = und ? RADIUS_UNDECIDED : 0u;
                    } else if (MODE == RCD_MODE_COMPUTE_NODE) {
                        det_keep = narrow_compute_node(P, a0, a1, a2, b0, b1, b2, si == sj, und);
                        det_word = und ? RADIUS_UNDECIDED : 0u;
                    } else {
                        const u32 pat = meta_pattern(__float_as_uint(a2.w));
                        const bool nohist = pat == RCD_PAT_NO_HISTORY;
                        if ((nohist || FUSED) && (inr || und)) {  // detect_collisions(100.0, 10.0): the defaults (:592)
                            const bool twice = nohist && FUSED;
                            det_keep = und || narrow_detect(a0, a1, a2, b0, b1, b2, 10.0f);
                            det_word = (und ? RADIUS_UNDECIDED : 0u) | (twice ? ENTRY_TWICE : 0u);
                        }
                        if (!nohist) {
                            if (COUNT_CAND) {
                                mask = predict_mask<true>(P, a0, a1, a2, b0, b1, b2, si, sj, pat, n_exact);
                            } else {
                                // the offsets whose 10 samples can come within the safe distance at all (offset_may_hit): the
                                // samples leave the offset state g(t_m) = centre_i(t_m) - predicted_j(t_m) along rv tau (+ at most
                                // 0.405 |ra|), tau in [0, 0.9] -- closest point of that segment to the origin, two offsets per
                                // packed instruction
                                const PredictCoef c = predict_coef(a0, a1, a2, b0, b1, b2, pat);
                                const float nir = -c.inv_rv2 * (1.0f / 0.9f);
                                const float r9x = 0.9f * c.rvx, r9y = 0.9f * c.rvy, r9z = 0.9f * c.rvz;
                                u32 fmask = 0;
#pragma unroll
                                for (int m = 0; m < PREDICT_OFFSETS; m += 2) {
                                    const float2 t2 = make_float2(0.5f * (float)m, 0.5f * (float)(m + 1));
                                    const float2 h2 = make_float2(0.125f * (float)(m * m), 0.125f * (float)((m + 1) * (m + 1)));
                                    const float2 gx = fma2(splat2(c.cvx), t2, fma2(splat2(c.cax), h2, splat2(-c.dx)));
                                    const float2 gy = fma2(splat2(c.cvy), t2, fma2(splat2(c.cay), h2, splat2(-c.dy)));
                                    const float2 gz = fma2(splat2(c.cvz), t2, fma2(splat2(c.caz), h2, splat2(-c.dz)));
                                    const float2 dot = fma2(gz, splat2(c.rvz), fma2(gy, splat2(c.rvy), mul2(gx, splat2(c.rvx))));
                                    const float2 sc = make_float2(__saturatef(dot.x * nir), __saturatef(dot.y * nir));  // tau / 0.9
                                    const float2 ex = fma2(splat2(r9x), sc, gx), ey = fma2(splat2(r9y), sc, gy), ez = fma2(splat2(r9z), sc, gz);
                                    const float2 e2 = fma2(ez, ez, fma2(ey, ey, mul2(ex, ex)));
                                    const float2 tf = fma2(e2, splat2(-1.0f), splat2(c.lim2));  // < 0 <=> out of reach
                                    fmask = shift_in_sign(shift_in_sign(fmask, tf.x), tf.y);
                                }
                                // offset m failed <=> bit (PREDICT_OFFSETS - 1 - m) of fmask
                                mask = (~__brev(fmask) >> (32 - PREDICT_OFFSETS)) & ((1u << PREDICT_OFFSETS) - 1u);
                            }
                        }
                    }
                }
            }
            if (!push_detect(P, det_keep, si, sj, det_word))
                n_pot += finish_entry_inline<MODE>(P, si, sj, det_word);  // queue full: decide here
            if (PRED) {  // the pairs with offsets to look at join the ring
                mask &= (1u << PREDICT_OFFSETS) - 1u;
                const u32 bal = __ballot_sync(FULL_MASK, mask != 0);
                if (mask) sh.ring[(head + n_pend + (u32)__popc(bal & lanemask_lt())) % NARROW_RING] = QEntry{si, sj, mask};
                n_pend += (u32)__popc(bal);
            }
        }
        if (PRED && (n_pend >= 32u || (!more && n_pend != 0u))) {
            __syncwarp();  // the ring entries are written
            const u32 ng = min(n_pend, 32u);
            run_group(ng);
            head = (head + ng) % NARROW_RING;
            n_pend -= ng;
        }
        if (!more) break;
    }
    unsigned long long ex = warp_sum((unsigned long long)n_exact);
    unsigned long long pt = warp_sum((unsigned long long)n_pot);
    if (lane == 0) {
        if (ex) atomicAdd(&P.counters->n_exact, ex);
        if (pt) atomicAdd(&P.counters->n_potential, pt);
    }
}

// k_exact: one queued pair per thread, decided in fp64; the output cursor is claimed once per warp.
// The three kinds of Q3 entries are mapped to different warps (a warp that mixes one offset scan into 31 single
// evaluations runs at the pace of the scan: 17 of 32 threads active per instruction before the split, 30 after).
// SEG 0: every entry (radius-query modes); the predict modes run two launches: SEG 2 takes the RESOLVED predict entries
// (one inlined fp64 evaluation each), SEG 1 the detect entries and the predict entries whose offsets fp64 has to scan.
#ifndef RCD_EXACT_MIN_BLOCKS
#define RCD_EXACT_MIN_BLOCKS 4
#endif
#ifndef RCD_EXACT_RES_MIN_BLOCKS
#define RCD_EXACT_RES_MIN_BLOCKS 4
#endif
template <int MODE, int SEG>
__global__ void __launch_bounds__(STAGE_THREADS, SEG == 2 ? RCD_EXACT_RES_MIN_BLOCKS : RCD_EXACT_MIN_BLOCKS) k_exact(PairParams P) {
    const u32 ub = q3_unresolved_begin(P);
    const unsigned long long nd = SEG == 2 ? 0ULL : min(P.counters->n_q3, (unsigned long long)P.q3_split);
    const unsigned long long np = SEG == 1 ? 0ULL : min(P.counters->n_q3p, (unsigned long long)(ub - P.q3_split));
    const unsigned long long nu = SEG == 2 ? 0ULL : min(P.counters->n_q3u, (unsigned long long)(P.qcap - ub));
    const unsigned long long nd_pad = (nd + 31ULL) & ~31ULL, np_end = nd_pad + np, np_pad = (np_end + 31ULL) & ~31ULL;
    const unsigned long long n = np_pad + nu;
    const unsigned long long stride = (unsigned long long)gridDim.x * STAGE_THREADS;
    const unsigned long long rounds = (n + stride - 1) / stride;
    const u32 lane = threadIdx.x & 31u;
    u32 n_pot = 0, n_exact = 0, n_high = 0, n_prio[4] = {0, 0, 0, 0};
    for (unsigned long long r = 0; r < rounds; ++r) {  // uniform trip count: the emission is warp-wide
        const unsigned long long k = r * stride + (unsigned long long)blockIdx.x * STAGE_THREADS + threadIdx.x;
        EmitRec e = no_rec();
        if (k < nd || (k >= nd_pad && k < np_end) || (k >= np_pad && k < n)) {
            const QEntry q = k < nd ? P.q3[k] : k < np_end ? P.q3[P.q3_split + (k - nd_pad)] : P.q3[ub + (k - np_pad)];
            if (SEG == 2)
                e = exact_predict_resolved_body(P, q.si, q.sj, meta_pattern(__float_as_uint(P.P2[q.si].w)), (int)(q.mask & 31u),
                                                (int)((q.mask >> 8) & 15u));
            else
                e = exact_entry<MODE>(P, q.si, q.sj, q.mask);
            n_pot += e.potential;
            n_exact += (is_predict(MODE) && (q.mask & 0xfffffu) && !(q.mask & RESOLVED)) ? (u32)__popc(q.mask & 0xfffffu) : 1u;
        }
        const u32 ballot = __ballot_sync(FULL_MASK, e.hit);
        if (ballot) {
            unsigned long long base = 0;
            const u32 leader = __ffs(ballot) - 1;
            if (lane == leader) base = atomicAdd(&P.counters->n_pairs, (unsigned long long)__popc(ballot));
            base = __shfl_sync(FULL_MASK, base, leader);
            if (e.hit) {
                store_pair(P, base + __popc(ballot & lanemask_lt()), e);
                n_high += e.high ? 1u : 0u;
                if (e.prio >= 0) n_prio[e.prio] += 1u;
            }
        }
        if (MODE == MODE_PREDICT_WITH_DETECT && SEG != 2) {  // second copy of the records that are owed twice
            const bool again = e.hit && e.twice;
            const u32 b2 = __ballot_sync(FULL_MASK, again);
            if (b2) {
                unsigned long long base = 0;
                const u32 leader = __ffs(b2) - 1;
                if (lane == leader) base = atomicAdd(&P.counters->n_pairs, (unsigned long long)__popc(b2));
                base = __shfl_sync(FULL_MASK, base, leader);
                if (again) {
                    store_pair(P, base + __popc(b2 & lanemask_lt()), e);
                    n_high += e.high ? 1u : 0u;
                    if (e.prio >= 0) n_prio[e.prio] += 1u;
                }
            }
        }
    }
    unsigned long long v[7] = {n_pot, n_exact, n_high, n_prio[0], n_prio[1], n_prio[2], n_prio[3]};
#pragma unroll
    for (int q = 0; q < 7; ++q) v[q] = warp_sum(v[q]);
    if (lane == 0) {
        if (v[0]) atomicAdd(&P.counters->n_potential, v[0]);
        if (v[1]) atomicAdd(&P.counters->n_exact, v[1]);
        if (v[2]) atomicAdd(&P.counters->n_high_risk, v[2]);
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (v[3 + q]) atomicAdd(&P.counters->n_alerts[q], v[3 + q]);
    }
}

// -------------------------------------------------------------------------------------------------
// Radius query for explicit points: SpatialIndex.get_nearby_vehicles (spatial_index.py:229-271)
// and compute_node.SpatialIndex.query_nearby (compute_node.py:98-119).  One warp per query;
// hits are appended as (query, upload slot) pairs, grouped and ordered on the host.
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
k_query_radius(u32 nq, const float *__restrict__ qx, const float *__restrict__ qy, const float *__restrict__ qz,
               float radius, GridParams g, u32 n, const float4 *__restrict__ P0, const u32 *__restrict__ cell_begin,
               const u32 *__restrict__ sorted_slot, uint2 *__restrict__ hits, unsigned long long cap,
               Counters *counters) {
    const u32 lane = threadIdx.x & 31u;
    const u32 qi = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (qi >= nq) return;
    const float x = qx[qi], y = qy[qi], z = qz[qi];
    const float R2 = radius * radius;
    // cells under the bounding box of the ball (cell_coord is monotone and clamps: objects outside the
    // grid sit in its border cells, a query point outside the grid reaches them through the same clamp)
    const float r = radius * (1.0f + 1.0e-5f) + 1.0e-3f;
    const int x0 = cell_coord(x - r - (0.05f + 4.0e-7f * fabsf(x)), g.ox, g.inv_cell, g.nx);
    const int x1 = cell_coord(x + r + (0.05f + 4.0e-7f * fabsf(x)), g.ox, g.inv_cell, g.nx);
    const int y0 = cell_coord(y - r - (0.05f + 4.0e-7f * fabsf(y)), g.oy, g.inv_cell, g.ny);
    const int y1 = cell_coord(y + r + (0.05f + 4.0e-7f * fabsf(y)), g.oy, g.inv_cell, g.ny);
    const int z0 = cell_coord(z - r - (0.05f + 4.0e-7f * fabsf(z)), g.oz, g.inv_cell_z, g.nz);
    const int z1 = cell_coord(z + r + (0.05f + 4.0e-7f * fabsf(z)), g.oz, g.inv_cell_z, g.nz);
    for (int zz = z0; zz <= z1; ++zz)
        for (int yy = y0; yy <= y1; ++yy) {
            const u32 c0 = (u32)((zz * g.ny + yy) * g.nx + x0), c1 = c0 + (u32)(x1 - x0);
            const u32 first = cell_begin[c0], last = cell_begin[c1 + 1u];
            for (u32 s = first + lane; s < last; s += 32) {
                float4 b = P0[s];
                float dx = b.x - x, dy = b.y - y, dz = b.z - z;
                float d2 = dx * dx + dy * dy + dz * dz;
                bool in = d2 <= R2 * (1.0f - BAND_R2);
                if (!in && d2 <= R2 * (1.0f + BAND_R2)) in = within_radius_d(x, y, z, b.x, b.y, b.z, (double)radius);
                if (in) {
                    unsigned long long pos = atomicAdd(&counters->n_query_hits, 1ULL);
                    if (pos < cap) hits[pos] = make_uint2(qi, sorted_slot[s]);
                }
            }
        }
}

// rcd_pair (48 bytes) -> rcd_pair_compact (32 bytes), before the records cross the bus
__global__ void __launch_bounds__(256)
k_compact_pairs(const rcd_pair *__restrict__ in, unsigned long long n_max, const unsigned long long *__restrict__ n_dev,
                rcd_pair_compact *__restrict__ out) {
    const unsigned long long n = min(*n_dev, n_max);
    for (unsigned long long k = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; k < n;
         k += (unsigned long long)gridDim.x * blockDim.x) {
        const rcd_pair p = in[k];
        rcd_pair_compact c;
        c.i = p.i; c.j = p.j; c.ttc = p.ttc; c.distance = p.distance; c.rel_speed = p.rel_speed; c.risk = p.risk;
        c.t_closest = p.t_closest; c.priority = p.priority; c.offset = p.offset; c.predicted = p.predicted; c.reserved = 0;
        const uint4 *src = reinterpret_cast<const uint4 *>(&c);
        uint4 *dst = reinterpret_cast<uint4 *>(out + k);
        dst[0] = src[0]; dst[1] = src[1];
    }
}

// -------------------------------------------------------------------------------------------------
// The per-pair helpers for explicit pairs (rcd_pair_exact / rcd_risk_assessment): one thread per pair,
// the same fp64 device functions the frame kernels decide with.
// -------------------------------------------------------------------------------------------------
__device__ __forceinline__ ObjD widen_object(const rcd_object &o) {
    ObjD d;
    d.px = o.px; d.py = o.py; d.pz = o.pz; d.vx = o.vx; d.vy = o.vy; d.vz = o.vz;
    d.ax = o.ax; d.ay = o.ay; d.az = o.az; d.size = o.size; d.heading = o.heading;
    d.type = o.type;
    return d;
}
__global__ void __launch_bounds__(128)
k_pair_exact(u32 n, const rcd_object *__restrict__ a, const rcd_object *__restrict__ b, int steps, double time_step,
             rcd_pair_exact_result *__restrict__ out) {
    const u32 k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const ObjD A = widen_object(a[k]), B = widen_object(b[k]);
    const double safe = safe_d(A.size, B.size);
    const HitD h = precise_hit_d(A.px, A.py, A.pz, B.px, B.py, B.pz, A, B, safe, steps, time_step);
    rcd_pair_exact_result r;
    r.hit = h.k >= 0 ? 1 : 0;
    r.step = h.k;
    r.collision_time = h.k >= 0 ? dmul((double)h.k, time_step) : 0.0;
    r.distance = h.dist;
    r.safe_distance = safe;
    r.relative_speed = mag3_d(dsub(A.vx, B.vx), dsub(A.vy, B.vy), dsub(A.vz, B.vz));
    r.cx = h.mx; r.cy = h.my; r.cz = h.mz;
    r.risk = h.k >= 0 ? risk_level_d(A.heading, B.heading, A.type, B.type, r.collision_time, h.dist, safe, r.relative_speed) : 0.0;
    out[k] = r;
}
__global__ void __launch_bounds__(128) k_risk_assessment(u32 n, const double *__restrict__ in, double *__restrict__ out) {
    const u32 k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const double *v = in + 7 * (size_t)k;
    out[k] = risk_level_d(v[0], v[1], v[2] != 0.0 ? 1u : 0u, 1u, v[3], v[4], v[5], v[6]);
}

// -------------------------------------------------------------------------------------------------
// Trajectory pattern classifier (collision_detection.py:623-711), one thread per object, fp64,
// streaming over the (already time-ordered) samples in the reference's summation order.
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
k_classify_patterns(u32 n, u32 stride, const double *__restrict__ samples /* [n][stride][4] */,
                    const u32 *__restrict__ count, uint8_t *__restrict__ out) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u32 cnt = min(count[i], stride);
    if (cnt < 2) { out[i] = RCD_PAT_NO_HISTORY; return; }
    const double *h = samples + (size_t)i * stride * 4;
    double svx = 0, svy = 0, svz = 0, sax = 0, say = 0, saz = 0;
    u32 nv = 0, na = 0;
    double pvx = 0, pvy = 0, pvz = 0, pvt = 0;
    double lx = h[0], ly = h[1], lz = h[2], lt = h[3];
    for (u32 k = 1; k < cnt; ++k) {
        double x = h[4 * k], y = h[4 * k + 1], z = h[4 * k + 2], t = h[4 * k + 3];
        double dt = dsub(t, lt);
        if (dt > 0) {
            double vx = __ddiv_rn(dsub(x, lx), dt), vy = __ddiv_rn(dsub(y, ly), dt), vz = __ddiv_rn(dsub(z, lz), dt);
            if (nv > 0) {
                double dtv = dsub(t, pvt);
                if (dtv > 0) {
                    sax = dadd(sax, __ddiv_rn(dsub(vx, pvx), dtv));
                    say = dadd(say, __ddiv_rn(dsub(vy, pvy), dtv));
                    saz = dadd(saz, __ddiv_rn(dsub(vz, pvz), dtv));
                    ++na;
                }
            }
            svx = dadd(svx, vx); svy = dadd(svy, vy); svz = dadd(svz, vz);
            ++nv;
            pvx = vx; pvy = vy; pvz = vz; pvt = t;
        }
        lx = x; ly = y; lz = z; lt = t;
    }
    if (nv == 0) { out[i] = RCD_PAT_STATIONARY; return; }
    svx = __ddiv_rn(svx, (double)nv); svy = __ddiv_rn(svy, (double)nv); svz = __ddiv_rn(svz, (double)nv);
    if (na) { sax = __ddiv_rn(sax, (double)na); say = __ddiv_rn(say, (double)na); saz = __ddiv_rn(saz, (double)na); }
    double speed = mag3_d(svx, svy, svz), accel = mag3_d(sax, say, saz);
    out[i] = speed < 0.1 ? RCD_PAT_STATIONARY : (accel < 0.1 ? RCD_PAT_CONSTANT_VELOCITY : RCD_PAT_ACCELERATING);
}

// -------------------------------------------------------------------------------------------------
// Device-resident trajectory rings: hist[k * cap + slot] = k-th ring entry of the object in `slot`
// (sample-major, so threads of a warp touch consecutive 32-byte samples), count[slot] = samples ever
// appended.  Same fp64 arithmetic and summation order as k_classify_patterns.
// -------------------------------------------------------------------------------------------------
struct Sample64 {
    double x, y, z, t;
};

__global__ void __launch_bounds__(256)
k_history_append(u32 n, const u32 *__restrict__ slot, const double *__restrict__ x, const double *__restrict__ y,
                 const double *__restrict__ z, const double *__restrict__ t, Sample64 *__restrict__ hist,
                 u32 *__restrict__ count, u32 cap, u32 H) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u32 s = slot ? slot[i] : i;
    if (s >= cap) return;
    const u32 c = count[s];
    Sample64 v;
    v.x = x[i]; v.y = y[i]; v.z = z[i]; v.t = t[i];
    hist[(size_t)(c % H) * cap + s] = v;
    count[s] = c + 1;
}

__global__ void __launch_bounds__(256) k_history_reset(u32 n, const u32 *__restrict__ slot, u32 *__restrict__ count, u32 cap) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && slot[i] < cap) count[slot[i]] = 0;
}

__global__ void __launch_bounds__(128) k_history_move(u32 dst, u32 src, Sample64 *__restrict__ hist, u32 *__restrict__ count, u32 cap, u32 H) {
    for (u32 k = threadIdx.x; k < H; k += blockDim.x) hist[(size_t)k * cap + dst] = hist[(size_t)k * cap + src];
    if (threadIdx.x == 0) count[dst] = count[src];
}

__global__ void __launch_bounds__(128)
k_history_classify(u32 n, const Sample64 *__restrict__ hist, const u32 *__restrict__ count, u32 cap, u32 H,
                   uint8_t *__restrict__ out) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u32 total = count[i];
    const u32 cnt = min(total, H);
    if (cnt < 2) { out[i] = RCD_PAT_NO_HISTORY; return; }
    const u32 first = total - cnt;  // ring position of the oldest kept sample is first % H
    double svx = 0, svy = 0, svz = 0, sax = 0, say = 0, saz = 0;
    u32 nv = 0, na = 0;
    double pvx = 0, pvy = 0, pvz = 0, pvt = 0;
    Sample64 last = hist[(size_t)(first % H) * cap + i];
    for (u32 k = 1; k < cnt; ++k) {
        const Sample64 cur = hist[(size_t)((first + k) % H) * cap + i];
        const double dt = dsub(cur.t, last.t);
        if (dt > 0) {
            const double vx = __ddiv_rn(dsub(cur.x, last.x), dt), vy = __ddiv_rn(dsub(cur.y, last.y), dt),
                         vz = __ddiv_rn(dsub(cur.z, last.z), dt);
            if (nv > 0) {
                const double dtv = dsub(cur.t, pvt);
                if (dtv > 0) {
                    sax = dadd(sax, __ddiv_rn(dsub(vx, pvx), dtv));
                    say = dadd(say, __ddiv_rn(dsub(vy, pvy), dtv));
                    saz = dadd(saz, __ddiv_rn(dsub(vz, pvz), dtv));
                    ++na;
                }
            }
            svx = dadd(svx, vx); svy = dadd(svy, vy); svz = dadd(svz, vz);
            ++nv;
            pvx = vx; pvy = vy; pvz = vz; pvt = cur.t;
        }
        last = cur;
    }
    if (nv == 0) { out[i] = RCD_PAT_STATIONARY; return; }
    svx = __ddiv_rn(svx, (double)nv); svy = __ddiv_rn(svy, (double)nv); svz = __ddiv_rn(svz, (double)nv);
    if (na) { sax = __ddiv_rn(sax, (double)na); say = __ddiv_rn(say, (double)na); saz = __ddiv_rn(saz, (double)na); }
    const double speed = mag3_d(svx, svy, svz), accel = mag3_d(sax, say, saz);
    out[i] = speed < 0.1 ? RCD_PAT_STATIONARY : (accel < 0.1 ? RCD_PAT_CONSTANT_VELOCITY : RCD_PAT_ACCELERATING);
}

// -------------------------------------------------------------------------------------------------
// Spatial slabs: select / pack / append halo objects (SURVEY.md 8e).  Record = 13 x u32:
// 11 floats (px..heading), meta (type | pattern << 8), id.
// -------------------------------------------------------------------------------------------------
constexpr int HALO_WORDS = 13;
constexpr int MAX_PEERS = 64;

struct SlabParams {
    int n_peers, self;
    float lo[MAX_PEERS], hi[MAX_PEERS];
    float halo;
};

// phase 0: count per peer; phase 1: pack at base[p] + cursor[p]++
__global__ void __launch_bounds__(256)
k_halo_pack(u32 n_owned, InputState in, SlabParams sp, int phase, unsigned long long *__restrict__ counts,
            const unsigned long long *__restrict__ base, u32 *__restrict__ out, unsigned long long cap) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_owned) return;
    float x = in.px[i];
    for (int p = 0; p < sp.n_peers; ++p) {
        if (p == sp.self) continue;
        if (x >= sp.lo[p] - sp.halo && x < sp.hi[p] + sp.halo) {
            unsigned long long k = atomicAdd(&counts[p], 1ULL);
            if (phase == 1) {
                unsigned long long pos = base[p] + k;
                if (pos < cap) {
                    u32 *r = out + pos * HALO_WORDS;
                    r[0] = __float_as_uint(x);
                    r[1] = __float_as_uint(in.py[i]);
                    r[2] = __float_as_uint(in.pz[i]);
                    r[3] = __float_as_uint(in.vx[i]);
                    r[4] = __float_as_uint(in.vy[i]);
                    r[5] = __float_as_uint(in.vz[i]);
                    r[6] = __float_as_uint(in.ax[i]);
                    r[7] = __float_as_uint(in.ay[i]);
                    r[8] = __float_as_uint(in.az[i]);
                    r[9] = __float_as_uint(in.size[i]);
                    r[10] = __float_as_uint(in.heading[i]);
                    r[11] = (u32)in.type[i] | ((u32)in.pattern[i] << 8);
                    r[12] = in.id ? in.id[i] : i;
                }
            }
        }
    }
}

// Single pass, nothing for the host to wait for: peer p's records go to its own region of the send buffer
// (offset[p], cap[p] records), the slot is claimed with one warp-aggregated atomic per peer.  counts[p] keeps the
// true number even when it exceeds cap[p] (the surplus is dropped: the caller checks the counts now and then and
// re-sizes the regions).
struct SlabRegions {
    unsigned long long offset[MAX_PEERS], cap[MAX_PEERS];
};
__global__ void __launch_bounds__(256)
k_halo_pack_regions(u32 n_owned, InputState in, SlabParams sp, SlabRegions rg, unsigned long long *__restrict__ counts,
                    u32 *__restrict__ out) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = i < n_owned;
    const float x = valid ? in.px[i] : 0.0f;
    const u32 lane = threadIdx.x & 31u;
    for (int p = 0; p < sp.n_peers; ++p) {
        if (p == sp.self) continue;
        const bool send = valid && x >= sp.lo[p] - sp.halo && x < sp.hi[p] + sp.halo;
        const u32 ballot = __ballot_sync(FULL_MASK, send);
        if (ballot == 0) continue;
        unsigned long long base = 0;
        const u32 leader = __ffs(ballot) - 1;
        if (lane == leader) base = atomicAdd(&counts[p], (unsigned long long)__popc(ballot));
        base = __shfl_sync(FULL_MASK, base, leader);
        if (!send) continue;
        const unsigned long long k = base + __popc(ballot & lanemask_lt());
        if (k >= rg.cap[p]) continue;
        u32 *r = out + (rg.offset[p] + k) * HALO_WORDS;
        r[0] = __float_as_uint(x);
        r[1] = __float_as_uint(in.py[i]);
        r[2] = __float_as_uint(in.pz[i]);
        r[3] = __float_as_uint(in.vx[i]);
        r[4] = __float_as_uint(in.vy[i]);
        r[5] = __float_as_uint(in.vz[i]);
        r[6] = __float_as_uint(in.ax[i]);
        r[7] = __float_as_uint(in.ay[i]);
        r[8] = __float_as_uint(in.az[i]);
        r[9] = __float_as_uint(in.size[i]);
        r[10] = __float_as_uint(in.heading[i]);
        r[11] = (u32)in.type[i] | ((u32)in.pattern[i] << 8);
        r[12] = in.id ? in.id[i] : i;
    }
}

struct MutableState {
    float *f[11];
    uint8_t *type, *pattern;
    u32 *id;
};

__global__ void __launch_bounds__(256)
k_halo_append(const u32 *__restrict__ rec, u32 n_rec, u32 dst_base, MutableState st) {
    u32 r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rec) return;
    const u32 *w = rec + (size_t)r * HALO_WORDS;
    u32 d = dst_base + r;
#pragma unroll
    for (int k = 0; k < 11; ++k) st.f[k][d] = __uint_as_float(w[k]);
    st.type[d] = (uint8_t)(w[11] & 0xffu);
    st.pattern[d] = (uint8_t)((w[11] >> 8) & 0xffu);
    st.id[d] = w[12];
}

__global__ void __launch_bounds__(256) k_iota(u32 *p, u32 n) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = i;
}

}  // namespace rcd
