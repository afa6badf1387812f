/*
 * rcd.h -- C-ABI of the B200-native collision core (librcd_b200.so).
 *
 * The reference (jectpro7/realtime-collision-detection) is pure Python and has no FFI; its hot
 * path sits behind plain in-process classes.  This header is the boundary a maintainer binds
 * with ctypes (see INTEGRATION.md): every entry point names the reference interface it replaces
 * (file:line relative to the reference tree).  Plain pointers and sizes only; no C++/torch types.
 *
 * Conventions
 *   - every function returns int: RCD_OK (0) or a negative RCD_E* code; never throws, never
 *     long-jumps; rcd_last_error() gives a message for the last failure on that handle.
 *   - the library never frees or keeps caller memory; inputs are copied during the call (host
 *     pointers) or enqueued on the handle's stream (device pointers, src = RCD_SRC_DEVICE).
 *   - one CUDA stream per handle; a handle is used from one thread at a time (the reference is
 *     single-threaded asyncio: src/collision/warning_system.py:680-714).
 *   - object state is fp32 SoA (48 B/object).  Decisions (pair sets, thresholds, alert classes)
 *     are taken exactly as the reference's float64 arithmetic would take them on these fp32
 *     values: the fp32 kernels only pre-filter, every pair near a threshold is re-evaluated in
 *     fp64 on the device (DESIGN.md, "exactness").
 *   - there is no CPU fallback: without a CUDA device rcd_create fails with RCD_ENODEVICE.
 */
#ifndef RCD_H_
#define RCD_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RCD_VERSION 100 /* 0.1.0 */

enum {
    RCD_OK = 0,
    RCD_EINVAL = -1,    /* bad argument */
    RCD_ENODEVICE = -2, /* no usable CUDA device */
    RCD_ENOMEM = -3,    /* host or device allocation failed */
    RCD_ECUDA = -4,     /* a CUDA call failed (see rcd_last_error) */
    RCD_ECAPACITY = -5, /* more objects than max_objects */
    RCD_ESTATE = -6     /* call order (e.g. download before step) */
};

/* frame modes for rcd_step */
enum {
    /* CollisionDetector.detect_collisions for every object
     * (src/collision/collision_detection.py:110-191, stages :208-389) */
    RCD_MODE_DETECT = 0,
    /* CollisionPredictionModel.predict_collisions for every object (:572-865); per-object
     * trajectory pattern from rcd_set_patterns (pattern 3 = history < 2 -> detect path, :590-592) */
    RCD_MODE_PREDICT = 1,
    /* compute-node detector: SpatialIndex.query_nearby + CollisionDetector.detect_collisions
     * (src/compute/compute_node.py:98-119, :229-321) */
    RCD_MODE_COMPUTE_NODE = 2
};

/* OR-ed into the mode of rcd_step: keep the pairs and totals of the previous rcd_step of this frame
 * and append to them.  The reference's perf harness runs detect and predict for every vehicle in
 * one frame (src/test/performance_test.py:794-813); that is rcd_step(DETECT) followed by
 * rcd_step(PREDICT | RCD_STEP_APPEND) on the same index. */
#define RCD_STEP_APPEND 0x100
/* OR-ed into RCD_MODE_PREDICT: the predict pass also runs detect_collisions(search_radius, time_window)
 * for every object, in the same sweep over the neighbourhoods -- the result (pairs, totals) is that of
 * rcd_step(DETECT, r, t) followed by rcd_step(PREDICT | RCD_STEP_APPEND), i.e. the reference harness's
 * frame (performance_test.py:794-813), for one pass over the data.  With search_radius = 100 and
 * time_window = 10 (the reference's defaults) the two are fused in one kernel; other values run the two
 * passes back to back.  Per-object candidate counts then cover both parts. */
#define RCD_STEP_WITH_DETECT 0x200

enum { RCD_SRC_HOST = 0, RCD_SRC_DEVICE = 1 };

/* trajectory pattern codes (collision_detection.py:698-703; 3 = fewer than 2 history samples) */
enum { RCD_PAT_STATIONARY = 0, RCD_PAT_CONSTANT_VELOCITY = 1, RCD_PAT_ACCELERATING = 2, RCD_PAT_NO_HISTORY = 3 };

typedef struct rcd_handle_s *rcd_handle;

typedef struct {
    int32_t device;       /* CUDA device ordinal */
    uint32_t flags;       /* RCD_FLAG_* */
    uint64_t max_objects; /* capacity of the handle (owned + halo objects) */
    uint64_t max_pairs;   /* capacity of the emitted-pair buffer; counts stay exact beyond it */
    /* grid bounds.  If world_min[0] > world_max[0] the bounds are taken from the data each
     * frame (one extra device->host sync per frame); objects outside the bounds are clamped
     * into the border cells, which stays exact (DESIGN.md, "grid"). */
    float world_min[3];
    float world_max[3];
} rcd_config;

#define RCD_FLAG_PROFILE 1u /* record CUDA events around every stage (rcd_stage_ms) */
/* Predict mode: also count the (i, j, offset) radius hits of collision_detection.py:801-803 in
 * n_candidates / the per-object counts.  The reference keeps no such statistic on the predict
 * path; it is a diagnostic (and the parity tests use it) and costs one more distance test per
 * offset.  Without the flag predict frames report candidates only for pattern-3 objects. */
#define RCD_FLAG_COUNT_PREDICT_CANDIDATES 2u
/* Replay rcd_step as a CUDA graph: when a call has the same shape as the one before it (mode, radius,
 * window, object counts, buffers), its launch sequence (~17 memsets and kernels) is captured once and
 * replayed with a single launch afterwards.  Pays off for small frames, where launch gaps are a third of
 * the frame (5 k objects: ~0.1 ms of 0.27 ms).  Needs static world bounds; ignored with RCD_FLAG_PROFILE. */
#define RCD_FLAG_GRAPH 4u

/* One emitted, directed pair (i -> j): the fields of the reference's CollisionRisk
 * (collision_detection.py:156-166, :831-842) plus the stage-2 values and the alert class
 * (src/collision/warning_system.py:259-311).  48 bytes. */
typedef struct {
    uint32_t i, j;      /* caller ids of the querying object and of the other object */
    float ttc;          /* time_to_collision: k*0.1 (detect) or k*0.1 + t_m (predict); B: formula ttc */
    float distance;     /* distance at the first sample inside the safe distance; B: future distance */
    float rel_speed;    /* |v_i - v_j| */
    float risk;         /* risk_level in [0, 1] */
    float cx, cy, cz;   /* collision_position (midpoint) */
    float t_closest;    /* detect: time_to_closest (stage 2); predict: winning offset time t_m */
    float d_closest;    /* detect: closest_distance (stage 2); otherwise 0 */
    int8_t priority;    /* alert class: -1 below RISK_LEVEL_LOW, else 0..3; B: -1 */
    uint8_t offset;     /* predict: winning offset index m (0..19); otherwise 255 */
    uint8_t predicted;  /* CollisionRisk.is_predicted */
    uint8_t reserved;
} rcd_pair;

/* frame totals (exact even when the pair buffer overflowed) */
typedef struct {
    uint64_t n_objects;    /* objects in the frame (owned + halo) */
    uint64_t n_owned;      /* objects queried */
    uint64_t n_candidates; /* directed broad-phase pairs (stage 1); compute-node mode counts self like
                              query_nearby; predict mode: see RCD_FLAG_COUNT_PREDICT_CANDIDATES */
    uint64_t n_potential;  /* stage-2 survivors (stats["potential_collisions"], :177) */
    uint64_t n_pairs;      /* emitted risks */
    uint64_t n_high_risk;  /* risk > 0.7 (stats["high_risk_collisions"], :178) */
    uint64_t n_written;    /* pairs actually stored (<= max_pairs) */
    uint64_t n_alerts[4];  /* alerts by priority 0..3 (risk >= 0.3) */
    uint64_t n_exact;      /* pairs that took the fp64 re-evaluation path (diagnostic) */
    uint64_t n_fallback;   /* fp32-settled pairs the fp64 stage had to redo in full: 0 while the guard
                              bands hold (diagnostic; results are exact either way) */
} rcd_counts_t;

#define RCD_NUM_STAGES 10
/* stage indices for rcd_stage_ms */
enum {
    RCD_STAGE_UPLOAD = 0,  /* host->device copies of the SoA state */
    RCD_STAGE_KEYS = 1,    /* k_pack_keys + k_scan_hist: cell keys + digit histograms */
    RCD_STAGE_SORT = 2,    /* k_onesweep_pass x passes */
    RCD_STAGE_REORDER = 3, /* k_reorder + k_cell_table: gather into cell order + dense cell table */
    RCD_STAGE_PAIRS = 4,   /* k_pairs: pair enumeration, radius test + closest-approach filter (fp32) */
    RCD_STAGE_NARROW = 5,  /* k_narrow: fp32 narrow phase (temporal filter; predict: window, 10 samples per offset) */
    RCD_STAGE_EXACT = 6,   /* k_exact: fp64 decision, merge, emit, alert class */
    RCD_STAGE_DOWNLOAD = 7,
    RCD_STAGE_TOTAL = 8,
    RCD_STAGE_QORDER = 9   /* k_query_keys + k_onesweep_pass x 3: query order (tiles of overlapping query volumes) */
};

int rcd_version(void);
const char *rcd_last_error(rcd_handle h); /* h may be NULL: last error of rcd_create */

int rcd_create(const rcd_config *cfg, rcd_handle *out);
int rcd_destroy(rcd_handle h);

/* ---- growing a handle in place ------------------------------------------------------------------------
 * Grow the handle to max_objects objects and / or max_pairs emitted pairs.  0 keeps the current value, and so does a
 * value below it: the handle never shrinks.  A call that changes neither is a no-op.
 *   - Kept: the first n entries (owned and halo) of the object state, type, pattern and caller id; n, n_owned, the
 *     record-built flag (rcd_retire_stale), the record times, the trajectory rings and their counts, the query list
 *     of rcd_set_queries, the compute-node parameters, the world bounds, the alert table with its counters and alert
 *     numbering, and the slot layout rcd_apply_records writes to.  A step after rcd_reserve, with no other call in
 *     between, emits exactly what the same step would have emitted without it.
 *   - Slots in [n, new max_objects) start as rcd_create and rcd_history_configure leave them: zero state, no ring
 *     samples, no record time.
 *   - Every buffer is sized exactly as in a handle created at the final size, so such a handle and a grown one step
 *     alike, pair-test counts (rcd_pair_tests) included.
 *   - Ends the frame, like rcd_set_queries: rcd_counts, rcd_download*, rcd_pair_tests and rcd_alerts_update return
 *     RCD_ESTATE until the next rcd_step, and so does a following RCD_STEP_APPEND.  The spatial index is rebuilt by
 *     the next step and every captured step graph (RCD_FLAG_GRAPH) is dropped, to be captured again.
 *   - RCD_ESTATE while a download or summary delivery is in flight (finish it first).  Otherwise the call first waits
 *     for the handle's streams, the alert stream included, and synchronises again before it returns.
 *   - Old and new buffers coexist during the call: peak device memory is the old set plus the new one.  The new set
 *     is complete before it replaces the old one, so a failure leaves the handle untouched and usable: RCD_ENOMEM for
 *     a refused allocation, RCD_EINVAL for max_objects >= 2^30 (as in rcd_create). */
int rcd_reserve(rcd_handle h, uint64_t max_objects, uint64_t max_pairs);

/* Replace the frame's object state.  Replaces N x CollisionDetector.update_vehicle +
 * SpatialIndex.insert_vehicle (collision_detection.py:74-85, spatial_index.py:162-200) and
 * compute_node.SpatialIndex.insert (compute_node.py:55-72).  All arrays have n entries; id may be
 * NULL (ids 0..n-1); type is a small integer per distinct type string (only equality is used,
 * collision_detection.py:498-513).  az/ay/ax/heading/size/type may be NULL (zeros). */
int rcd_upload(rcd_handle h, uint64_t n, const float *px, const float *py, const float *pz,
               const float *vx, const float *vy, const float *vz, const float *ax, const float *ay,
               const float *az, const float *size, const float *heading, const uint8_t *type,
               const uint32_t *id, int32_t src);

/* Per-object flags: predict mode = trajectory pattern code (RCD_PAT_*); compute-node mode =
 * 1 if the VehicleState has >= 2 history samples (compute_node.py:202-203), else 0.
 * NULL resets to the default (RCD_PAT_ACCELERATING / has history). */
int rcd_set_patterns(rcd_handle h, uint64_t n, const uint8_t *pattern, int32_t src);

/* Objects [0, n_owned) are queried; objects [n_owned, n) are halo copies owned by another
 * shard: they are neighbours only (spatial slabs, SURVEY.md 8e).  Default: all owned. */
int rcd_set_owned(rcd_handle h, uint64_t n_owned);

/* Query only the listed objects in the following rcd_step calls; every object stays a neighbour.
 * The reference's partitioned queries (collision_system.py:437-446).  slots: upload-order indices,
 * each < n_owned, no repeats, any order; host or device memory (src), copied.  NULL: back to every
 * owned object.  n = 0 with a non-NULL list: no queries.
 *   - A step with query set Q emits exactly the records the same step without a list emits for i in Q
 *     (the same bytes after rcd_download's sort).  rcd_counts_t.n_owned is |Q|; n_candidates,
 *     n_potential, n_pairs, n_high_risk and n_alerts are the totals over Q; the per-object candidate
 *     and risk counts are zero for objects outside Q.
 *   - A slot >= n_owned (a halo copy) or a repeated slot: RCD_EINVAL, and the previous set stays.
 *     Host lists are checked on the host; device lists by a kernel with one 4-byte readback, so
 *     such a call synchronises.
 *   - The set stays in force across steps.  rcd_upload, rcd_set_owned and rcd_truncate reset it to
 *     every owned object; rcd_halo_append, rcd_apply_records, rcd_set_patterns, rcd_invalidate and
 *     rcd_set_compute_node_params keep it.
 *   - The spatial index is kept: a new set only rebuilds the query order, O(|Q|).  Like
 *     rcd_set_owned, the call ends the frame (a following RCD_STEP_APPEND gets RCD_ESTATE).
 *   - The first call with a list allocates about 8 bytes of device memory per object. */
int rcd_set_queries(rcd_handle h, uint64_t n, const uint32_t *slots, int32_t src);

/* Run one frame for every owned object, asynchronously on the handle's stream.
 * search_radius / time_window: the arguments of detect_collisions (collision_detection.py:110-111);
 * predict mode always uses 100.0 / 1.0 like the reference (:802, :821) and ignores them except
 * for pattern-3 objects, which use the defaults 100.0 / 10.0 (:592).  Compute-node mode uses
 * search_radius as NodeConfig.search_radius (compute_node.py:620-622). */
int rcd_step(rcd_handle h, int32_t mode, float search_radius, float time_window);

/* Compute-node mode parameters: CollisionDetector(prediction_time=5.0, risk_threshold=0.5)
 * (src/compute/compute_node.py:218-227).  Defaults are the reference's. */
int rcd_set_compute_node_params(rcd_handle h, float prediction_time, float risk_threshold);

/* Keep only the first n objects (drop halo copies appended after the owned objects); the
 * remaining objects all become owned.  n must not exceed the current object count. */
int rcd_truncate(rcd_handle h, uint64_t n);

/* The object state was modified in place (device-resident frames): rebuild the index on the next
 * rcd_step even though rcd_upload was not called. */
int rcd_invalidate(rcd_handle h);

/* Build the spatial index only (cell keys -> radix sort -> cell-ordered state + cell ranges) for
 * a query radius `cell_radius`; rcd_step and rcd_query_radius do this implicitly.  Replaces the
 * clear() + N x insert part of the reference's timed region (src/test/performance_test.py:794-800).
 * Stage times are reported under mode RCD_MODE_DETECT. */
int rcd_build_index(rcd_handle h, float cell_radius);

/* Wait for the frame and return its totals. */
int rcd_counts(rcd_handle h, rcd_counts_t *out);

/* Copy the emitted pairs to host memory, sorted by (i, j, predicted); *n_out = pairs copied (<= cap). */
int rcd_download(rcd_handle h, rcd_pair *out, uint64_t cap, uint64_t *n_out);

/* Same without the ordering (emission order is not deterministic): for consumers that group or
 * sort on their own, or only stream the pairs onwards. */
int rcd_download_unsorted(rcd_handle h, rcd_pair *out, uint64_t cap, uint64_t *n_out);

/* Pipelined delivery: start handing the frame just stepped over to the host and return at once.  The
 * handle keeps two pair buffers and two sets of totals; the next rcd_upload / rcd_step may be issued
 * immediately and writes into the other set, so the device->host copy of frame k (on the handle's copy
 * stream) overlaps the kernels of frame k + 1.  rcd_download_finish waits for frame k, copies
 * min(n_written, cap) pairs (emission order, like rcd_download_unsorted) to `out` -- pinned host memory
 * for a copy that really overlaps -- and returns that frame's totals.  One download in flight at a time.
 * Between begin and finish the totals / pairs of frame k stay readable through rcd_counts,
 * rcd_download*, rcd_alerts_update until the next rcd_step. */
int rcd_download_begin(rcd_handle h, rcd_pair *out, uint64_t cap);
int rcd_download_finish(rcd_handle h, rcd_counts_t *counts, uint64_t *n_out);

/* Compact pair record for consumers that do not need the collision position or the stage-2 values: the fields
 * AlertManager.process_collision_risks reads (warning_system.py:259-285, 313-329) plus the relative speed.  32 bytes. */
typedef struct {
    uint32_t i, j;
    float ttc, distance, rel_speed, risk;
    float t_closest;    /* detect: time_to_closest; predict: winning offset time t_m */
    int8_t priority;
    uint8_t offset;
    uint8_t predicted;
    uint8_t reserved;
} rcd_pair_compact;
/* Like rcd_download_begin / rcd_download_finish with compact records: the frame's pairs are narrowed to 32 bytes on
 * the device (one pass over the pair buffer) before they cross the bus.  rcd_download_finish serves both kinds. */
int rcd_download_begin_compact(rcd_handle h, rcd_pair_compact *out, uint64_t cap);

/* Risks emitted for every object of the last frame (as the querying vehicle), upload order, n entries. */
int rcd_download_risk_counts(rcd_handle h, uint32_t *out, uint64_t n);

/* Per-object broad-phase candidate counts of the last frame, in upload order (n entries). */
int rcd_download_candidate_counts(rcd_handle h, uint32_t *out, uint64_t n);

/* Radius queries against the uploaded objects.  Replaces SpatialIndex.get_nearby_vehicles
 * (spatial_index.py:229-271) and compute_node.SpatialIndex.query_nearby (compute_node.py:98-119):
 * all ids with distance <= radius, the querying object included (quirk Q8).  Results are
 * returned CSR-style: offsets[nq + 1], ids (ascending upload order per query) up to cap. */
int rcd_query_radius(rcd_handle h, uint64_t nq, const float *qx, const float *qy, const float *qz,
                     float radius, uint64_t *offsets, uint32_t *ids, uint64_t cap);

/* ---- the per-pair helpers of the detector ----------------------------------------------------------
 * CollisionPredictionModel calls two semi-private methods of the detector for every pair it examines
 * (collision_detection.py:821-830): _precise_collision_detection (:296-342) and _risk_assessment (:344-389).
 * Inside a frame their work is fused into the pair kernels; these entry points evaluate them for explicit
 * pairs, in float64 on the device, in the reference's operation order (the same device functions the
 * frame kernels use: rcd_exact.cuh), so that callers of the helpers -- and unit tests -- get the same bits. */
typedef struct {
    float px, py, pz, vx, vy, vz, ax, ay, az, size, heading;
    uint32_t type;
} rcd_object;  /* one vehicle, 48 bytes */
typedef struct {
    int32_t hit;    /* 0: no sample within the safe distance (the reference returns None) */
    int32_t step;   /* index of the first such sample */
    double collision_time, distance, safe_distance, relative_speed;
    double cx, cy, cz;  /* collision_position (midpoint) */
    double risk;        /* _risk_assessment of that collision_info */
} rcd_pair_exact_result;  /* 72 bytes */
/* _precise_collision_detection(a[k], b[k], time_window, time_step) + _risk_assessment for n pairs (host arrays). */
int rcd_pair_exact(rcd_handle h, uint64_t n, const rcd_object *a, const rcd_object *b, double time_window,
                   double time_step, rcd_pair_exact_result *out);
/* _risk_assessment for n explicit collision_info records: in[k] = {heading_i, heading_j, same type ? 1 : 0,
 * collision_time, distance, safe_distance, relative_speed} (7 doubles each) -> risk_out[k]. */
int rcd_risk_assessment(rcd_handle h, uint64_t n, const double *in, double *risk_out);

/* Trajectory-pattern classifier (collision_detection.py:623-711) for n objects with up to
 * `stride` (x, y, z, t) float64 samples each, already in timestamp order; count[i] samples are
 * valid.  Writes RCD_PAT_* codes to pattern_out (host). */
int rcd_classify_patterns(rcd_handle h, uint64_t n, uint32_t stride, const double *samples,
                          const uint32_t *count, uint8_t *pattern_out);

/* Trajectory history on the device: replaces CollisionPredictionModel.update_trajectory +
 * _analyze_trajectory_pattern (collision_detection.py:553-570, 623-711) without re-staging every
 * vehicle's samples from the host each frame.  The handle keeps a ring of the last `max_history`
 * (default 100, :539) float64 (x, y, z, t) samples per object slot (= upload order index).
 * Samples of one object must arrive with non-decreasing timestamps (the reference sorts by
 * timestamp before classifying; callers with out-of-order samples use rcd_classify_patterns). */
int rcd_history_configure(rcd_handle h, uint32_t max_history);
/* Append one sample for each listed slot (slot may be NULL: slots 0..n-1; a slot must not appear
 * twice in one call).  Host arrays. */
int rcd_history_append(rcd_handle h, uint64_t n, const uint32_t *slot, const double *x, const double *y,
                       const double *z, const double *t);
/* Forget the history of the listed slots (new vehicle in a recycled slot). */
int rcd_history_reset(rcd_handle h, uint64_t n, const uint32_t *slot);
/* Copy the history of slot src to slot dst (the host table moved an object, e.g. swap-remove). */
int rcd_history_move(rcd_handle h, uint32_t dst, uint32_t src);
/* Classify every uploaded object from its ring and store the codes as the frame's patterns
 * (what rcd_set_patterns would set); optionally copy the n codes to pattern_out (host, may be NULL). */
int rcd_history_classify(rcd_handle h, uint8_t *pattern_out);

/* ---- batched ingest (SURVEY.md 8f rank 2) ---------------------------------------------------------
 * The reference receives one JSON message per vehicle update (src/test/vehicle_simulator.py:721-752)
 * and rebuilds a Vehicle from it in Python (src/collision/warning_system.py:638-678).  rcd_ingest_*
 * decodes whole buffers of those messages on the host into fixed records; rcd_apply_records scatters
 * the records into the device-resident frame state and trajectory rings. */
typedef struct {
    double x, y, z;      /* position, float64 as on the wire (the ring keeps float64, the frame state fp32) */
    double timestamp;
    float vx, vy, vz, ax, ay, az, size, heading;
    uint32_t slot;       /* dense object index = position in the frame (rcd_ingest interns the id string) */
    uint8_t type;        /* interned type string */
    uint8_t seq;         /* how many earlier records of the same batch carry the same slot */
    uint16_t reserved;
} rcd_record;            /* 72 bytes */

typedef struct rcd_ingest_s *rcd_ingest;
int rcd_ingest_create(rcd_ingest *out);
int rcd_ingest_destroy(rcd_ingest g);
const char *rcd_ingest_last_error(rcd_ingest g);
/* Decode every message in buf[0, len): JSON objects separated by whitespace / newlines / commas,
 * optionally inside one array.  threads: 0 = all host cores, 1 = sequential; with more than one thread
 * (and len >= 1 MiB) the buffer is cut at newlines, so a message must not contain a raw newline
 * (json.dumps never emits one).  Messages that are malformed or lack a field the reference reads are
 * skipped and counted in *n_bad (the reference logs and drops them, warning_system.py:677-678).
 * *n_out = messages decoded, *max_seq = largest rcd_record.seq of the batch.  If the buffer holds more than
 * `cap` well-formed messages nothing is decoded, *n_out = how many there are and the call returns RCD_ECAPACITY
 * (no state has changed: call again with a larger buffer).  Every message is taken or dropped on its own, like
 * in the reference's handler: the limits of the record format never fail a batch -- the 256th and later
 * messages of one vehicle in one call are dropped (counted in *n_bad), type strings beyond the first 255
 * distinct ones share code 255, and once rcd_ingest_set_limit's id limit is reached messages of unknown
 * vehicles are dropped (counted in *n_bad) while known vehicles keep being served.  Needs no CUDA device. */
int rcd_ingest_decode_json(rcd_ingest g, const char *buf, uint64_t len, int32_t threads, rcd_record *out,
                           uint64_t cap, uint64_t *n_out, uint64_t *n_bad, uint32_t *max_seq);
int rcd_ingest_counts(rcd_ingest g, uint64_t *n_ids, uint64_t *n_types);
/* At most max_ids distinct vehicle ids are interned (= the frame capacity the records are applied to). */
int rcd_ingest_set_limit(rcd_ingest g, uint64_t max_ids);
/* Messages dropped since creation because of the id limit or the 255-messages-per-vehicle-per-call limit. */
int rcd_ingest_rejected(rcd_ingest g, uint64_t *n);
/* interned strings (UTF-8, not NUL-terminated; valid until the next decode call) */
int rcd_ingest_id_name(rcd_ingest g, uint32_t slot, const char **name, uint32_t *len);
int rcd_ingest_type_name(rcd_ingest g, uint32_t code, const char **name, uint32_t *len);
int rcd_ingest_lookup(rcd_ingest g, const char *id, uint32_t len, uint32_t *slot); /* RCD_ESTATE if unknown */
/* Forget the ids of the listed slots (vehicles retired with rcd_retire / rcd_retire_stale); the next new ids take the
 * freed slots, lowest first, before any fresh slot.  The id limit (rcd_ingest_set_limit) then counts live ids;
 * rcd_ingest_counts' n_ids stays "slots handed out" (the frame size to pass to rcd_apply_records).  *n_live = ids
 * interned afterwards (may be NULL).  A free or out-of-range slot, or a repeat: RCD_EINVAL, nothing changes.  After a
 * release, rcd_ingest_lookup of a released id gives RCD_ESTATE and rcd_ingest_id_name of a free slot RCD_EINVAL.
 * Records decoded before a release must be applied before it. */
int rcd_ingest_release(rcd_ingest g, uint64_t n, const uint32_t *slots, uint64_t *n_live);

/* Apply n decoded records to the frame: state[slot] = record for every record, in seq order
 * (N x CollisionDetector.update_vehicle, collision_detection.py:74-85), and -- if the trajectory rings
 * are configured (rcd_history_configure) and append_history != 0 -- one ring sample per record
 * (N x update_trajectory, :553-570).  n_objects = frame size afterwards (>= every slot + 1, >= the
 * current size; objects without a record keep their state).  records: host or device memory (src).
 * The timestamp of each slot's newest record is kept for rcd_retire_stale (8 bytes of device memory per
 * object, allocated at the first call).  A record for a retired slot brings it back as a fresh vehicle. */
int rcd_apply_records(rcd_handle h, uint64_t n, const rcd_record *records, uint32_t max_seq,
                      uint64_t n_objects, int32_t append_history, int32_t src);

/* ---- alert lifecycle on the device (SURVEY.md 8f rank 3) --------------------------------------------
 * Replaces the per-risk dict walk of AlertManager.process_collision_risks / update_alert / create_alert
 * (src/collision/warning_system.py:259-285, 120-197), _cleanup_expired_alerts (:488-517) and
 * acknowledge_alert (:199-213): one alert per directed pair (i, j) lives in a device hash table; a
 * frame's emitted pairs are folded into it without leaving the device and only the changes come back. */
enum {
    RCD_ALERT_REFRESHED = 0,        /* existing alert updated, same priority (not reported unless asked for) */
    RCD_ALERT_CREATED = 1,          /* create_alert: no alert existed for (i, j) */
    RCD_ALERT_PRIORITY_CHANGED = 2, /* update_alert with a different priority (the reference re-queues it) */
    RCD_ALERT_EXPIRED = 3           /* removed by the cleanup: acknowledged, or older than max_age */
};
typedef struct {
    uint32_t i, j;        /* caller ids: vehicle_id, other_vehicle_id */
    uint32_t alert_id;    /* running number given at creation (the reference draws a uuid) */
    float risk, ttc;      /* risk_level, time_to_collision after the update */
    float distance;       /* CollisionRisk.distance of that risk (the alert message quotes it, :313-329) */
    int8_t priority;      /* after the update */
    int8_t old_priority;  /* before it (-1: none) */
    uint8_t kind;         /* RCD_ALERT_* */
    uint8_t acknowledged;
    uint32_t reserved;
    double timestamp;     /* AlertInfo.timestamp: `now` of the last update */
} rcd_alert_event;        /* 40 bytes */
typedef struct {
    uint64_t n_events;    /* events produced by the call (only min(n_events, cap) were stored) */
    uint64_t n_created, n_changed, n_refreshed, n_expired;
    uint64_t n_live;      /* alerts in the table after the call */
    uint64_t n_dropped;   /* risks that found the table full (size it with rcd_alerts_configure) */
} rcd_alert_stats;
/* Allocate (or reset) the table for up to max_alerts live alerts. */
int rcd_alerts_configure(rcd_handle h, uint64_t max_alerts);
/* Grow the table to max_alerts live alerts, keeping every live alert (unlike rcd_alerts_configure, which empties it):
 * each keeps its alert number, timestamp, risk / ttc / distance, priority and acknowledged flag, and the next created
 * alert gets the next number.  The event buffers grow to max_alerts.  max_alerts <= the current size: no-op.
 * RCD_ESTATE if the table was never configured or while a summary delivery is in flight; max_alerts > 2^31:
 * RCD_EINVAL.  Old and new tables coexist during the call; a refused allocation (RCD_ENOMEM) leaves the table as it
 * was.  Synchronises. */
int rcd_alerts_reserve(rcd_handle h, uint64_t max_alerts);
/* process_collision_risks on every pair the last rcd_step(s) of this frame emitted (risk >= 0.3 only,
 * :273), with time.time() = now.  events (host, may be NULL with cap 0) receives the CREATED and
 * PRIORITY_CHANGED events, plus the REFRESHED ones if report_refreshed != 0; order is not deterministic.
 * After a step with a query list (rcd_set_queries) only the pairs of listed objects are folded in: the alerts
 * of the other objects are not refreshed and age towards expiry, as the reference's alerts do for the vehicles
 * a shard does not process. */
int rcd_alerts_update(rcd_handle h, double now, int32_t report_refreshed, rcd_alert_event *events, uint64_t cap,
                      rcd_alert_stats *stats);
/* The same for an explicit list of risks (host array of rcd_pair; i, j, ttc, risk, distance, priority and predicted
 * are read; a pair with priority < 0 is skipped).  If (i, j) occurs more than once, a non-predicted entry
 * is applied before a predicted one; other duplicates are the caller's to split into separate calls. */
int rcd_alerts_update_pairs(rcd_handle h, const rcd_pair *pairs, uint64_t n, double now, int32_t report_refreshed,
                            rcd_alert_event *events, uint64_t cap, rcd_alert_stats *stats);
/* _cleanup_expired_alerts: drop every alert that is acknowledged or has now - timestamp > max_age
 * (the reference uses 30.0); events receives one EXPIRED event per dropped alert. */
int rcd_alerts_expire(rcd_handle h, double now, double max_age, rcd_alert_event *events, uint64_t cap,
                      rcd_alert_stats *stats);
/* acknowledge_alert for the alerts of the listed (i, j) pairs; *n_found = how many existed. */
int rcd_alerts_acknowledge(rcd_handle h, uint64_t n, const uint32_t *i, const uint32_t *j, uint64_t *n_found);
/* Every live alert, sorted by (i, j), as event records with kind = RCD_ALERT_REFRESHED. */
int rcd_alerts_download(rcd_handle h, rcd_alert_event *out, uint64_t cap, uint64_t *n_out);

/* Summary delivery: what the reference's consumer acts on -- the alert changes of the frame
 * (process_collision_risks folded into the device alert table: created alerts and priority changes, plus the
 * refreshed ones on request) and how many risks every object has -- while the pair records stay on the device.
 * Pipelined like rcd_download_begin / _finish: `begin` returns at once and the next rcd_upload / rcd_step may be
 * issued; `finish` waits for that frame, copies min(n_events, cap) events, the per-object risk counts (upload
 * order, n entries; NULL / 0 to skip) and the frame's totals.  Needs rcd_alerts_configure.  One delivery
 * (download or summary) in flight at a time. */
int rcd_summary_begin(rcd_handle h, double now, int32_t report_refreshed);
int rcd_summary_finish(rcd_handle h, rcd_alert_event *events, uint64_t cap, uint64_t *n_events, rcd_alert_stats *stats,
                       uint32_t *risk_counts, uint64_t n, rcd_counts_t *counts);
/* ---- retiring departed vehicles ----------------------------------------------------------------------
 * CollisionDetector.remove_vehicle / SpatialIndex.remove_vehicle (collision_detection.py:74-108,
 * spatial_index.py:202-227) and compute_node.SpatialIndex.remove for the device-resident frame.  A retired slot:
 *   - has no position (the all-bits-set ghost state of rcd_halo_pack_async), type 0, the default pattern
 *     (RCD_PAT_ACCELERATING), an empty trajectory ring and no record time; its caller id stays;
 *   - is nobody's neighbour and is never queried: it emits nothing and is counted nowhere -- its candidate and risk
 *     counts are 0, it adds nothing to n_candidates / n_potential / n_pairs / n_high_risk / n_alerts, and it is never
 *     a hit of rcd_query_radius;
 *   - keeps its place in the frame: n_objects / n_owned still count slots, retired ones included; nothing is compacted.
 * A later record for the slot (rcd_apply_records) brings it back as a fresh vehicle whose ring starts from 0.
 * Equivalence: a step on a frame whose live slots are L -- any mode, with or without a query list (a listed retired
 * slot emits nothing) or graph replay -- emits the same records (byte for byte after mapping upload index to slot)
 * with the same totals, and takes the same number of pair tests (rcd_pair_tests), as the same step on a frame
 * uploaded with only the vehicles of L, in slot order, with the same world bounds.
 * Alerts: when rcd_alerts_configure was called, every alert whose i or j is the caller id of a retired slot is
 * dropped and reported as an RCD_ALERT_EXPIRED event (n_expired / n_live follow), after an in-flight summary fold,
 * like rcd_alerts_expire; a recycled slot never inherits the previous vehicle's alerts.  events / cap / stats are
 * those of rcd_alerts_expire (NULL / 0 when alerts are not configured).
 * Both calls end the frame (a following RCD_STEP_APPEND gets RCD_ESTATE), invalidate the spatial index, keep the
 * query list of rcd_set_queries, and synchronise. */
/* Retire the listed slots (host array; each < n_objects; repeats and already-retired slots are no-ops).  A slot out
 * of range: RCD_EINVAL and nothing changes. */
int rcd_retire(rcd_handle h, uint64_t n, const uint32_t *slots, rcd_alert_event *events, uint64_t cap,
               rcd_alert_stats *stats);
/* Retire every live slot whose newest applied record has now - timestamp > max_age (strict, the form of the alert
 * expiry) and write those slots in ascending order to slots_out; *n_retired = how many.  More than slots_cap of them:
 * RCD_ECAPACITY, nothing is retired, *n_retired = how many there are (the rcd_ingest_decode_json convention).  Slots
 * with no record time (never written by a record, or retired) are never reported, so a second call at the same `now`
 * retires nothing.  A frame whose slots were not all written by rcd_apply_records since the last rcd_upload /
 * rcd_halo_append (an rcd_upload of 0 objects starts a record-built frame): RCD_ESTATE. */
int rcd_retire_stale(rcd_handle h, double now, double max_age, uint32_t *slots_out, uint64_t slots_cap,
                     uint64_t *n_retired, rcd_alert_event *events, uint64_t cap, rcd_alert_stats *stats);

/* Spatial-slab support (SURVEY.md 8e): pack every owned object whose x lies within `halo` of
 * peer p's slab [slab_lo[p], slab_hi[p]) -- p != self -- into 52-byte records
 * (11 floats, meta u32 = type | pattern << 8, id u32), grouped by peer.  out_records is a DEVICE
 * buffer of cap records; counts[n_peers] is written to host memory (synchronises).  out_records = NULL with
 * cap = 0 only counts. */
int rcd_halo_pack(rcd_handle h, int32_t n_peers, int32_t self, const float *slab_lo,
                  const float *slab_hi, float halo, void *out_records, uint64_t cap,
                  uint64_t *counts);
/* The same without a host round trip: peer p's records go to the region [peer_offset[p], peer_offset[p + 1]) of
 * out_records (a DEVICE buffer of peer_offset[n_peers] records; peer_offset is a host array); unused slots of
 * every region are left as ghost records (all bits set: an object without a position, which pairs with
 * nothing).  counts_dev (DEVICE, n_peers entries) receives the true counts, which may exceed a region: the
 * surplus is dropped, so the caller looks at the counts now and then and re-sizes the regions.  Fixed region
 * sizes make the exchange a fixed-size all_to_all and rcd_halo_append(everything received) the whole
 * receiving side: nothing in the per-frame path waits for the host. */
int rcd_halo_pack_async(rcd_handle h, int32_t n_peers, int32_t self, const float *slab_lo, const float *slab_hi,
                        float halo, void *out_records, const uint64_t *peer_offset, uint64_t *counts_dev);
/* Append n_records packed halo records (DEVICE buffer) after the owned objects. */
int rcd_halo_append(rcd_handle h, const void *records, uint64_t n_records);

/* Milliseconds of each stage of the last rcd_step that ran in `mode` (needs RCD_FLAG_PROFILE);
 * synchronises.  Index stages (keys, sort, reorder) are reported under the mode that built it;
 * upload / download are reported under every mode. */
int rcd_stage_ms(rcd_handle h, int32_t mode, float *ms /* RCD_NUM_STAGES */);
/* The handle's CUDA stream (a cudaStream_t), so the caller can order its own work -- halo
 * exchange with NCCL, timing events -- with the frame without extra synchronisation. */
int rcd_get_stream(rcd_handle h, void **stream);
/* (query, neighbour) tests the fp32 filter of the pair kernel took in the last frame (waits for it): the unit of work
 * of the kernel that dominates a frame -- it is issue-bound, not HBM-bound -- for bench.py's roofline object. */
int rcd_pair_tests(rcd_handle h, uint64_t *n);
/* Kernel launches issued by the last rcd_step (for bench.py's gpu_launches). */
int rcd_launch_count(rcd_handle h, uint64_t *n);
/* Steps served by graph replay since the handle was created (RCD_FLAG_GRAPH; diagnostic). */
int rcd_graph_replays(rcd_handle h, uint64_t *n);
int rcd_sync(rcd_handle h);

#ifdef __cplusplus
}
#endif
#endif /* RCD_H_ */
