// C-ABI of the collision core (include/rcd.h): handle, device buffers, frame orchestration.
// One stream per handle; every frame is a fixed sequence of kernel launches on that stream.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include "rcd_common.cuh"
#include "rcd_index.cuh"
#include "rcd_pairs.cuh"
#include "rcd_ingest.cuh"
#include "rcd_alerts.cuh"
#include "rcd_ingest.hpp"

using namespace rcd;

namespace {

thread_local std::string g_create_error;

constexpr u32 CELLS_CAP_MAX = 1u << 24;
constexpr u32 CELLS_CAP_MIN = 1u << 16;

// ---- owning handles of CUDA resources: move-only, released by the destructor --------------------------------
template <typename T, cudaError_t (*Release)(T)>
class Owned {
public:
    Owned() = default;
    Owned(Owned &&o) noexcept : v_(std::exchange(o.v_, nullptr)) {}
    Owned &operator=(Owned &&o) noexcept {
        if (this != &o) { reset(); v_ = std::exchange(o.v_, nullptr); }
        return *this;
    }
    ~Owned() { reset(); }
    void reset() {
        if (v_) Release(v_);
        v_ = nullptr;
    }
    T get() const { return v_; }
    operator T() const { return v_; }

protected:
    T v_ = nullptr;
};

template <typename T> cudaError_t alloc_device(T **p, size_t bytes) { return cudaMalloc(reinterpret_cast<void **>(p), bytes); }
template <typename T> cudaError_t free_device(T *p) { return cudaFree(p); }
template <typename T> cudaError_t alloc_host(T **p, size_t bytes) { return cudaMallocHost(reinterpret_cast<void **>(p), bytes); }
template <typename T> cudaError_t free_host(T *p) { return cudaFreeHost(p); }

// An array of T (at least one element); kernels take it as a T *.
template <typename T, cudaError_t (*Alloc)(T **, size_t), cudaError_t (*Free)(T *)>
struct Buffer : Owned<T *, Free> {
    cudaError_t alloc(size_t count = 1) {
        this->reset();
        return Alloc(&this->v_, std::max<size_t>(count, 1) * sizeof(T));
    }
    T *operator->() const { return this->v_; }
};
template <typename T> using DevBuf = Buffer<T, alloc_device<T>, free_device<T>>;
template <typename T> using HostBuf = Buffer<T, alloc_host<T>, free_host<T>>;  // pinned

struct Stream : Owned<cudaStream_t, cudaStreamDestroy> {
    cudaError_t create(int priority = 0) {
        reset();
        return cudaStreamCreateWithPriority(&v_, cudaStreamNonBlocking, priority);
    }
};

struct Event : Owned<cudaEvent_t, cudaEventDestroy> {
    cudaError_t create(unsigned flags = cudaEventDisableTiming) {
        reset();
        return cudaEventCreateWithFlags(&v_, flags);
    }
};

struct GraphExec : Owned<cudaGraphExec_t, cudaGraphExecDestroy> {
    cudaError_t instantiate(cudaGraph_t g) {
        reset();
        return cudaGraphInstantiate(&v_, g, 0);
    }
};

struct Stage {
    Event begin, end;
    bool used = false;
};

// The cell-ordered index a step derives from the objects; a graph replay restores it.
struct IndexState {
    GridParams grid = {};
    bool valid = false;
    float cell_req = 0.0f;
    int sorted_buf = 0;
    int qorder_kind = 0;   // 0 none, 1 balls (radius queries), 2 capsules (predict queries)
    int q_sorted_buf = 0;
    bool slot_pos = false; // q_pos holds the inverse of sorted_slot (built for a query list only)
};

// What a frame writes.  A pending delivery still reads the previous frame's set, so the handle keeps a twin.
struct FrameBuffers {
    DevBuf<rcd_pair> out;
    DevBuf<Counters> counters;
    DevBuf<u32> risk_count;
};

// Resources of the pipelined deliveries (rcd_download_begin / _finish, rcd_summary_begin / _finish), made at
// their first use.  Built completely before the handle takes them, so a failed attempt leaves nothing behind.
struct Delivery {
    HostBuf<Counters> counters_host;             // snapshot of the pending frame's totals
    HostBuf<AlertCounters> alert_counters_host;
    Stream copy_stream;
    Event pend_event;
    // summary deliveries fold the frame into the alert table on a stream of their own, next to the kernels of the
    // following frame (random 40-byte accesses beside ALU-bound pair kernels)
    Stream alert_stream;
    Event ev_frame_done, ev_alert_done;
};

// The kernels of one frame variant (index: the variant number of step_impl).
struct FrameKernels {
    void (*tile_plan)(PairParams);
    void (*pairs)(PairParams);
    void (*pairs_overflow)(PairParams);
    void (*narrow)(PairParams);
    void (*exact)(PairParams);
    void (*exact_resolved)(PairParams);  // second k_exact launch (RESOLVED records); null: none
};

const FrameKernels FRAME_KERNELS[5] = {
    // 0: detect
    {k_tile_plan<RCD_MODE_DETECT>, k_pairs<RCD_MODE_DETECT, false, false>, k_pairs<RCD_MODE_DETECT, false, true>,
     k_narrow<RCD_MODE_DETECT, false>, k_exact<RCD_MODE_DETECT, 0>, nullptr},
    // 1: predict
    {k_tile_plan<RCD_MODE_PREDICT>, k_pairs<RCD_MODE_PREDICT, false, false>, k_pairs<RCD_MODE_PREDICT, false, true>,
     k_narrow<RCD_MODE_PREDICT, false>, k_exact<RCD_MODE_PREDICT, 1>, k_exact<RCD_MODE_PREDICT, 2>},
    // 2: predict, counting candidates (RCD_FLAG_COUNT_PREDICT_CANDIDATES)
    {k_tile_plan<RCD_MODE_PREDICT>, k_pairs<RCD_MODE_PREDICT, true, false>, k_pairs<RCD_MODE_PREDICT, true, true>,
     k_narrow<RCD_MODE_PREDICT, true>, k_exact<RCD_MODE_PREDICT, 1>, k_exact<RCD_MODE_PREDICT, 2>},
    // 3: compute node
    {k_tile_plan<RCD_MODE_COMPUTE_NODE>, k_pairs<RCD_MODE_COMPUTE_NODE, false, false>,
     k_pairs<RCD_MODE_COMPUTE_NODE, false, true>, k_narrow<RCD_MODE_COMPUTE_NODE, false>, k_exact<RCD_MODE_COMPUTE_NODE, 0>,
     nullptr},
    // 4: detect + predict in one sweep
    {k_tile_plan<RCD_MODE_PREDICT>, k_pairs<MODE_PREDICT_WITH_DETECT, false, false>,
     k_pairs<MODE_PREDICT_WITH_DETECT, false, true>, k_narrow<MODE_PREDICT_WITH_DETECT, false>,
     k_exact<MODE_PREDICT_WITH_DETECT, 1>, k_exact<MODE_PREDICT_WITH_DETECT, 2>},
};

// RCD_FLAG_GRAPH: the launch sequence of a step is a pure function of this key (every other kernel argument is
// a buffer that lives as long as the handle).
struct StepKey {
    int32_t mode = -1;
    float R = 0, T = 0, pt = 0, thr = 0, index_cell_req = 0;
    u64 n = 0, n_owned = 0;  // n_owned: queries (the length of a query list)
    int index_valid = 0, sorted_buf = 0, frame_done = 0, qorder_kind = 0, q_sorted_buf = 0, listed = 0, slot_pos = 0;
    const void *out = nullptr;
    bool operator==(const StepKey &o) const {
        return mode == o.mode && R == o.R && T == o.T && pt == o.pt && thr == o.thr && index_cell_req == o.index_cell_req &&
               n == o.n && n_owned == o.n_owned && index_valid == o.index_valid && sorted_buf == o.sorted_buf &&
               frame_done == o.frame_done && qorder_kind == o.qorder_kind && q_sorted_buf == o.q_sorted_buf &&
               listed == o.listed && slot_pos == o.slot_pos && out == o.out;
    }
};

struct StepGraph {
    GraphExec exec;
    StepKey key;
    IndexState idx;
    int last_mode = 0;
    u64 launches = 0;
};

// Every buffer whose size follows from the handle's capacity (max_objects, max_pairs).  rcd_create makes one set
// (size_buffers); rcd_reserve makes a larger one the same way and swaps it in whole.  The optional parts, made at
// their first use, are sized by the same functions.
struct Sized {
    u64 cap = 0, max_pairs = 0;

    DevBuf<float> in_f[11];
    DevBuf<uint8_t> in_type, in_pattern;
    DevBuf<u32> in_id;

    DevBuf<u32> keys[2], vals[2];
    DevBuf<u32> tile_status;
    size_t tile_status_words = 0;

    DevBuf<float4> P0, P1, P2;
    DevBuf<float4> U;  // packed 48-byte records in upload order
    DevBuf<u32> sorted_slot;
    DevBuf<u32> sorted_id;   // caller ids in cell order (the frame kernels never touch the upload buffers)
    DevBuf<u32> cell_begin;  // [cells_cap + 1] dense cell table
    u32 cells_cap = 0;
    DevBuf<u32> qkeys[2], qvals[2];  // query order: Morton keys of the query volumes + permutation
    // rcd_set_queries: the listed query set.  Made at the first call with a list (about 8 B per object).
    DevBuf<u32> q_list;      // [cap] upload slots of the listed queries
    DevBuf<u32> q_pos;       // [cap] upload slot -> position in cell order (IndexState::slot_pos)
    DevBuf<u32> q_seen;      // [cap / 32 + 2] bitmap of the device-list check, then its error word
    HostBuf<u32> q_host;     // [cap] pinned copy of a host list on its way to q_list

    FrameBuffers bufs[2];  // the current set and the twin of the pipelined deliveries (made at their first use)
    DevBuf<u32> cand_count;
    DevBuf<QEntry> q3;
    u32 qcap = 0;
    DevBuf<uint2> qa;        // pair queue k_pairs -> k_narrow
    DevBuf<u32> qa_fill;
    u32 qa_blocks_cap = 0;
    DevBuf<uint4> ovf;       // work items (or rests of them) left to the overflow pass of k_pairs
    u32 ovf_cap = 0;
    DevBuf<uint4> items;     // work items of k_pairs (k_tile_plan)
    u32 items_cap = 0;
    DevBuf<int4> tile_box;   // [2 * tiles]
    DevBuf<uint2> tile_rowx; // [TILE_ROWS * tiles]
    DevBuf<rcd_pair_compact> compact_dev;    // scratch of rcd_download_begin_compact

    DevBuf<Sample64> traj;  // trajectory rings, [max_history][cap]
    DevBuf<u32> traj_count;
    u32 traj_len = 0;
    // rcd_retire_stale: per slot, the timestamp of the newest applied record (no_record_time(): none).  Made at the
    // first rcd_apply_records (8 B per object).
    DevBuf<double> last_seen;
};

}  // namespace

struct rcd_handle_s : Sized {
    int device = 0;
    u32 flags = 0;
    int sms = 1;  // multiprocessors of the device
    Stream stream;
    u64 n = 0, n_owned = 0;

    DevBuf<u32> hist, tile_counter;

    // uploads from host memory run on their own stream and overlap the previous frame: the upload buffers are
    // free again as soon as that frame's index is built (k_pack_keys + k_reorder have consumed them)
    Stream up_stream;
    Event ev_upload_done, ev_inputs_free;
    bool upload_pending = false, inputs_busy = false, capturing = false;
    float cell_scale = 0.5f;    // grid cell edge (x, y) as a fraction of the query radius
    Event q_copied;          // q_host is free again
    bool q_listed = false;
    u64 q_n = 0;
    // the objects a frame queries
    u64 queried() const { return q_listed ? q_n : n_owned; }

    bool world_static = false;
    float wmin[3] = {}, wmax[3] = {};
    DevBuf<int> bbox_dev;
    HostBuf<int> bbox_host;
    IndexState idx;

    int cur = 0;
    HostBuf<Counters> counters_host;
    DevBuf<u32> pair_tile_counter;
    int narrow_blocks[5] = {0, 0, 0, 0, 0};
    int pair_blocks[5] = {0, 0, 0, 0, 0};  // resident blocks per SM x SMs, per kernel variant
    bool frame_done = false;
    int last_mode = -1;

    Stage stages[3][RCD_NUM_STAGES];  // per frame mode
    int stage_mode = 0;
    float cn_prediction_time = 5.0f, cn_risk_threshold = 0.5f;
    // records_only: every slot of the frame came from rcd_apply_records (rcd_upload of a non-empty frame and
    // rcd_halo_append clear it, rcd_upload of an empty one sets it).
    bool records_only = true;
    u64 launches = 0;
    // CUDA-graph replay of rcd_step (RCD_FLAG_GRAPH)
    StepGraph graphs[4];
    int graph_next = 0;
    StepKey graph_candidates[4];  // keys seen recently (twin pair buffers make consecutive frames alternate)
    int graph_cand_next = 0;
    bool graph_broken = false;
    u64 graph_replays = 0;
    Delivery dl;
    bool alert_async = false;  // work on alert_stream the handle's stream has not been ordered after yet
    u64 last_n_pairs = 0;      // emitted pairs of the last frame whose totals reached the host (sizes the alert fold's grid)
    u64 last_n_detect_end = 0; // ... and where its records with predicted = 0 ended (grid of the fold's detect pass)
    bool flip_pending = false, download_pending = false;
    rcd_pair *pend_dev = nullptr, *pend_out = nullptr;
    u64 pend_cap = 0, pend_n = 0, pend_n_owned = 0;
    int pend_kind = 0;                       // 0 pairs, 1 compact pairs, 2 summary (alert events + risk counts)
    rcd_pair_compact *pend_out_compact = nullptr;
    u32 *pend_risk = nullptr;
    rcd_alert_event *pend_ev = nullptr;
    // alert table (rcd_alerts.cuh)
    DevBuf<AlertEntry> alert_tab[2];
    int alert_cur = 0;
    u64 alert_cap = 0, alert_ev_cap = 0;
    DevBuf<rcd_alert_event> alert_ev, alert_ev_alt;  // (twin: summary deliveries in flight)
    DevBuf<AlertCounters> alert_counters;
    HostBuf<AlertCounters> alert_counters_host;
    std::string err;

    FrameBuffers &fb() { return bufs[cur]; }
    // The previous frame is being delivered: the next one writes into the twin buffers.
    void flip() {
        cur ^= 1;
        flip_pending = false;
    }

    // The streams finish their work before the members release themselves.
    ~rcd_handle_s() {
        cudaSetDevice(device);
        if (up_stream) cudaStreamSynchronize(up_stream);
        if (stream) cudaStreamSynchronize(stream);
        if (dl.alert_stream) cudaStreamSynchronize(dl.alert_stream);
        if (dl.copy_stream) cudaStreamSynchronize(dl.copy_stream);
        (void)cudaGetLastError();
    }
};

namespace {

int fail(rcd_handle h, int code, const std::string &msg) {
    if (h) h->err = msg; else g_create_error = msg;
    return code;
}

#define CUDA_TRY(h, call)                                                                          \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) {                                                                  \
            return fail((h), e__ == cudaErrorMemoryAllocation ? RCD_ENOMEM : RCD_ECUDA,            \
                        std::string(#call) + ": " + cudaGetErrorString(e__));                      \
        }                                                                                          \
    } while (0)

// Return a status other than RCD_OK to the caller.
#define RC_TRY(call)                                                                               \
    do {                                                                                           \
        const int rc__ = (call);                                                                   \
        if (rc__ != RCD_OK) return rc__;                                                           \
    } while (0)

#define KERNEL_CHECK(h)                                                                            \
    do {                                                                                           \
        cudaError_t e__ = cudaGetLastError();                                                      \
        if (e__ != cudaSuccess) return fail((h), RCD_ECUDA, std::string("launch: ") + cudaGetErrorString(e__)); \
        ++(h)->launches;                                                                           \
    } while (0)

// Mark the profiling stages of one frame mode (mode < 0: of every mode, upload and download included) unused.
void reset_stages(rcd_handle h, int mode) {
    for (int m = 0; m < 3; ++m)
        for (int s = 0; s < RCD_NUM_STAGES; ++s)
            if (mode < 0 || (m == mode && s != RCD_STAGE_UPLOAD && s != RCD_STAGE_DOWNLOAD && s != RCD_STAGE_TOTAL))
                h->stages[m][s].used = false;
}

void stage_begin(rcd_handle h, int s, cudaStream_t on = nullptr) {
    if (h->flags & RCD_FLAG_PROFILE) {
        cudaEventRecord(h->stages[h->stage_mode][s].begin, on ? on : h->stream);
        h->stages[h->stage_mode][s].used = true;
    }
}
void stage_end(rcd_handle h, int s, cudaStream_t on = nullptr) {
    if (h->flags & RCD_FLAG_PROFILE) cudaEventRecord(h->stages[h->stage_mode][s].end, on ? on : h->stream);
}

// Order the handle's stream after an upload that is still running on the upload stream.
int wait_upload(rcd_handle h) {
    if (h->upload_pending && !h->capturing) {
        CUDA_TRY(h, cudaStreamWaitEvent(h->stream, h->ev_upload_done, 0));
        h->upload_pending = false;
    }
    return RCD_OK;
}
// The frame no longer reads the upload buffers: the next upload may overwrite them.
int release_inputs(rcd_handle h) {
    if (!h->capturing) {
        CUDA_TRY(h, cudaEventRecord(h->ev_inputs_free, h->stream));
        h->inputs_busy = true;
    }
    return RCD_OK;
}

InputState input_state(rcd_handle h) {
    InputState in;
    in.px = h->in_f[0]; in.py = h->in_f[1]; in.pz = h->in_f[2];
    in.vx = h->in_f[3]; in.vy = h->in_f[4]; in.vz = h->in_f[5];
    in.ax = h->in_f[6]; in.ay = h->in_f[7]; in.az = h->in_f[8];
    in.size = h->in_f[9]; in.heading = h->in_f[10];
    in.type = h->in_type; in.pattern = h->in_pattern; in.id = h->in_id;
    return in;
}

MutableState mutable_state(rcd_handle h) {
    MutableState st;
    for (int k = 0; k < 11; ++k) st.f[k] = h->in_f[k];
    st.type = h->in_type; st.pattern = h->in_pattern; st.id = h->in_id;
    return st;
}

// ---- sizing: every capacity-dependent buffer is made by one of these (h may be null: errors of rcd_create) ----------
// The pair buffer, totals and per-object risk counts of one frame.
int alloc_frame_buffers(rcd_handle h, u64 cap, u64 max_pairs, FrameBuffers &fb) {
    CUDA_TRY(h, fb.out.alloc(max_pairs));
    CUDA_TRY(h, fb.counters.alloc());
    CUDA_TRY(h, fb.risk_count.alloc(cap));
    return RCD_OK;
}
// rcd_set_queries: the list, the inverse map, the bitmap of the device-list check and the pinned staging copy.
int alloc_queries(rcd_handle h, u64 cap, Sized &s) {
    CUDA_TRY(h, s.q_list.alloc(cap));
    CUDA_TRY(h, s.q_pos.alloc(cap));
    CUDA_TRY(h, s.q_seen.alloc(cap / 32 + 2));
    CUDA_TRY(h, s.q_host.alloc(cap));
    return RCD_OK;
}
// Trajectory rings [len][cap], every ring empty.
int alloc_history(rcd_handle h, u64 cap, u32 len, cudaStream_t on, Sized &s) {
    CUDA_TRY(h, s.traj.alloc((size_t)len * cap));
    CUDA_TRY(h, s.traj_count.alloc(cap));
    CUDA_TRY(h, cudaMemsetAsync(s.traj_count, 0, (size_t)cap * sizeof(u32), on));
    s.traj_len = len;
    return RCD_OK;
}
// rcd_retire_stale's record times, none yet.
int alloc_last_seen(rcd_handle h, u64 cap, cudaStream_t on, Sized &s) {
    CUDA_TRY(h, s.last_seen.alloc(cap));
    CUDA_TRY(h, cudaMemsetAsync(s.last_seen, 0xff, (size_t)cap * sizeof(double), on));  // no record time
    return RCD_OK;
}

// The whole set for (cap, max_pairs), every buffer as rcd_create leaves it; `like` (rcd_reserve: the set being
// replaced) adds the optional parts it has.  The memsets run on `on`.
int size_buffers(rcd_handle h, u64 cap, u64 max_pairs, const Sized *like, cudaStream_t on, Sized &s) {
    s.cap = cap;
    s.max_pairs = max_pairs;
    s.cells_cap = (u32)std::min<u64>(std::max<u64>(4 * cap, CELLS_CAP_MIN), CELLS_CAP_MAX);
    for (int k = 0; k < 11; ++k) {
        CUDA_TRY(h, s.in_f[k].alloc(cap));
        CUDA_TRY(h, cudaMemsetAsync(s.in_f[k], 0, cap * sizeof(float), on));
    }
    CUDA_TRY(h, s.in_type.alloc(cap));
    CUDA_TRY(h, s.in_pattern.alloc(cap));
    CUDA_TRY(h, s.in_id.alloc(cap));
    for (int k = 0; k < 2; ++k) {
        CUDA_TRY(h, s.keys[k].alloc(cap + 4));
        CUDA_TRY(h, s.vals[k].alloc(cap + 4));
    }
    s.tile_status_words = (size_t)MAX_PASSES * ((cap + SORT_TILE - 1) / SORT_TILE) * RADIX;
    CUDA_TRY(h, s.tile_status.alloc(s.tile_status_words));
    CUDA_TRY(h, s.P0.alloc(cap));
    CUDA_TRY(h, s.P1.alloc(cap));
    CUDA_TRY(h, s.P2.alloc(cap));
    CUDA_TRY(h, s.U.alloc(4 * (cap + 4)));
    CUDA_TRY(h, s.sorted_slot.alloc(cap));
    CUDA_TRY(h, s.sorted_id.alloc(cap));
    CUDA_TRY(h, s.cell_begin.alloc((size_t)s.cells_cap + 2));
    for (int k = 0; k < 2; ++k) {
        CUDA_TRY(h, s.qkeys[k].alloc(cap + 4));
        CUDA_TRY(h, s.qvals[k].alloc(cap + 4));
    }
    for (int k = 0; k < 2; ++k)  // (the twin exists once a delivery made it; the current set is bufs[0] until then)
        if (k == 0 || (like && like->bufs[k].out)) RC_TRY(alloc_frame_buffers(h, cap, max_pairs, s.bufs[k]));
    CUDA_TRY(h, s.cand_count.alloc(cap));
    // the fp32 stages forward about 5 candidate entries per emitted pair on clustered frames; a full
    // queue is not an error (the pair is then finished in place) but it is slower
    s.qcap = (u32)std::min<u64>(6 * max_pairs + 65536, (1ull << 31) - (1ull << 24));  // (32-bit entry indices)
    CUDA_TRY(h, s.q3.alloc(s.qcap));
    // the S1 filter forwards ~60 (predict) / ~20 (detect) pairs per object at the density of the bench frame;
    // the pair queue is handed out in blocks of QA_BLOCK entries, one per warp at a time
    // (+ one partly filled block per resident warp of k_pairs)
    s.qa_blocks_cap = (u32)(s.qcap / QA_BLOCK + 148 * 8 * PAIR_WARPS);
    CUDA_TRY(h, s.qa.alloc((size_t)s.qa_blocks_cap * QA_BLOCK));
    CUDA_TRY(h, s.qa_fill.alloc(s.qa_blocks_cap));
    s.items_cap = (u32)((cap / TQ + 1) * ITEMS_PER_TILE_CAP);  // k_tile_plan never makes more
    CUDA_TRY(h, s.items.alloc(s.items_cap));
    CUDA_TRY(h, s.tile_box.alloc(2 * (cap / TQ + 1)));
    CUDA_TRY(h, s.tile_rowx.alloc((size_t)TILE_ROWS * (cap / TQ + 1)));
    s.ovf_cap = s.items_cap;  // every work item is handed over at most once
    CUDA_TRY(h, s.ovf.alloc(s.ovf_cap));
    if (!like) return RCD_OK;
    if (like->compact_dev) CUDA_TRY(h, s.compact_dev.alloc(max_pairs));
    if (like->q_list) RC_TRY(alloc_queries(h, cap, s));
    if (like->traj_len) RC_TRY(alloc_history(h, cap, like->traj_len, on, s));
    if (like->last_seen) RC_TRY(alloc_last_seen(h, cap, on, s));
    return RCD_OK;
}

// A frame's totals reached the host: they size the next alert fold's grid, and fill `out` unless it is null.
void fill_counts(rcd_handle h, const Counters &c, u64 n, u64 n_owned, rcd_counts_t *out) {
    h->last_n_pairs = c.n_pairs;
    h->last_n_detect_end = c.n_detect_end;
    if (!out) return;
    out->n_objects = n;
    out->n_owned = n_owned;
    out->n_candidates = c.n_candidates;
    out->n_potential = c.n_potential;
    out->n_pairs = c.n_pairs;
    out->n_high_risk = c.n_high_risk;
    out->n_written = std::min<u64>(c.n_pairs, h->max_pairs);
    for (int k = 0; k < 4; ++k) out->n_alerts[k] = c.n_alerts[k];
    out->n_exact = c.n_exact;
    out->n_fallback = c.n_fallback;
}

void fill_alert_stats(const AlertCounters &c, rcd_alert_stats *st) {
    if (!st) return;
    st->n_events = c.n_events; st->n_created = c.n_created; st->n_changed = c.n_changed;
    st->n_refreshed = c.n_refreshed; st->n_expired = c.n_expired; st->n_live = c.n_live; st->n_dropped = c.n_dropped;
}

// Grid for a query radius.  The pair kernel and the radius queries walk the cells under the bounding box of
// their query volumes, so any cell size is exact (cell_coord is monotone); the x/y edge is a fraction of
// the query radius (finer cells = tighter boxes in dense regions, more rows per box), the z edge is the
// radius itself (the reference's worlds are ~100 m high).  Cells grow until the grid fits cells_cap.
GridParams make_grid(const float *wmin, const float *wmax, float cell_req, float cell_scale, u32 cells_cap) {
    GridParams g;
    double cell_z = (double)cell_req * 1.002 + 0.02;
    if (!(cell_z > 1e-3)) cell_z = 1e-3;
    double cell = cell_z * (double)cell_scale;
    if (!(cell > 1e-3)) cell = 1e-3;
    double ext[3];
    for (int d = 0; d < 3; ++d) {
        double e = (double)wmax[d] - (double)wmin[d];
        ext[d] = (e > 0 && std::isfinite(e)) ? e : 0.0;
    }
    for (;;) {
        double nx = std::floor(ext[0] / cell) + 1, ny = std::floor(ext[1] / cell) + 1, nz = std::floor(ext[2] / cell_z) + 1;
        if (nx * ny * nz <= (double)cells_cap) {
            g.nx = (int)nx; g.ny = (int)ny; g.nz = (int)nz;
            break;
        }
        cell *= 1.25;
        cell_z *= 1.25;
    }
    g.ox = wmin[0]; g.oy = wmin[1]; g.oz = wmin[2];
    g.cell = (float)cell;
    g.inv_cell = (float)(1.0 / cell);
    g.cell_z = (float)cell_z;
    g.inv_cell_z = (float)(1.0 / cell_z);
    g.ncells = (u32)g.nx * (u32)g.ny * (u32)g.nz;
    return g;
}

int key_passes(u32 ncells) {
    int bits = 1;
    while (bits < 32 && (1ull << bits) < (unsigned long long)ncells) ++bits;
    return std::max(1, (bits + RADIX_BITS - 1) / RADIX_BITS);
}

// Build the cell-ordered index for the current objects (keys -> sort -> reorder + ranges).
int build_index(rcd_handle h, float cell_req) {
    const u32 n = (u32)h->n;
    if (h->idx.valid && h->idx.cell_req == cell_req) return RCD_OK;
    h->idx.valid = false;
    h->idx.qorder_kind = 0;
    h->idx.slot_pos = false;
    RC_TRY(wait_upload(h));
    if (n == 0) {
        float z[3] = {0, 0, 0};
        h->idx.grid = make_grid(z, z, cell_req, h->cell_scale, h->cells_cap);
        h->idx.valid = true;
        h->idx.cell_req = cell_req;
        return RCD_OK;
    }
    if (!h->world_static) {
        h->bbox_host[0] = h->bbox_host[1] = h->bbox_host[2] = 0x7fffffff;
        h->bbox_host[3] = h->bbox_host[4] = h->bbox_host[5] = (int)0x80000000;
        CUDA_TRY(h, cudaMemcpyAsync(h->bbox_dev, h->bbox_host, 6 * sizeof(int), cudaMemcpyHostToDevice, h->stream));
        int blocks = (int)std::min<u64>((n + 255) / 256, 148 * 8);
        k_bbox<<<blocks, 256, 0, h->stream>>>(h->in_f[0], h->in_f[1], h->in_f[2], n, h->bbox_dev);
        KERNEL_CHECK(h);
        CUDA_TRY(h, cudaMemcpyAsync(h->bbox_host, h->bbox_dev, 6 * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        for (int d = 0; d < 3; ++d) {
            h->wmin[d] = ordered_float(h->bbox_host[d]);
            h->wmax[d] = ordered_float(h->bbox_host[3 + d]);
            if (!(h->wmin[d] <= h->wmax[d])) h->wmin[d] = h->wmax[d] = 0.0f;  // no finite coordinate
        }
    }
    h->idx.grid = make_grid(h->wmin, h->wmax, cell_req, h->cell_scale, h->cells_cap);
    const GridParams g = h->idx.grid;
    const int passes = key_passes(g.ncells + 1);  // + the cell of the objects without a position (rcd_index.cuh)
    const u32 tiles = (n + SORT_TILE - 1) / SORT_TILE;

    stage_begin(h, RCD_STAGE_KEYS);
    CUDA_TRY(h, cudaMemsetAsync(h->hist, 0, MAX_PASSES * RADIX * sizeof(u32), h->stream));
    CUDA_TRY(h, cudaMemsetAsync(h->tile_status, 0, (size_t)passes * tiles * RADIX * sizeof(u32), h->stream));
    CUDA_TRY(h, cudaMemsetAsync(h->tile_counter, 0, MAX_PASSES * sizeof(u32), h->stream));
    {
        int blocks = (int)std::min<u64>(((u64)n + KEYS_THREADS - 1) / KEYS_THREADS, 148 * 8);
        k_pack_keys<<<blocks, KEYS_THREADS, 0, h->stream>>>(input_state(h), n, (u32)h->n_owned, g, passes, h->keys[0],
                                                            h->hist, h->U);
        KERNEL_CHECK(h);
        k_scan_hist<<<1, RADIX, 0, h->stream>>>(h->hist, passes);
        KERNEL_CHECK(h);
    }
    stage_end(h, RCD_STAGE_KEYS);

    stage_begin(h, RCD_STAGE_SORT);
    u32 *const keys[2] = {h->keys[0], h->keys[1]}, *const vals[2] = {h->vals[0], h->vals[1]};
    const int cur = launch_onesweep(keys, vals, n, passes, h->hist, h->tile_status, h->tile_counter, h->stream);
    KERNEL_CHECK(h);
    h->idx.sorted_buf = cur;
    stage_end(h, RCD_STAGE_SORT);

    stage_begin(h, RCD_STAGE_REORDER);
    k_reorder<<<(n + REORDER_THREADS - 1) / REORDER_THREADS, REORDER_THREADS, 0, h->stream>>>(
        h->vals[cur], n, h->U, h->P0, h->P1, h->P2, h->sorted_slot, h->sorted_id);
    KERNEL_CHECK(h);
    RC_TRY(release_inputs(h));
    k_cell_table<<<(g.ncells + 1 + CT_CELLS - 1) / CT_CELLS, CT_THREADS, 0, h->stream>>>(h->keys[cur], n, g.ncells + 1, h->cell_begin);
    KERNEL_CHECK(h);
    stage_end(h, RCD_STAGE_REORDER);
    h->idx.valid = true;
    h->idx.cell_req = cell_req;
    return RCD_OK;
}

// Query order for the pair kernel (k_query_keys + the same onesweep passes): tiles of 32 queries whose
// volumes overlap.  kind 1: balls about the objects; kind 2: capsules of the predict queries.
// With a query list only the listed objects are keyed and sorted (k_query_keys_list): O(k) instead of O(n).
int build_query_order(rcd_handle h, int kind) {
    const u32 n = (u32)h->n;
    if (h->idx.qorder_kind == kind || n == 0) return RCD_OK;
    const GridParams g = h->idx.grid;
    const u32 nq = h->q_listed ? (u32)h->q_n : n;  // keys to sort
    const u32 tiles = (nq + SORT_TILE - 1) / SORT_TILE;
    stage_begin(h, RCD_STAGE_QORDER);
    CUDA_TRY(h, cudaMemsetAsync(h->hist, 0, MAX_PASSES * RADIX * sizeof(u32), h->stream));
    CUDA_TRY(h, cudaMemsetAsync(h->tile_status, 0, (size_t)QKEY_PASSES * tiles * RADIX * sizeof(u32), h->stream));
    CUDA_TRY(h, cudaMemsetAsync(h->tile_counter, 0, MAX_PASSES * sizeof(u32), h->stream));
    QueryKeyParams q;
    q.ox = g.ox; q.oy = g.oy;
    const double ex = std::max((double)g.nx * g.cell, 1e-3), ey = std::max((double)g.ny * g.cell, 1e-3);
    // QKEY_BITS bits for both axes, split so that the lattice cells are as square as they get (x-slabs are long in y)
    int bits_x = (int)std::floor(0.5 * (QKEY_BITS + std::log2(ex / ey)) + 0.5);
    bits_x = std::min(16, std::max(QKEY_BITS - 16, bits_x));
    const int bits_y = QKEY_BITS - bits_x;
    q.max_x = (float)((1u << bits_x) - 1u);
    q.max_y = (float)((1u << bits_y) - 1u);
    q.inv_res_x = (float)((double)(1u << bits_x) / ex);
    q.inv_res_y = (float)((double)(1u << bits_y) / ey);
    q.bits_lo = std::min(bits_x, bits_y);
    q.x_longer = bits_x > bits_y ? 1 : 0;
    q.capsule = kind == 2 ? 1 : 0;
    const int blocks = (int)std::min<u64>(((u64)nq + KEYS_THREADS - 1) / KEYS_THREADS, 148 * 8);
    if (h->q_listed) {
        if (!h->idx.slot_pos) {  // once per index build
            k_slot_pos<<<(n + 255) / 256, 256, 0, h->stream>>>(h->sorted_slot, n, h->q_pos);
            KERNEL_CHECK(h);
            h->idx.slot_pos = true;
        }
        k_query_keys_list<<<blocks, KEYS_THREADS, 0, h->stream>>>(h->P0, h->P1, h->P2, h->q_list, h->q_pos, nq, q,
                                                                   h->qkeys[0], h->qvals[0], h->hist);
    } else {
        k_query_keys<<<blocks, KEYS_THREADS, 0, h->stream>>>(h->P0, h->P1, h->P2, n, q, h->qkeys[0], h->hist);
    }
    KERNEL_CHECK(h);
    k_scan_hist<<<1, RADIX, 0, h->stream>>>(h->hist, QKEY_PASSES);
    KERNEL_CHECK(h);
    u32 *const keys[2] = {h->qkeys[0], h->qkeys[1]}, *const vals[2] = {h->qvals[0], h->qvals[1]};
    const int cur = launch_onesweep(keys, vals, nq, QKEY_PASSES, h->hist, h->tile_status, h->tile_counter, h->stream,
                                    !h->q_listed);
    KERNEL_CHECK(h);
    stage_end(h, RCD_STAGE_QORDER);
    h->idx.q_sorted_buf = cur;
    h->idx.qorder_kind = kind;
    return RCD_OK;
}

int copy_in(rcd_handle h, void *dst, const void *src, size_t bytes, int32_t srckind, cudaStream_t on) {
    CUDA_TRY(h, cudaMemcpyAsync(dst, src, bytes, srckind == RCD_SRC_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, on));
    return RCD_OK;
}

// The stream an upload of kind `src` runs on.  Host memory: the upload stream, after the previous frame has
// released the upload buffers.  Device memory: the handle's stream (ordered after a pending host upload).
int upload_stream(rcd_handle h, int32_t src, cudaStream_t *on) {
    if (src == RCD_SRC_DEVICE) {
        RC_TRY(wait_upload(h));
        *on = h->stream;
        return RCD_OK;
    }
    if (h->inputs_busy) {
        CUDA_TRY(h, cudaStreamWaitEvent(h->up_stream, h->ev_inputs_free, 0));
        h->inputs_busy = false;
    }
    *on = h->up_stream;
    return RCD_OK;
}
int upload_issued(rcd_handle h, cudaStream_t on) {
    if (on == h->up_stream) {
        CUDA_TRY(h, cudaEventRecord(h->ev_upload_done, h->up_stream));
        h->upload_pending = true;
        return RCD_OK;
    }
    return release_inputs(h);  // written on the handle's stream: a later host upload must come after it
}

}  // namespace

extern "C" {

int rcd_version(void) { return RCD_VERSION; }

const char *rcd_last_error(rcd_handle h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int rcd_create(const rcd_config *cfg, rcd_handle *out) {
    if (!cfg || !out) return fail(nullptr, RCD_EINVAL, "rcd_create: null argument");
    *out = nullptr;
    if (cfg->max_objects == 0 || cfg->max_objects >= (1ull << 30))
        return fail(nullptr, RCD_EINVAL, "rcd_create: max_objects must be in [1, 2^30)");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || cfg->device < 0 || cfg->device >= ndev) {
        (void)cudaGetLastError();
        return fail(nullptr, RCD_ENODEVICE, "rcd_create: no usable CUDA device (this library has no CPU fallback)");
    }
    std::unique_ptr<rcd_handle_s> h(new (std::nothrow) rcd_handle_s());  // (a failed create frees what it made)
    if (!h) return fail(nullptr, RCD_ENOMEM, "rcd_create: out of host memory");
    h->device = cfg->device;
    h->flags = cfg->flags;
    h->world_static = cfg->world_min[0] <= cfg->world_max[0];
    for (int d = 0; d < 3; ++d) { h->wmin[d] = cfg->world_min[d]; h->wmax[d] = cfg->world_max[d]; }

    CUDA_TRY(nullptr, cudaSetDevice(h->device));
    {
        int sms = 0;
        CUDA_TRY(nullptr, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device));
        h->sms = std::max(1, sms);
    }
    {   // the frame's stream outranks the alert stream: block slots go to the frame's kernels first
        int least = 0, greatest = 0;
        CUDA_TRY(nullptr, cudaDeviceGetStreamPriorityRange(&least, &greatest));
        CUDA_TRY(nullptr, h->stream.create(greatest));
    }
    CUDA_TRY(nullptr, h->up_stream.create());
    CUDA_TRY(nullptr, h->ev_upload_done.create());
    CUDA_TRY(nullptr, h->ev_inputs_free.create());
    RC_TRY(size_buffers(nullptr, cfg->max_objects, std::max<u64>(cfg->max_pairs, 1), nullptr, h->stream, *h));
    CUDA_TRY(nullptr, h->hist.alloc(MAX_PASSES * RADIX));
    CUDA_TRY(nullptr, h->tile_counter.alloc(MAX_PASSES));
    if (const char *e = getenv("RCD_CELL_SCALE")) {  // kernel-tuning experiments only
        const double v = atof(e);
        if (v >= 0.05 && v <= 4.0) h->cell_scale = (float)v;
    }
    CUDA_TRY(nullptr, h->bbox_dev.alloc(6));
    CUDA_TRY(nullptr, h->bbox_host.alloc(6));
    CUDA_TRY(nullptr, h->counters_host.alloc());
    CUDA_TRY(nullptr, h->pair_tile_counter.alloc(2));
    for (auto &mode : h->stages)
        for (Stage &st : mode) {
            CUDA_TRY(nullptr, st.begin.create(cudaEventDefault));
            CUDA_TRY(nullptr, st.end.create(cudaEventDefault));
        }
    CUDA_TRY(nullptr, cudaStreamSynchronize(h->stream));
    *out = h.release();
    return RCD_OK;
}

int rcd_destroy(rcd_handle h) {
    delete h;
    return RCD_OK;
}

int rcd_reserve(rcd_handle h, uint64_t max_objects, uint64_t max_pairs) {
    if (!h) return RCD_EINVAL;
    if (max_objects >= (1ull << 30)) return fail(h, RCD_EINVAL, "rcd_reserve: max_objects must be below 2^30");
    const u64 cap = std::max<u64>(h->cap, max_objects), pairs = std::max<u64>(h->max_pairs, max_pairs);
    if (cap == h->cap && pairs == h->max_pairs) return RCD_OK;
    if (h->download_pending) return fail(h, RCD_ESTATE, "rcd_reserve: a delivery is in flight");
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaStreamSynchronize(h->up_stream));
    if (h->dl.alert_stream) CUDA_TRY(h, cudaStreamSynchronize(h->dl.alert_stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    Sized s;
    int rc = size_buffers(h, cap, pairs, h, h->stream, s);
    // the state the handle keeps: the first n slots of every per-object buffer, the query list
    const size_t n = (size_t)h->n;
    auto check = [&](cudaError_t e) {
        if (rc == RCD_OK && e != cudaSuccess) rc = fail(h, RCD_ECUDA, std::string("rcd_reserve: ") + cudaGetErrorString(e));
    };
    auto copy = [&](void *dst, const void *src, size_t bytes) {
        if (rc == RCD_OK && bytes) check(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, h->stream));
    };
    for (int k = 0; k < 11; ++k) copy(s.in_f[k], h->in_f[k], n * sizeof(float));
    copy(s.in_type, h->in_type, n);
    copy(s.in_pattern, h->in_pattern, n);
    copy(s.in_id, h->in_id, n * sizeof(u32));
    if (h->traj_len) {
        copy(s.traj_count, h->traj_count, n * sizeof(u32));
        if (rc == RCD_OK && n)  // sample-major rings [traj_len][cap]: the row pitch grows with the capacity
            check(cudaMemcpy2DAsync(s.traj, cap * sizeof(Sample64), h->traj, h->cap * sizeof(Sample64), n * sizeof(Sample64),
                                    h->traj_len, cudaMemcpyDeviceToDevice, h->stream));
    }
    if (h->last_seen) copy(s.last_seen, h->last_seen, n * sizeof(double));
    if (h->q_listed) copy(s.q_list, h->q_list, (size_t)h->q_n * sizeof(u32));
    // swap only a complete set, and only when nothing in flight touches either set any more
    check(cudaStreamSynchronize(h->stream));
    if (rc != RCD_OK) {
        (void)cudaGetLastError();  // (a refused allocation is not a fault of the handle)
        return rc;
    }
    static_cast<Sized &>(*h) = std::move(s);
    // the index, the frame and every captured step graph referred to the old buffers
    h->idx = IndexState{};
    h->frame_done = false;
    for (StepGraph &g : h->graphs) g = StepGraph{};
    for (StepKey &k : h->graph_candidates) k = StepKey{};
    return RCD_OK;
}

int rcd_upload(rcd_handle h, uint64_t n, const float *px, const float *py, const float *pz, const float *vx,
               const float *vy, const float *vz, const float *ax, const float *ay, const float *az,
               const float *size, const float *heading, const uint8_t *type, const uint32_t *id, int32_t src) {
    if (!h) return RCD_EINVAL;
    if (n > h->cap) return fail(h, RCD_ECAPACITY, "rcd_upload: n exceeds max_objects");
    if (n && (!px || !py || !pz || !vx || !vy || !vz)) return fail(h, RCD_EINVAL, "rcd_upload: position/velocity arrays are required");
    CUDA_TRY(h, cudaSetDevice(h->device));
    reset_stages(h, -1);
    h->stage_mode = 0;
    cudaStream_t on = nullptr;
    RC_TRY(upload_stream(h, src, &on));
    stage_begin(h, RCD_STAGE_UPLOAD, on);
    const float *f[11] = {px, py, pz, vx, vy, vz, ax, ay, az, size, heading};
    const size_t bytes = (size_t)n * sizeof(float);
    for (int k = 0; k < 11 && n; ++k) {
        if (f[k]) {
            RC_TRY(copy_in(h, h->in_f[k], f[k], bytes, src, on));
        } else {
            CUDA_TRY(h, cudaMemsetAsync(h->in_f[k], 0, bytes, on));
        }
    }
    if (n) {
        if (type) RC_TRY(copy_in(h, h->in_type, type, (size_t)n, src, on));
        else CUDA_TRY(h, cudaMemsetAsync(h->in_type, 0, (size_t)n, on));
        CUDA_TRY(h, cudaMemsetAsync(h->in_pattern, RCD_PAT_ACCELERATING, (size_t)n, on));
        if (id) RC_TRY(copy_in(h, h->in_id, id, (size_t)n * sizeof(u32), src, on));
        else {
            k_iota<<<(unsigned)((n + 255) / 256), 256, 0, on>>>(h->in_id, (u32)n);
            KERNEL_CHECK(h);
        }
    }
    stage_end(h, RCD_STAGE_UPLOAD, on);
    RC_TRY(upload_issued(h, on));
    h->n = n;
    h->n_owned = n;
    h->records_only = n == 0;
    h->q_listed = false;
    h->idx.valid = false;
    h->frame_done = false;
    return RCD_OK;
}

int rcd_set_patterns(rcd_handle h, uint64_t n, const uint8_t *pattern, int32_t src) {
    if (!h) return RCD_EINVAL;
    if (n > h->n) return fail(h, RCD_EINVAL, "rcd_set_patterns: n exceeds the uploaded object count");
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (n) {
        cudaStream_t on = nullptr;
        RC_TRY(upload_stream(h, pattern ? src : RCD_SRC_HOST, &on));
        if (pattern) RC_TRY(copy_in(h, h->in_pattern, pattern, (size_t)n, src, on));
        else CUDA_TRY(h, cudaMemsetAsync(h->in_pattern, RCD_PAT_ACCELERATING, (size_t)n, on));
        RC_TRY(upload_issued(h, on));
    }
    h->idx.valid = false;  // the pattern is packed into the cell-ordered state
    h->frame_done = false;
    return RCD_OK;
}

int rcd_set_owned(rcd_handle h, uint64_t n_owned) {
    if (!h) return RCD_EINVAL;
    if (n_owned > h->n) return fail(h, RCD_EINVAL, "rcd_set_owned: n_owned exceeds the object count");
    h->n_owned = n_owned;
    h->q_listed = false;
    h->idx.valid = false;
    h->frame_done = false;
    return RCD_OK;
}

// the list, inverse-map, bitmap and staging buffers of rcd_set_queries (all or nothing)
static int queries_ready(rcd_handle h) {
    if (h->q_list) return RCD_OK;
    Sized s;
    Event copied;
    RC_TRY(alloc_queries(h, h->cap, s));
    CUDA_TRY(h, copied.create());
    h->q_list = std::move(s.q_list);
    h->q_pos = std::move(s.q_pos);
    h->q_seen = std::move(s.q_seen);
    h->q_host = std::move(s.q_host);
    h->q_copied = std::move(copied);
    return RCD_OK;
}

int rcd_set_queries(rcd_handle h, uint64_t n, const uint32_t *slots, int32_t src) {
    if (!h) return RCD_EINVAL;
    if (!slots) {
        if (h->q_listed) h->idx.qorder_kind = 0;
        h->q_listed = false;
        h->frame_done = false;
        return RCD_OK;
    }
    const u64 owned = h->n_owned;
    if (n > owned) return fail(h, RCD_EINVAL, "rcd_set_queries: more slots than owned objects");
    CUDA_TRY(h, cudaSetDevice(h->device));
    RC_TRY(queries_ready(h));
    if (n && src == RCD_SRC_DEVICE) {
        const u64 words = (owned + 31) / 32;
        u32 *const err = h->q_seen.get() + words;
        CUDA_TRY(h, cudaMemsetAsync(h->q_seen, 0, (words + 1) * sizeof(u32), h->stream));
        k_check_queries<<<(unsigned)std::min<u64>((n + 255) / 256, (u64)h->sms * 8), 256, 0, h->stream>>>(
            slots, (u32)n, (u32)owned, h->q_seen, err);
        KERNEL_CHECK(h);
        u32 bad = 0;
        CUDA_TRY(h, cudaMemcpyAsync(&bad, err, sizeof(u32), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        if (bad & 1u) return fail(h, RCD_EINVAL, "rcd_set_queries: a slot is not an owned object");
        if (bad & 2u) return fail(h, RCD_EINVAL, "rcd_set_queries: a slot is listed twice");
        CUDA_TRY(h, cudaMemcpyAsync(h->q_list, slots, (size_t)n * sizeof(u32), cudaMemcpyDeviceToDevice, h->stream));
    } else if (n) {
        std::vector<uint64_t> seen((size_t)((owned + 63) / 64), 0);
        for (u64 t = 0; t < n; ++t) {
            const u32 s = slots[t];
            if (s >= owned) return fail(h, RCD_EINVAL, "rcd_set_queries: slot " + std::to_string(s) + " is not an owned object");
            const uint64_t bit = 1ull << (s & 63u);
            if (seen[s >> 6] & bit) return fail(h, RCD_EINVAL, "rcd_set_queries: slot " + std::to_string(s) + " is listed twice");
            seen[s >> 6] |= bit;
        }
        // (the previous list's copy out of the pinned buffer has to be done before it is overwritten)
        CUDA_TRY(h, cudaEventSynchronize(h->q_copied));
        std::memcpy(h->q_host.get(), slots, (size_t)n * sizeof(u32));
        CUDA_TRY(h, cudaMemcpyAsync(h->q_list, h->q_host, (size_t)n * sizeof(u32), cudaMemcpyHostToDevice, h->stream));
        CUDA_TRY(h, cudaEventRecord(h->q_copied, h->stream));
    }
    h->q_listed = true;
    h->q_n = n;
    h->idx.qorder_kind = 0;  // the index stays; only the query order is rebuilt
    h->frame_done = false;
    return RCD_OK;
}

static int step_impl(rcd_handle h, int32_t mode, float search_radius, float time_window) {
    if (!h) return RCD_EINVAL;
    const bool append = (mode & RCD_STEP_APPEND) != 0;
    const bool with_detect = (mode & RCD_STEP_WITH_DETECT) != 0;
    mode &= ~(RCD_STEP_APPEND | RCD_STEP_WITH_DETECT);
    if (mode < RCD_MODE_DETECT || mode > RCD_MODE_COMPUTE_NODE) return fail(h, RCD_EINVAL, "rcd_step: unknown mode");
    if (with_detect && mode != RCD_MODE_PREDICT) return fail(h, RCD_EINVAL, "rcd_step: RCD_STEP_WITH_DETECT goes with RCD_MODE_PREDICT");
    bool fused = false;
    if (with_detect) {
        fused = search_radius == PREDICT_RADIUS && time_window == 10.0f && !(h->flags & RCD_FLAG_COUNT_PREDICT_CANDIDATES);
        if (!fused) {  // other parameters: the two passes back to back
            RC_TRY(step_impl(h, RCD_MODE_DETECT | (append ? RCD_STEP_APPEND : 0), search_radius, time_window));
            return step_impl(h, RCD_MODE_PREDICT | RCD_STEP_APPEND, search_radius, time_window);
        }
    }
    if (append && !h->frame_done) return fail(h, RCD_ESTATE, "rcd_step: RCD_STEP_APPEND needs a previous step of this frame");
    if (!(search_radius > 0.0f) || !std::isfinite(search_radius)) return fail(h, RCD_EINVAL, "rcd_step: search_radius must be positive");
    if (mode == RCD_MODE_DETECT && !(time_window >= 0.0f)) return fail(h, RCD_EINVAL, "rcd_step: time_window must be >= 0");
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (!append) h->launches = 0;
    if (!append && h->flip_pending) h->flip();
    h->frame_done = false;
    h->stage_mode = mode;
    reset_stages(h, mode);
    stage_begin(h, RCD_STAGE_TOTAL);
    const float cell_req = (mode == RCD_MODE_PREDICT) ? PREDICT_RADIUS : search_radius;
    RC_TRY(build_index(h, cell_req));

    if (h->n && h->queried()) {
        RC_TRY(build_query_order(h, mode == RCD_MODE_PREDICT ? 2 : 1));
    }
    stage_begin(h, RCD_STAGE_PAIRS);
    if (!append) CUDA_TRY(h, cudaMemsetAsync(h->fb().counters, 0, sizeof(Counters), h->stream));
    if (h->n) CUDA_TRY(h, cudaMemsetAsync(h->cand_count, 0, (size_t)h->n * sizeof(u32), h->stream));
    if (h->n && !append) CUDA_TRY(h, cudaMemsetAsync(h->fb().risk_count, 0, (size_t)h->n * sizeof(u32), h->stream));
    if (h->n && h->queried()) {
        PairParams P;
        P.n = (u32)h->n;
        P.n_owned = (u32)h->queried();
        P.g = h->idx.grid;
        P.P0 = h->P0; P.P1 = h->P1; P.P2 = h->P2;
        P.qorder = h->qvals[h->idx.q_sorted_buf];
        P.sorted_slot = h->sorted_slot;
        P.sorted_id = h->sorted_id;
        P.cell_begin = h->cell_begin;
        P.R = search_radius;
        P.T = time_window;
        P.steps = (int)((double)time_window / 0.1);  // int(time_window / time_step), collision_detection.py:322
        P.pt = h->cn_prediction_time;  // CollisionDetector(prediction_time=5.0, risk_threshold=0.5), compute_node.py:218
        P.threshold = h->cn_risk_threshold;
        // T1 window of the S1 filter: detect looks at [0, time_window]; the predict modes at [0, 10] (offsets up
        // to 9.5 s, and detect_collisions(100, 10) for objects without history / the fused detect pass)
        if (mode == RCD_MODE_DETECT) {
            P.tm = P.D = 0.5f * time_window;
            P.use_t1 = 1;
        } else {
            P.tm = P.D = 5.0f;
            P.use_t1 = mode == RCD_MODE_PREDICT ? 1 : 0;
        }
        P.D *= 1.0f + 1.0e-6f;
        P.out = h->fb().out;
        P.out_cap = h->max_pairs;
        P.counters = h->fb().counters;
        P.cand_count = h->cand_count;
        P.risk_count = h->fb().risk_count;
        P.ntiles = (u32)((P.n_owned + TQ - 1) / TQ);
        P.tile_counter = h->pair_tile_counter;
        P.qa = h->qa; P.qa_fill = h->qa_fill; P.qa_blocks_cap = h->qa_blocks_cap;
        P.ovf = h->ovf; P.ovf_cap = h->ovf_cap;
        P.items = h->items; P.items_cap = h->items_cap; P.tile_box = h->tile_box; P.tile_rowx = h->tile_rowx;
        // work items of about 16 chunks (16 k pair tests per lane-pass); small frames get smaller items so that
        // every resident warp finds work
        P.item_chunks = P.ntiles >= 16384 ? 16u : P.ntiles >= 4096 ? 8u : P.ntiles >= 1024 ? 4u : P.ntiles >= 256 ? 2u : 1u;
        P.q3 = h->q3; P.qcap = h->qcap;
        P.q3_split = mode == RCD_MODE_PREDICT ? h->qcap / 4 : h->qcap;
        CUDA_TRY(h, cudaMemsetAsync(h->pair_tile_counter, 0, 2 * sizeof(u32), h->stream));
        CUDA_TRY(h, cudaMemsetAsync(&h->fb().counters->n_qa_blocks, 0, 6 * sizeof(unsigned long long), h->stream));
        const bool count = (h->flags & RCD_FLAG_COUNT_PREDICT_CANDIDATES) != 0;
        // persistent launch: as many blocks as can be resident, warps pull tiles from a counter
        const int variant = fused ? 4 : mode == RCD_MODE_DETECT ? 0 : (mode == RCD_MODE_COMPUTE_NODE ? 3 : (count ? 2 : 1));
        const FrameKernels &K = FRAME_KERNELS[variant];
        if (h->pair_blocks[variant] == 0) {
            int per_sm = 0;
            CUDA_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, K.pairs, PAIR_THREADS, 0));
            h->pair_blocks[variant] = std::max(1, per_sm) * h->sms;
            CUDA_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, K.narrow, STAGE_THREADS, 0));
            h->narrow_blocks[variant] = std::max(1, per_sm) * h->sms;
        }
        // plan: the tiles' cell boxes and work items of even size; then the persistent pair kernel
        const unsigned pb = (unsigned)std::min<u64>((P.ntiles + 3) / 4, (u64)h->sms * 8);
        K.tile_plan<<<pb, 128, 0, h->stream>>>(P);
        KERNEL_CHECK(h);
        const u64 items = (u64)P.ntiles * PLAN_ITEMS_PER_TILE;  // (upper estimate: the grid is capped by residency)
        const unsigned blocks = (unsigned)std::min<u64>((items + PAIR_WARPS - 1) / PAIR_WARPS, (u64)h->pair_blocks[variant]);
        // the regular pass, then the overflow pass (returns at once unless the pair queue ran out)
        const unsigned oblocks = std::min(blocks, (unsigned)h->sms * 4u);
        K.pairs<<<blocks, PAIR_THREADS, 0, h->stream>>>(P);
        K.pairs_overflow<<<oblocks, PAIR_THREADS, 0, h->stream>>>(P);
        ++h->launches;
        KERNEL_CHECK(h);
        stage_end(h, RCD_STAGE_PAIRS);
        // the later stages read their queue lengths on the device: fixed grids, no host round trip
        stage_begin(h, RCD_STAGE_NARROW);
        const unsigned nb = (unsigned)std::min<u64>((u64)h->narrow_blocks[variant], (u64)P.ntiles * 8 / STAGE_WARPS + 1);
        K.narrow<<<nb, STAGE_THREADS, 0, h->stream>>>(P);
        KERNEL_CHECK(h);
        stage_end(h, RCD_STAGE_NARROW);
        const unsigned sb = (unsigned)std::min<u64>((u64)h->sms * 8, (h->n + STAGE_THREADS - 1) / STAGE_THREADS + 1);
        stage_begin(h, RCD_STAGE_EXACT);
        K.exact<<<sb, STAGE_THREADS, 0, h->stream>>>(P);
        KERNEL_CHECK(h);
        // every record with predicted = 0 has been emitted by now (overflow passes, in-place fall-backs, detect entries):
        // the alert fold's detect pass stops here instead of walking the whole buffer
        CUDA_TRY(h, cudaMemcpyAsync(&h->fb().counters->n_detect_end, &h->fb().counters->n_pairs, sizeof(unsigned long long),
                                    cudaMemcpyDeviceToDevice, h->stream));
        if (K.exact_resolved) K.exact_resolved<<<sb, STAGE_THREADS, 0, h->stream>>>(P);
        KERNEL_CHECK(h);  // (counted with or without the RESOLVED pass)
        stage_end(h, RCD_STAGE_EXACT);
    } else {
        stage_end(h, RCD_STAGE_PAIRS);
    }
    stage_end(h, RCD_STAGE_TOTAL);
    h->frame_done = true;
    h->last_mode = mode;
    return RCD_OK;
}

// The graph key of a step: the index fields count only while the index is valid (q_sorted_buf only with a query
// order), and `out` is the pair buffer the step will write, after a pending flip.
static StepKey step_key(rcd_handle h, int32_t mode, float search_radius, float time_window, bool append, bool flip) {
    const IndexState &ix = h->idx;
    StepKey key;
    key.mode = mode; key.R = search_radius; key.T = time_window;
    key.pt = h->cn_prediction_time; key.thr = h->cn_risk_threshold;
    key.n = h->n; key.n_owned = h->queried();
    key.listed = h->q_listed ? 1 : 0;
    key.slot_pos = (ix.valid && ix.slot_pos) ? 1 : 0;
    key.index_valid = ix.valid ? 1 : 0;
    key.index_cell_req = ix.valid ? ix.cell_req : 0.0f;
    key.sorted_buf = ix.valid ? ix.sorted_buf : 0;
    key.qorder_kind = ix.valid ? ix.qorder_kind : 0;
    key.q_sorted_buf = (ix.valid && ix.qorder_kind) ? ix.q_sorted_buf : 0;
    key.frame_done = append ? (h->frame_done ? 1 : 0) : 0;
    key.out = h->bufs[flip ? h->cur ^ 1 : h->cur].out.get();
    return key;
}

// RCD_FLAG_GRAPH: the launch sequence of a step is a pure function of its StepKey.  First sighting of a key: run
// normally and remember it; second sighting in a row: capture, instantiate, launch; from then on: one graph
// launch plus the host-side state changes step_impl would have made.
int rcd_step(rcd_handle h, int32_t mode, float search_radius, float time_window) {
    if (!h) return RCD_EINVAL;
    const bool want = (h->flags & RCD_FLAG_GRAPH) && !(h->flags & RCD_FLAG_PROFILE) && h->world_static && !h->graph_broken &&
                      h->n > 0 && h->queried() > 0;
    if (!want) return step_impl(h, mode, search_radius, time_window);
    const bool append = (mode & RCD_STEP_APPEND) != 0;
    const bool flip = !append && h->flip_pending;
    {   // (events of other streams stay outside the graph: order the stream before the launch / the capture)
        CUDA_TRY(h, cudaSetDevice(h->device));
        RC_TRY(wait_upload(h));
    }
    const StepKey key = step_key(h, mode, search_radius, time_window, append, flip);
    for (auto &g : h->graphs) {
        if (!g.exec || !(g.key == key)) continue;
        // ---- replay ----
        CUDA_TRY(h, cudaSetDevice(h->device));
        if (flip) h->flip();
        h->frame_done = false;
        CUDA_TRY(h, cudaGraphLaunch(g.exec, h->stream));
        RC_TRY(release_inputs(h));  // (at the end of the step: a graph has no events inside)
        h->launches = (append ? h->launches : 0) + g.launches;
        h->idx = g.idx;
        h->stage_mode = g.last_mode;
        h->last_mode = g.last_mode;
        h->frame_done = true;
        ++h->graph_replays;
        return RCD_OK;
    }
    bool seen = false;
    for (auto &c : h->graph_candidates) seen = seen || c == key;
    if (!seen) {  // first sighting: run it, remember it
        h->graph_candidates[h->graph_cand_next] = key;
        h->graph_cand_next = (h->graph_cand_next + 1) % 4;
        return step_impl(h, mode, search_radius, time_window);
    }
    // ---- second sighting: capture ----
    CUDA_TRY(h, cudaSetDevice(h->device));
    struct Saved {
        IndexState idx;
        int cur, last_mode, stage_mode;
        bool flip_pending, frame_done;
        u64 launches;
    };
    const Saved pre = {h->idx, h->cur, h->last_mode, h->stage_mode, h->flip_pending, h->frame_done, h->launches};
    auto restore = [&]() {
        h->idx = pre.idx; h->cur = pre.cur; h->last_mode = pre.last_mode; h->stage_mode = pre.stage_mode;
        h->flip_pending = pre.flip_pending; h->frame_done = pre.frame_done; h->launches = pre.launches;
    };
    cudaGraph_t graph = nullptr;
    GraphExec exec;
    cudaError_t e = cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal);
    int rc = RCD_OK;
    if (e == cudaSuccess) {
        h->capturing = true;
        rc = step_impl(h, mode, search_radius, time_window);
        h->capturing = false;
        cudaError_t e2 = cudaStreamEndCapture(h->stream, &graph);
        if (e2 != cudaSuccess) e = e2;
    }
    if (e == cudaSuccess && rc == RCD_OK && graph) e = exec.instantiate(graph);
    if (graph) cudaGraphDestroy(graph);
    if (e != cudaSuccess || rc != RCD_OK || !exec) {  // not capturable here: never try again, run the step for real
        (void)cudaGetLastError();
        exec.reset();
        restore();
        h->graph_broken = true;
        return step_impl(h, mode, search_radius, time_window);
    }
    e = cudaGraphLaunch(exec, h->stream);
    if (e != cudaSuccess) {
        exec.reset();
        restore();
        h->graph_broken = true;
        return step_impl(h, mode, search_radius, time_window);
    }
    RC_TRY(release_inputs(h));
    StepGraph &slot = h->graphs[h->graph_next];
    h->graph_next = (h->graph_next + 1) % 4;
    slot.exec = std::move(exec);  // (releases the graph the slot held)
    slot.key = key;
    slot.idx = h->idx;
    slot.last_mode = h->last_mode;
    slot.launches = h->launches - (append ? pre.launches : 0);
    return RCD_OK;
}

int rcd_graph_replays(rcd_handle h, uint64_t *n) {
    if (!h || !n) return RCD_EINVAL;
    *n = h->graph_replays;
    return RCD_OK;
}

int rcd_set_compute_node_params(rcd_handle h, float prediction_time, float risk_threshold) {
    if (!h) return RCD_EINVAL;
    if (!(prediction_time >= 0.0f) || !std::isfinite(prediction_time) || !std::isfinite(risk_threshold))
        return fail(h, RCD_EINVAL, "rcd_set_compute_node_params: bad parameter");
    h->cn_prediction_time = prediction_time;
    h->cn_risk_threshold = risk_threshold;
    h->frame_done = false;
    return RCD_OK;
}

int rcd_truncate(rcd_handle h, uint64_t n) {
    if (!h) return RCD_EINVAL;
    if (n > h->n) return fail(h, RCD_EINVAL, "rcd_truncate: n exceeds the object count");
    h->n = n;
    h->n_owned = n;
    h->q_listed = false;
    h->idx.valid = false;
    h->frame_done = false;
    return RCD_OK;
}

int rcd_invalidate(rcd_handle h) {
    if (!h) return RCD_EINVAL;
    h->idx.valid = false;
    h->frame_done = false;
    return RCD_OK;
}

int rcd_build_index(rcd_handle h, float cell_radius) {
    if (!h) return RCD_EINVAL;
    if (!(cell_radius > 0.0f) || !std::isfinite(cell_radius)) return fail(h, RCD_EINVAL, "rcd_build_index: bad radius");
    CUDA_TRY(h, cudaSetDevice(h->device));
    h->launches = 0;
    h->stage_mode = RCD_MODE_DETECT;
    reset_stages(h, RCD_MODE_DETECT);
    stage_begin(h, RCD_STAGE_TOTAL);
    int rc = build_index(h, cell_radius);
    stage_end(h, RCD_STAGE_TOTAL);
    return rc;
}

int rcd_counts(rcd_handle h, rcd_counts_t *out) {
    if (!h || !out) return RCD_EINVAL;
    if (!h->frame_done) return fail(h, RCD_ESTATE, "rcd_counts: no frame has been stepped");
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaMemcpyAsync(h->counters_host, h->fb().counters, sizeof(Counters), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    fill_counts(h, *h->counters_host, h->n, h->queried(), out);
    return RCD_OK;
}

static int download_impl(rcd_handle h, rcd_pair *out, uint64_t cap, uint64_t *n_out, bool sorted) {
    if (!h || !n_out || (cap && !out)) return RCD_EINVAL;
    rcd_counts_t c;
    RC_TRY(rcd_counts(h, &c));
    h->stage_mode = 0;
    stage_begin(h, RCD_STAGE_DOWNLOAD);
    u64 m = std::min<u64>(c.n_written, cap);
    if (m) {
        CUDA_TRY(h, cudaMemcpyAsync(out, h->fb().out, (size_t)m * sizeof(rcd_pair), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        if (sorted) {
            // sort 16-byte (key, index) records instead of the 48-byte pairs, then permute once
            struct KeyIdx { u64 key; u32 idx; u32 sub; };
            std::vector<KeyIdx> keys((size_t)m);
            for (u64 k = 0; k < m; ++k) keys[k] = {((u64)out[k].i << 32) | out[k].j, (u32)k, out[k].predicted};
            std::sort(keys.begin(), keys.end(), [](const KeyIdx &a, const KeyIdx &b) {
                return a.key != b.key ? a.key < b.key : a.sub < b.sub;
            });
            std::vector<rcd_pair> tmp(out, out + m);
            for (u64 k = 0; k < m; ++k) out[k] = tmp[keys[k].idx];
        }
    }
    stage_end(h, RCD_STAGE_DOWNLOAD);
    *n_out = m;
    return RCD_OK;
}

int rcd_download(rcd_handle h, rcd_pair *out, uint64_t cap, uint64_t *n_out) {
    return download_impl(h, out, cap, n_out, true);
}

int rcd_download_unsorted(rcd_handle h, rcd_pair *out, uint64_t cap, uint64_t *n_out) {
    return download_impl(h, out, cap, n_out, false);
}

// twin buffers + copy stream of the pipelined deliveries (made at the first use, all or nothing)
static int delivery_ready(rcd_handle h) {
    if (h->dl.pend_event) return RCD_OK;
    FrameBuffers twin;
    Delivery d;
    RC_TRY(alloc_frame_buffers(h, h->cap, h->max_pairs, twin));
    CUDA_TRY(h, d.counters_host.alloc());
    CUDA_TRY(h, d.alert_counters_host.alloc());
    CUDA_TRY(h, d.copy_stream.create());
    CUDA_TRY(h, d.pend_event.create());
    {
        int least = 0, greatest = 0;
        CUDA_TRY(h, cudaDeviceGetStreamPriorityRange(&least, &greatest));
        CUDA_TRY(h, d.alert_stream.create(least));
    }
    CUDA_TRY(h, d.ev_frame_done.create());
    CUDA_TRY(h, d.ev_alert_done.create());
    h->bufs[h->cur ^ 1] = std::move(twin);
    h->dl = std::move(d);
    return RCD_OK;
}
// Order the handle's stream after the alert-table work a summary delivery left on alert_stream.
static int alerts_join(rcd_handle h) {
    if (h->alert_async) {
        CUDA_TRY(h, cudaStreamWaitEvent(h->stream, h->dl.ev_alert_done, 0));
        h->alert_async = false;
    }
    return RCD_OK;
}
static int delivery_begin(rcd_handle h, const char *who) {
    if (!h->frame_done) return fail(h, RCD_ESTATE, std::string(who) + ": no frame has been stepped");
    if (h->download_pending) return fail(h, RCD_ESTATE, std::string(who) + ": a delivery is already in flight");
    CUDA_TRY(h, cudaSetDevice(h->device));
    return delivery_ready(h);
}
static int delivery_issued(rcd_handle h, cudaStream_t on = nullptr) {  // the frame's totals ride along; later work goes to the twin buffers
    if (!on) on = h->stream;
    CUDA_TRY(h, cudaMemcpyAsync(h->dl.counters_host, h->fb().counters, sizeof(Counters), cudaMemcpyDeviceToHost, on));
    CUDA_TRY(h, cudaEventRecord(h->dl.pend_event, on));
    h->pend_dev = h->fb().out;
    h->pend_risk = h->fb().risk_count;
    h->pend_n = h->n;
    h->pend_n_owned = h->queried();
    h->download_pending = true;
    h->flip_pending = true;
    return RCD_OK;
}

int rcd_download_begin(rcd_handle h, rcd_pair *out, uint64_t cap) {
    if (!h || (cap && !out)) return RCD_EINVAL;
    RC_TRY(delivery_begin(h, "rcd_download_begin"));
    h->pend_kind = 0;
    h->pend_out = out;
    h->pend_cap = cap;
    return delivery_issued(h);
}

int rcd_download_begin_compact(rcd_handle h, rcd_pair_compact *out, uint64_t cap) {
    if (!h || (cap && !out)) return RCD_EINVAL;
    RC_TRY(delivery_begin(h, "rcd_download_begin_compact"));
    if (!h->compact_dev) CUDA_TRY(h, h->compact_dev.alloc(h->max_pairs));
    // (one scratch buffer: the narrowing of frame k + 1 runs on the handle's stream after frame k's copy was issued
    // and waited for by rcd_download_finish -- one delivery in flight at a time)
    k_compact_pairs<<<(unsigned)h->sms * 8, 256, 0, h->stream>>>(h->fb().out, h->max_pairs, &h->fb().counters->n_pairs, h->compact_dev);
    KERNEL_CHECK(h);
    h->pend_kind = 1;
    h->pend_out_compact = out;
    h->pend_cap = cap;
    return delivery_issued(h);
}

int rcd_download_finish(rcd_handle h, rcd_counts_t *counts, uint64_t *n_out) {
    if (!h || !n_out) return RCD_EINVAL;
    if (!h->download_pending || h->pend_kind == 2) return fail(h, RCD_ESTATE, "rcd_download_finish: no download in flight");
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaEventSynchronize(h->dl.pend_event));  // the frame is complete; later work keeps running
    const Counters &c = *h->dl.counters_host;
    const u64 m = std::min<u64>(std::min<u64>(c.n_pairs, h->max_pairs), h->pend_cap);
    if (m) {
        if (h->pend_kind == 0)
            CUDA_TRY(h, cudaMemcpyAsync(h->pend_out, h->pend_dev, (size_t)m * sizeof(rcd_pair), cudaMemcpyDeviceToHost, h->dl.copy_stream));
        else
            CUDA_TRY(h, cudaMemcpyAsync(h->pend_out_compact, h->compact_dev, (size_t)m * sizeof(rcd_pair_compact),
                                        cudaMemcpyDeviceToHost, h->dl.copy_stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->dl.copy_stream));
    }
    fill_counts(h, c, h->pend_n, h->pend_n_owned, counts);
    *n_out = m;
    h->download_pending = false;
    return RCD_OK;
}

int rcd_download_risk_counts(rcd_handle h, uint32_t *out, uint64_t n) {
    if (!h || (n && !out)) return RCD_EINVAL;
    if (!h->frame_done) return fail(h, RCD_ESTATE, "rcd_download_risk_counts: no frame has been stepped");
    if (n > h->n) return fail(h, RCD_EINVAL, "rcd_download_risk_counts: n exceeds the object count");
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (n) CUDA_TRY(h, cudaMemcpyAsync(out, h->fb().risk_count, (size_t)n * sizeof(u32), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return RCD_OK;
}

int rcd_download_candidate_counts(rcd_handle h, uint32_t *out, uint64_t n) {
    if (!h || (n && !out)) return RCD_EINVAL;
    if (!h->frame_done) return fail(h, RCD_ESTATE, "rcd_download_candidate_counts: no frame has been stepped");
    if (n > h->n) return fail(h, RCD_EINVAL, "rcd_download_candidate_counts: n exceeds the object count");
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (n) CUDA_TRY(h, cudaMemcpyAsync(out, h->cand_count, (size_t)n * sizeof(u32), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return RCD_OK;
}

int rcd_query_radius(rcd_handle h, uint64_t nq, const float *qx, const float *qy, const float *qz, float radius,
                     uint64_t *offsets, uint32_t *ids, uint64_t cap) {
    if (!h || !offsets || (nq && (!qx || !qy || !qz)) || (cap && !ids)) return RCD_EINVAL;
    if (!(radius >= 0.0f) || !std::isfinite(radius)) return fail(h, RCD_EINVAL, "rcd_query_radius: bad radius");
    for (u64 q = 0; q <= nq; ++q) offsets[q] = 0;
    if (nq == 0 || h->n == 0) return RCD_OK;
    CUDA_TRY(h, cudaSetDevice(h->device));
    RC_TRY(wait_upload(h));
    // reuse the index of the last frame if there is one, else build one with the default cell
    RC_TRY(build_index(h, h->idx.valid ? h->idx.cell_req : std::max(radius, 1.0f)));
    DevBuf<float> dq;
    DevBuf<uint2> dhits;
    CUDA_TRY(h, dq.alloc(3 * (size_t)nq));
    CUDA_TRY(h, dhits.alloc(std::max<u64>(cap, 1)));
    cudaMemcpyAsync(dq, qx, nq * sizeof(float), cudaMemcpyHostToDevice, h->stream);
    cudaMemcpyAsync(dq.get() + nq, qy, nq * sizeof(float), cudaMemcpyHostToDevice, h->stream);
    cudaMemcpyAsync(dq.get() + 2 * nq, qz, nq * sizeof(float), cudaMemcpyHostToDevice, h->stream);
    cudaMemsetAsync(&h->fb().counters->n_query_hits, 0, sizeof(unsigned long long), h->stream);
    const unsigned blocks = (unsigned)((nq * 32 + 127) / 128);
    k_query_radius<<<blocks, 128, 0, h->stream>>>((u32)nq, dq, dq.get() + nq, dq.get() + 2 * nq, radius, h->idx.grid, (u32)h->n,
                                                   h->P0, h->cell_begin, h->sorted_slot, dhits, cap, h->fb().counters);
    CUDA_TRY(h, cudaGetLastError());  // (the copies above report their errors here)
    unsigned long long total = 0;
    CUDA_TRY(h, cudaMemcpyAsync(&total, &h->fb().counters->n_query_hits, sizeof(total), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    ++h->launches;
    if (total > cap) {
        offsets[nq] = total;  // tells the caller how much room a retry needs
        return fail(h, RCD_ECAPACITY, "rcd_query_radius: result buffer too small");
    }
    std::vector<uint2> hits((size_t)total);
    if (total) CUDA_TRY(h, cudaMemcpy(hits.data(), dhits, (size_t)total * sizeof(uint2), cudaMemcpyDeviceToHost));
    std::vector<u32> idmap((size_t)h->n);
    CUDA_TRY(h, cudaMemcpy(idmap.data(), h->in_id, (size_t)h->n * sizeof(u32), cudaMemcpyDeviceToHost));
    std::sort(hits.begin(), hits.end(), [](const uint2 &a, const uint2 &b) { return a.x != b.x ? a.x < b.x : a.y < b.y; });
    for (const uint2 &hq : hits) offsets[hq.x + 1]++;
    for (u64 q = 0; q < nq; ++q) offsets[q + 1] += offsets[q];
    for (size_t k = 0; k < hits.size(); ++k) ids[k] = idmap[hits[k].y];
    return RCD_OK;
}

int rcd_classify_patterns(rcd_handle h, uint64_t n, uint32_t stride, const double *samples, const uint32_t *count,
                          uint8_t *pattern_out) {
    if (!h || (n && (!samples || !count || !pattern_out)) || stride == 0) return RCD_EINVAL;
    if (n == 0) return RCD_OK;
    CUDA_TRY(h, cudaSetDevice(h->device));
    const size_t ns = (size_t)n * stride * 4;
    DevBuf<double> ds;
    DevBuf<u32> dc;
    DevBuf<uint8_t> dout;
    CUDA_TRY(h, ds.alloc(ns));
    CUDA_TRY(h, dc.alloc(n));
    CUDA_TRY(h, dout.alloc(n));
    CUDA_TRY(h, cudaMemcpyAsync(ds, samples, ns * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(dc, count, (size_t)n * sizeof(u32), cudaMemcpyHostToDevice, h->stream));
    k_classify_patterns<<<(unsigned)((n + 127) / 128), 128, 0, h->stream>>>((u32)n, stride, ds, dc, dout);
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaMemcpyAsync(pattern_out, dout, (size_t)n, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    ++h->launches;
    return RCD_OK;
}

int rcd_pair_exact(rcd_handle h, uint64_t n, const rcd_object *a, const rcd_object *b, double time_window, double time_step,
                   rcd_pair_exact_result *out) {
    if (!h || (n && (!a || !b || !out))) return RCD_EINVAL;
    if (!(time_step > 0.0) || !std::isfinite(time_step) || !(time_window >= 0.0) || !std::isfinite(time_window))
        return fail(h, RCD_EINVAL, "rcd_pair_exact: bad time_window / time_step");
    if (n == 0) return RCD_OK;
    if (n > 0x7fffffffull) return fail(h, RCD_ECAPACITY, "rcd_pair_exact: too many pairs");
    const double nsteps = std::floor(time_window / time_step);  // int(time_window / time_step), :322
    const int steps = nsteps > 1.0e9 ? 1000000000 : (int)nsteps;
    CUDA_TRY(h, cudaSetDevice(h->device));
    DevBuf<rcd_object> da, db;
    DevBuf<rcd_pair_exact_result> dout;
    CUDA_TRY(h, da.alloc(n));
    CUDA_TRY(h, db.alloc(n));
    CUDA_TRY(h, dout.alloc(n));
    CUDA_TRY(h, cudaMemcpyAsync(da, a, (size_t)n * sizeof(rcd_object), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(db, b, (size_t)n * sizeof(rcd_object), cudaMemcpyHostToDevice, h->stream));
    k_pair_exact<<<(unsigned)((n + 127) / 128), 128, 0, h->stream>>>((u32)n, da, db, steps, time_step, dout);
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaMemcpyAsync(out, dout, (size_t)n * sizeof(rcd_pair_exact_result), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    ++h->launches;
    return RCD_OK;
}

int rcd_risk_assessment(rcd_handle h, uint64_t n, const double *in, double *risk_out) {
    if (!h || (n && (!in || !risk_out))) return RCD_EINVAL;
    if (n == 0) return RCD_OK;
    if (n > 0x7fffffffull) return fail(h, RCD_ECAPACITY, "rcd_risk_assessment: too many records");
    CUDA_TRY(h, cudaSetDevice(h->device));
    DevBuf<double> din, dout;
    CUDA_TRY(h, din.alloc(7 * (size_t)n));
    CUDA_TRY(h, dout.alloc(n));
    CUDA_TRY(h, cudaMemcpyAsync(din, in, 7 * (size_t)n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    k_risk_assessment<<<(unsigned)((n + 127) / 128), 128, 0, h->stream>>>((u32)n, din, dout);
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaMemcpyAsync(risk_out, dout, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    ++h->launches;
    return RCD_OK;
}

int rcd_history_configure(rcd_handle h, uint32_t max_history) {
    if (!h) return RCD_EINVAL;
    if (max_history < 2 || max_history > 4096) return fail(h, RCD_EINVAL, "rcd_history_configure: max_history must be in [2, 4096]");
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    h->traj.reset(); h->traj_count.reset(); h->traj_len = 0;
    return alloc_history(h, h->cap, max_history, h->stream, *h);
}

static int history_ready(rcd_handle h) {
    if (h->traj_len == 0) {
        RC_TRY(rcd_history_configure(h, 100));  // max_history_length = 100 (collision_detection.py:539)
    }
    return RCD_OK;
}

int rcd_history_append(rcd_handle h, uint64_t n, const uint32_t *slot, const double *x, const double *y,
                       const double *z, const double *t) {
    if (!h || (n && (!x || !y || !z || !t))) return RCD_EINVAL;
    if (n > h->cap) return fail(h, RCD_ECAPACITY, "rcd_history_append: n exceeds max_objects");
    if (n == 0) return RCD_OK;
    CUDA_TRY(h, cudaSetDevice(h->device));
    RC_TRY(history_ready(h));
    DevBuf<double> d;
    DevBuf<u32> ds;
    CUDA_TRY(h, d.alloc(4 * (size_t)n));
    if (slot) CUDA_TRY(h, ds.alloc(n));
    const double *src[4] = {x, y, z, t};
    for (int k = 0; k < 4; ++k)
        CUDA_TRY(h, cudaMemcpyAsync(d.get() + (size_t)k * n, src[k], (size_t)n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    if (slot) CUDA_TRY(h, cudaMemcpyAsync(ds, slot, (size_t)n * sizeof(u32), cudaMemcpyHostToDevice, h->stream));
    k_history_append<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>((u32)n, ds, d, d.get() + n, d.get() + 2 * n, d.get() + 3 * n,
                                                                         h->traj, h->traj_count, (u32)h->cap, h->traj_len);
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));  // the staging buffers are freed on return
    ++h->launches;
    return RCD_OK;
}

int rcd_history_reset(rcd_handle h, uint64_t n, const uint32_t *slot) {
    if (!h || (n && !slot)) return RCD_EINVAL;
    if (n == 0) return RCD_OK;
    CUDA_TRY(h, cudaSetDevice(h->device));
    RC_TRY(history_ready(h));
    DevBuf<u32> ds;
    CUDA_TRY(h, ds.alloc(n));
    CUDA_TRY(h, cudaMemcpyAsync(ds, slot, (size_t)n * sizeof(u32), cudaMemcpyHostToDevice, h->stream));
    k_history_reset<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>((u32)n, ds, h->traj_count, (u32)h->cap);
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return RCD_OK;
}

int rcd_history_move(rcd_handle h, uint32_t dst, uint32_t src) {
    if (!h) return RCD_EINVAL;
    if (dst >= h->cap || src >= h->cap) return fail(h, RCD_EINVAL, "rcd_history_move: slot out of range");
    if (dst == src) return RCD_OK;
    CUDA_TRY(h, cudaSetDevice(h->device));
    RC_TRY(history_ready(h));
    k_history_move<<<1, 128, 0, h->stream>>>(dst, src, h->traj, h->traj_count, (u32)h->cap, h->traj_len);
    KERNEL_CHECK(h);
    return RCD_OK;
}

int rcd_history_classify(rcd_handle h, uint8_t *pattern_out) {
    if (!h) return RCD_EINVAL;
    CUDA_TRY(h, cudaSetDevice(h->device));
    RC_TRY(history_ready(h));
    RC_TRY(wait_upload(h));
    if (h->n) {
        k_history_classify<<<(unsigned)((h->n + 127) / 128), 128, 0, h->stream>>>((u32)h->n, h->traj, h->traj_count,
                                                                                  (u32)h->cap, h->traj_len, h->in_pattern);
        KERNEL_CHECK(h);
        if (pattern_out) {
            CUDA_TRY(h, cudaMemcpyAsync(pattern_out, h->in_pattern, (size_t)h->n, cudaMemcpyDeviceToHost, h->stream));
            CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        }
    }
    h->idx.valid = false;  // the pattern is packed into the cell-ordered state
    h->frame_done = false;
    return RCD_OK;
}

int rcd_apply_records(rcd_handle h, uint64_t n, const rcd_record *records, uint32_t max_seq, uint64_t n_objects,
                      int32_t append_history, int32_t src) {
    if (!h || (n && !records)) return RCD_EINVAL;
    if (n_objects > h->cap) return fail(h, RCD_ECAPACITY, "rcd_apply_records: n_objects exceeds max_objects");
    if (n_objects < h->n) return fail(h, RCD_EINVAL, "rcd_apply_records: n_objects is smaller than the current frame");
    if (n > 0xffffffffull / 16) return fail(h, RCD_ECAPACITY, "rcd_apply_records: batch too large");
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (append_history) {
        RC_TRY(history_ready(h));
    }
    const bool hist = append_history && h->traj.get();
    if (!h->last_seen) RC_TRY(alloc_last_seen(h, h->cap, h->stream, *h));
    RC_TRY(wait_upload(h));
    reset_stages(h, -1);
    h->stage_mode = 0;
    stage_begin(h, RCD_STAGE_UPLOAD);
    if (n_objects > h->n) {
        const u32 fresh = (u32)(n_objects - h->n);
        k_init_slots<<<(fresh + 255) / 256, 256, 0, h->stream>>>((u32)h->n, (u32)n_objects, h->in_id, h->in_pattern,
                                                                 h->last_seen);
        KERNEL_CHECK(h);
    }
    const unsigned long long *dev = reinterpret_cast<const unsigned long long *>(records);
    DevBuf<unsigned long long> staged;
    if (n && src == RCD_SRC_HOST) {
        CUDA_TRY(h, staged.alloc((size_t)n * RECORD_WORDS));
        CUDA_TRY(h, cudaMemcpyAsync(staged, records, (size_t)n * sizeof(rcd_record), cudaMemcpyHostToDevice, h->stream));
        dev = staged;
    }
    const MutableState st = mutable_state(h);
    for (u32 seq = 0; n && seq <= max_seq; ++seq) {
        k_apply_records<<<(unsigned)((n + APPLY_THREADS - 1) / APPLY_THREADS), APPLY_THREADS, 0, h->stream>>>(
            (u32)n, dev, seq, (u32)n_objects, st, hist ? h->traj.get() : nullptr, h->traj_count, (u32)h->cap, h->traj_len,
            h->last_seen);
        KERNEL_CHECK(h);
    }
    stage_end(h, RCD_STAGE_UPLOAD);
    RC_TRY(release_inputs(h));
    if (staged) CUDA_TRY(h, cudaStreamSynchronize(h->stream));  // the staging buffer is freed on return
    h->n = n_objects;
    h->n_owned = n_objects;
    h->idx.valid = false;
    h->frame_done = false;
    return RCD_OK;
}

// ---- alert lifecycle -------------------------------------------------------------------------------------
static int alerts_ready(rcd_handle h, const char *who) {
    if (!h->alert_cap) return fail(h, RCD_ESTATE, std::string(who) + ": call rcd_alerts_configure first");
    return RCD_OK;
}
// zero the per-call counters (n_live and next_id persist), run `launch`, bring counters + events back
extern "C++" {
template <typename F>
static int alerts_call(rcd_handle h, rcd_alert_event *events, uint64_t cap, rcd_alert_stats *stats, bool reset_live, F launch) {
    CUDA_TRY(h, cudaSetDevice(h->device));
    RC_TRY(alerts_join(h));
    CUDA_TRY(h, cudaMemsetAsync(h->alert_counters, 0, offsetof(AlertCounters, n_live), h->stream));
    if (reset_live) CUDA_TRY(h, cudaMemsetAsync(&h->alert_counters->n_live, 0, sizeof(unsigned long long), h->stream));
    RC_TRY(launch());
    CUDA_TRY(h, cudaMemcpyAsync(h->alert_counters_host, h->alert_counters, sizeof(AlertCounters), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    const u64 n_ev = std::min<u64>(std::min<u64>(h->alert_counters_host->n_events, h->alert_ev_cap), cap);
    if (n_ev && events)
        CUDA_TRY(h, cudaMemcpy(events, h->alert_ev, (size_t)n_ev * sizeof(rcd_alert_event), cudaMemcpyDeviceToHost));
    fill_alert_stats(*h->alert_counters_host, stats);
    return RCD_OK;
}
}  // extern "C++"

int rcd_alerts_configure(rcd_handle h, uint64_t max_alerts) {
    if (!h || max_alerts == 0 || max_alerts > (1ull << 31)) return h ? fail(h, RCD_EINVAL, "rcd_alerts_configure: max_alerts must be in [1, 2^31]") : RCD_EINVAL;
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (h->dl.alert_stream) CUDA_TRY(h, cudaStreamSynchronize(h->dl.alert_stream));
    h->alert_async = false;
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    h->alert_tab[0].reset(); h->alert_tab[1].reset(); h->alert_ev.reset(); h->alert_ev_alt.reset(); h->alert_counters.reset();
    h->alert_counters_host.reset();
    h->alert_cap = 0;
    u64 cap = 1024;
    while (cap < 2 * max_alerts) cap <<= 1;  // load factor <= 0.5
    CUDA_TRY(h, h->alert_tab[0].alloc(cap));
    CUDA_TRY(h, h->alert_tab[1].alloc(cap));
    CUDA_TRY(h, h->alert_ev.alloc(max_alerts));
    CUDA_TRY(h, h->alert_counters.alloc());
    CUDA_TRY(h, h->alert_counters_host.alloc());
    CUDA_TRY(h, cudaMemsetAsync(h->alert_tab[0], 0xff, (size_t)cap * sizeof(AlertEntry), h->stream));
    CUDA_TRY(h, cudaMemsetAsync(h->alert_counters, 0, sizeof(AlertCounters), h->stream));
    h->alert_cur = 0;
    h->alert_cap = cap;
    h->alert_ev_cap = max_alerts;
    return RCD_OK;
}

int rcd_alerts_reserve(rcd_handle h, uint64_t max_alerts) {
    if (!h) return RCD_EINVAL;
    RC_TRY(alerts_ready(h, "rcd_alerts_reserve"));
    if (max_alerts > (1ull << 31)) return fail(h, RCD_EINVAL, "rcd_alerts_reserve: max_alerts must be at most 2^31");
    if (max_alerts <= h->alert_ev_cap) return RCD_OK;
    if (h->download_pending && h->pend_kind == 2) return fail(h, RCD_ESTATE, "rcd_alerts_reserve: a summary is in flight");
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (h->dl.alert_stream) CUDA_TRY(h, cudaStreamSynchronize(h->dl.alert_stream));
    h->alert_async = false;
    u64 cap = 1024;
    while (cap < 2 * max_alerts) cap <<= 1;  // load factor <= 0.5, as in rcd_alerts_configure
    // the new table, its twin and the event buffers exist before anything of the old ones changes
    DevBuf<AlertEntry> tab, twin;
    DevBuf<rcd_alert_event> ev, ev_alt;
    auto make = [&]() -> int {
        CUDA_TRY(h, tab.alloc(cap));
        CUDA_TRY(h, twin.alloc(cap));
        CUDA_TRY(h, ev.alloc(max_alerts));
        if (h->alert_ev_alt) CUDA_TRY(h, ev_alt.alloc(max_alerts));
        return RCD_OK;
    };
    if (const int rc = make()) {
        (void)cudaGetLastError();  // (a refused allocation is not a fault of the handle)
        return rc;
    }
    // every live entry is rehashed into the new table; n_live is recounted, the alert numbering goes on
    CUDA_TRY(h, cudaMemsetAsync(tab, 0xff, (size_t)cap * sizeof(AlertEntry), h->stream));
    CUDA_TRY(h, cudaMemsetAsync(&h->alert_counters->n_live, 0, sizeof(unsigned long long), h->stream));
    const unsigned blocks = (unsigned)std::min<u64>((h->alert_cap + ALERT_THREADS - 1) / ALERT_THREADS, (u64)h->sms * 8);
    k_alert_rebuild<<<blocks, ALERT_THREADS, 0, h->stream>>>(h->alert_tab[h->alert_cur], h->alert_cap, AlertKeep{cap - 1}, tab, ev, 0,
                                                             h->alert_counters);
    KERNEL_CHECK(h);
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    h->alert_tab[0] = std::move(tab);
    h->alert_tab[1] = std::move(twin);
    h->alert_cur = 0;
    h->alert_ev = std::move(ev);
    if (h->alert_ev_alt) h->alert_ev_alt = std::move(ev_alt);
    h->alert_cap = cap;
    h->alert_ev_cap = max_alerts;
    return RCD_OK;
}

// fold pairs into the table (both passes), events -> h->alert_ev
static int alerts_enqueue_update(rcd_handle h, const rcd_pair *dev_pairs, u64 n_max, const unsigned long long *n_dev, double now,
                                 int32_t report_refreshed, cudaStream_t on = nullptr,
                                 const unsigned long long *n_dev_detect = nullptr /* bound of the detect pass (null: n_dev) */) {
    if (n_max == 0) return RCD_OK;
    const int sms = h->sms;
    u64 blocks = std::min<u64>((n_max + ALERT_THREADS - 1) / ALERT_THREADS, (u64)sms * 16);
    if (on) {
        // beside the next frame (lower-priority stream): many short-lived blocks -- about one pair per thread, sized from
        // the last pair count the host has seen; the grid-stride loop covers whatever the estimate misses -- so that
        // block slots go back to the frame's kernels as soon as they ask for them
        const u64 est = h->last_n_pairs ? h->last_n_pairs + h->last_n_pairs / 4 : (u64)sms * 16 * ALERT_THREADS;
        blocks = std::min<u64>((n_max + ALERT_THREADS - 1) / ALERT_THREADS, std::max<u64>((est + ALERT_THREADS - 1) / ALERT_THREADS, (u64)sms));
    } else {
        on = h->stream;
    }
    for (int pass = 0; pass < 2; ++pass) {
        u64 grid = blocks;
        if (pass == 0 && n_dev_detect && h->last_n_detect_end) {  // the detect pass ends early: a grid to match
            const u64 est_d = h->last_n_detect_end + h->last_n_detect_end / 4;
            grid = std::min<u64>(blocks, std::max<u64>((est_d + ALERT_THREADS - 1) / ALERT_THREADS, (u64)sms));
        }
        k_alert_update<<<(unsigned)grid, ALERT_THREADS, 0, on>>>(dev_pairs, n_max, (pass == 0 && n_dev_detect) ? n_dev_detect : n_dev,
                                                        pass, now, h->alert_tab[h->alert_cur],
                                                        h->alert_cap - 1, h->alert_ev, h->alert_ev_cap,
                                                        h->alert_counters, report_refreshed);
        KERNEL_CHECK(h);
    }
    return RCD_OK;
}
static int alerts_update_impl(rcd_handle h, const rcd_pair *dev_pairs, u64 n_max, const unsigned long long *n_dev, double now,
                              int32_t report_refreshed, rcd_alert_event *events, uint64_t cap, rcd_alert_stats *stats) {
    return alerts_call(h, events, cap, stats, false,
                       [&]() -> int { return alerts_enqueue_update(h, dev_pairs, n_max, n_dev, now, report_refreshed); });
}

int rcd_summary_begin(rcd_handle h, double now, int32_t report_refreshed) {
    if (!h) return RCD_EINVAL;
    RC_TRY(alerts_ready(h, "rcd_summary_begin"));
    RC_TRY(delivery_begin(h, "rcd_summary_begin"));
    if (!h->alert_ev_alt) CUDA_TRY(h, h->alert_ev_alt.alloc(h->alert_ev_cap));
    std::swap(h->alert_ev, h->alert_ev_alt);  // the events of the previous summary may still be on their way to the host
    // the fold runs on alert_stream, after the frame and beside whatever the handle's stream does next (the next
    // frame writes the twin pair buffer and twin totals; other alert calls join alert_stream first)
    cudaStream_t as = h->dl.alert_stream;
    CUDA_TRY(h, cudaEventRecord(h->dl.ev_frame_done, h->stream));
    CUDA_TRY(h, cudaStreamWaitEvent(as, h->dl.ev_frame_done, 0));
    CUDA_TRY(h, cudaMemsetAsync(h->alert_counters, 0, offsetof(AlertCounters, n_live), as));
    RC_TRY(alerts_enqueue_update(h, h->fb().out, h->max_pairs, &h->fb().counters->n_pairs, now, report_refreshed, as, &h->fb().counters->n_detect_end));
    CUDA_TRY(h, cudaMemcpyAsync(h->dl.alert_counters_host, h->alert_counters, sizeof(AlertCounters), cudaMemcpyDeviceToHost, as));
    h->pend_kind = 2;
    h->pend_ev = h->alert_ev;
    RC_TRY(delivery_issued(h, as));
    CUDA_TRY(h, cudaEventRecord(h->dl.ev_alert_done, as));
    h->alert_async = true;
    return RCD_OK;
}

int rcd_summary_finish(rcd_handle h, rcd_alert_event *events, uint64_t cap, uint64_t *n_events, rcd_alert_stats *stats,
                       uint32_t *risk_counts, uint64_t n, rcd_counts_t *counts) {
    if (!h || (cap && !events) || (n && !risk_counts)) return RCD_EINVAL;
    if (!h->download_pending || h->pend_kind != 2) return fail(h, RCD_ESTATE, "rcd_summary_finish: no summary in flight");
    if (n > h->pend_n) return fail(h, RCD_EINVAL, "rcd_summary_finish: n exceeds the frame's object count");
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaEventSynchronize(h->dl.pend_event));
    const AlertCounters &ac = *h->dl.alert_counters_host;
    const u64 n_ev = std::min<u64>(std::min<u64>(ac.n_events, h->alert_ev_cap), cap);
    if (n_ev) CUDA_TRY(h, cudaMemcpyAsync(events, h->pend_ev, (size_t)n_ev * sizeof(rcd_alert_event), cudaMemcpyDeviceToHost, h->dl.copy_stream));
    if (n) CUDA_TRY(h, cudaMemcpyAsync(risk_counts, h->pend_risk, (size_t)n * sizeof(u32), cudaMemcpyDeviceToHost, h->dl.copy_stream));
    if (n_ev || n) CUDA_TRY(h, cudaStreamSynchronize(h->dl.copy_stream));
    if (n_events) *n_events = n_ev;
    fill_alert_stats(ac, stats);
    fill_counts(h, *h->dl.counters_host, h->pend_n, h->pend_n_owned, counts);
    h->download_pending = false;
    return RCD_OK;
}

int rcd_alerts_update(rcd_handle h, double now, int32_t report_refreshed, rcd_alert_event *events, uint64_t cap,
                      rcd_alert_stats *stats) {
    if (!h) return RCD_EINVAL;
    RC_TRY(alerts_ready(h, "rcd_alerts_update"));
    if (!h->frame_done) return fail(h, RCD_ESTATE, "rcd_alerts_update: no frame has been stepped");
    return alerts_update_impl(h, h->fb().out, h->max_pairs, &h->fb().counters->n_pairs, now, report_refreshed, events, cap, stats);
}

int rcd_alerts_update_pairs(rcd_handle h, const rcd_pair *pairs, uint64_t n, double now, int32_t report_refreshed,
                            rcd_alert_event *events, uint64_t cap, rcd_alert_stats *stats) {
    if (!h || (n && !pairs)) return RCD_EINVAL;
    RC_TRY(alerts_ready(h, "rcd_alerts_update_pairs"));
    CUDA_TRY(h, cudaSetDevice(h->device));
    DevBuf<rcd_pair> staged;
    if (n) {
        CUDA_TRY(h, staged.alloc(n));
        CUDA_TRY(h, cudaMemcpyAsync(staged, pairs, (size_t)n * sizeof(rcd_pair), cudaMemcpyHostToDevice, h->stream));
    }
    return alerts_update_impl(h, staged, n, nullptr, now, report_refreshed, events, cap, stats);  // (synchronises)
}

int rcd_alerts_expire(rcd_handle h, double now, double max_age, rcd_alert_event *events, uint64_t cap, rcd_alert_stats *stats) {
    if (!h) return RCD_EINVAL;
    RC_TRY(alerts_ready(h, "rcd_alerts_expire"));
    const int rc = alerts_call(h, events, cap, stats, true, [&]() -> int {
        AlertEntry *src = h->alert_tab[h->alert_cur], *dst = h->alert_tab[h->alert_cur ^ 1];
        CUDA_TRY(h, cudaMemsetAsync(dst, 0xff, (size_t)h->alert_cap * sizeof(AlertEntry), h->stream));
        const unsigned blocks = (unsigned)std::min<u64>((h->alert_cap + ALERT_THREADS - 1) / ALERT_THREADS, (u64)h->sms * 8);
        k_alert_rebuild<<<blocks, ALERT_THREADS, 0, h->stream>>>(src, h->alert_cap, AlertTooOld{now, max_age}, dst, h->alert_ev,
                                                                 h->alert_ev_cap, h->alert_counters);
        KERNEL_CHECK(h);
        return RCD_OK;
    });
    if (rc == RCD_OK) h->alert_cur ^= 1;
    return rc;
}

int rcd_alerts_acknowledge(rcd_handle h, uint64_t n, const uint32_t *i, const uint32_t *j, uint64_t *n_found) {
    if (!h || (n && (!i || !j))) return RCD_EINVAL;
    RC_TRY(alerts_ready(h, "rcd_alerts_acknowledge"));
    if (n_found) *n_found = 0;
    if (n == 0) return RCD_OK;
    if (n > 0xffffffffull) return fail(h, RCD_ECAPACITY, "rcd_alerts_acknowledge: too many pairs");
    CUDA_TRY(h, cudaSetDevice(h->device));
    RC_TRY(alerts_join(h));
    DevBuf<u32> d;
    CUDA_TRY(h, d.alloc(2 * (size_t)n + 1));
    u32 *const di = d, *const dj = d.get() + n, *const dfound = d.get() + 2 * n;
    CUDA_TRY(h, cudaMemcpyAsync(di, i, (size_t)n * sizeof(u32), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(dj, j, (size_t)n * sizeof(u32), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaMemsetAsync(dfound, 0, sizeof(u32), h->stream));
    k_alert_ack<<<(unsigned)((n + ALERT_THREADS - 1) / ALERT_THREADS), ALERT_THREADS, 0, h->stream>>>(
        di, dj, (u32)n, h->alert_tab[h->alert_cur], h->alert_cap - 1, dfound);
    KERNEL_CHECK(h);
    u32 found = 0;
    CUDA_TRY(h, cudaMemcpyAsync(&found, dfound, sizeof(u32), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (n_found) *n_found = found;
    return RCD_OK;
}

int rcd_alerts_download(rcd_handle h, rcd_alert_event *out, uint64_t cap, uint64_t *n_out) {
    if (!h || !n_out || (cap && !out)) return RCD_EINVAL;
    RC_TRY(alerts_ready(h, "rcd_alerts_download"));
    CUDA_TRY(h, cudaSetDevice(h->device));
    rcd_alert_stats st;
    const int rc = alerts_call(h, out, cap, &st, false, [&]() -> int {
        const unsigned blocks = (unsigned)std::min<u64>((h->alert_cap + ALERT_THREADS - 1) / ALERT_THREADS, (u64)h->sms * 8);
        k_alert_dump<<<blocks, ALERT_THREADS, 0, h->stream>>>(h->alert_tab[h->alert_cur], h->alert_cap, h->alert_ev, h->alert_ev_cap,
                                                              h->alert_counters);
        KERNEL_CHECK(h);
        return RCD_OK;
    });
    if (rc) return rc;
    const u64 n = std::min<u64>(std::min<u64>(st.n_events, h->alert_ev_cap), cap);
    std::sort(out, out + n, [](const rcd_alert_event &a, const rcd_alert_event &b) { return a.i != b.i ? a.i < b.i : a.j < b.j; });
    *n_out = n;
    return RCD_OK;
}

// ---- retirement (rcd_retire, rcd_retire_stale) -------------------------------------------------------------
// Retire the n slots of the device list d_slots (checked: each < h->n); d_ids has room for n caller ids.  Both entry
// points end the frame and invalidate the index; the query list stays (a listed retired slot emits nothing).
static int retire_slots(rcd_handle h, u64 n, const u32 *d_slots, u32 *d_ids, rcd_alert_event *events, uint64_t cap,
                        rcd_alert_stats *stats) {
    if (stats) *stats = rcd_alert_stats{};
    h->idx.valid = false;
    h->frame_done = false;
    if (n) {
        RC_TRY(wait_upload(h));
        k_retire_slots<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(d_slots, (u32)n, mutable_state(h),
                                                                           h->traj_count.get(), h->last_seen.get(), d_ids);
        KERNEL_CHECK(h);
        RC_TRY(release_inputs(h));
    }
    if (!h->alert_cap) return RCD_OK;
    // the purge: every alert of a retired caller id, after an in-flight summary fold (like rcd_alerts_expire)
    RC_TRY(alerts_join(h));
    std::vector<u32> ids((size_t)n);
    if (n) CUDA_TRY(h, cudaMemcpyAsync(ids.data(), d_ids, (size_t)n * sizeof(u32), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(h->alert_counters_host, h->alert_counters, sizeof(AlertCounters), cudaMemcpyDeviceToHost,
                                h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    const u64 live = h->alert_counters_host->n_live;
    std::sort(ids.begin(), ids.end());
    ids.erase(std::unique(ids.begin(), ids.end()), ids.end());
    if (ids.empty() || live == 0) {  // nothing can match: no rebuild
        if (stats) stats->n_live = live;
        return RCD_OK;
    }
    CUDA_TRY(h, cudaMemcpyAsync(d_ids, ids.data(), ids.size() * sizeof(u32), cudaMemcpyHostToDevice, h->stream));
    const int rc = alerts_call(h, events, cap, stats, true, [&]() -> int {
        AlertEntry *src = h->alert_tab[h->alert_cur], *dst = h->alert_tab[h->alert_cur ^ 1];
        CUDA_TRY(h, cudaMemsetAsync(dst, 0xff, (size_t)h->alert_cap * sizeof(AlertEntry), h->stream));
        const unsigned blocks = (unsigned)std::min<u64>((h->alert_cap + ALERT_THREADS - 1) / ALERT_THREADS, (u64)h->sms * 8);
        k_alert_rebuild<<<blocks, ALERT_THREADS, 0, h->stream>>>(src, h->alert_cap, AlertOfRetired{d_ids, (u32)ids.size()}, dst,
                                                                 h->alert_ev, h->alert_ev_cap, h->alert_counters);
        KERNEL_CHECK(h);
        return RCD_OK;
    });
    if (rc == RCD_OK) h->alert_cur ^= 1;
    return rc;
}

int rcd_retire(rcd_handle h, uint64_t n, const uint32_t *slots, rcd_alert_event *events, uint64_t cap, rcd_alert_stats *stats) {
    if (!h || (n && !slots) || (cap && !events)) return RCD_EINVAL;
    for (u64 k = 0; k < n; ++k)
        if (slots[k] >= h->n) return fail(h, RCD_EINVAL, "rcd_retire: slot " + std::to_string(slots[k]) + " is not in the frame");
    if (n > 0xffffffffull) return fail(h, RCD_ECAPACITY, "rcd_retire: too many slots");
    CUDA_TRY(h, cudaSetDevice(h->device));
    DevBuf<u32> d;  // [n] slots, [n] caller ids
    if (n) {
        CUDA_TRY(h, d.alloc(2 * (size_t)n));
        CUDA_TRY(h, cudaMemcpyAsync(d, slots, (size_t)n * sizeof(u32), cudaMemcpyHostToDevice, h->stream));
    }
    RC_TRY(retire_slots(h, n, d, d.get() + n, events, cap, stats));
    if (n) CUDA_TRY(h, cudaStreamSynchronize(h->stream));  // d is freed on return
    return RCD_OK;
}

int rcd_retire_stale(rcd_handle h, double now, double max_age, uint32_t *slots_out, uint64_t slots_cap, uint64_t *n_retired,
                     rcd_alert_event *events, uint64_t cap, rcd_alert_stats *stats) {
    if (!h || !n_retired || (slots_cap && !slots_out) || (cap && !events)) return RCD_EINVAL;
    if (!h->records_only)
        return fail(h, RCD_ESTATE, "rcd_retire_stale: the frame has objects that rcd_apply_records did not write (rcd_upload / "
                                   "rcd_halo_append): they have no record time");
    *n_retired = 0;
    CUDA_TRY(h, cudaSetDevice(h->device));
    const u32 n = (u32)h->n;
    u64 total = 0;
    DevBuf<u32> tiles_buf, d;
    if (n && h->last_seen) {
        RC_TRY(wait_upload(h));
        const u32 tiles = (n + STALE_TILE - 1) / STALE_TILE;
        CUDA_TRY(h, tiles_buf.alloc((size_t)tiles + 1));
        k_stale_count<<<tiles, STALE_THREADS, 0, h->stream>>>(h->last_seen, n, now, max_age, tiles_buf);
        KERNEL_CHECK(h);
        k_scan_tiles<<<1, 1024, 0, h->stream>>>(tiles_buf, tiles);
        KERNEL_CHECK(h);
        u32 count = 0;
        CUDA_TRY(h, cudaMemcpyAsync(&count, tiles_buf.get() + tiles, sizeof(u32), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        total = count;
        *n_retired = total;
        if (total > slots_cap) {
            if (stats) *stats = rcd_alert_stats{};
            return fail(h, RCD_ECAPACITY, "rcd_retire_stale: " + std::to_string(total) + " stale slots, room for " +
                                              std::to_string(slots_cap));
        }
        if (total) {
            CUDA_TRY(h, d.alloc(2 * (size_t)total));  // [total] slots, ascending, [total] caller ids
            k_stale_scatter<<<tiles, STALE_THREADS, 0, h->stream>>>(h->last_seen, n, now, max_age, tiles_buf, d);
            KERNEL_CHECK(h);
            CUDA_TRY(h, cudaMemcpyAsync(slots_out, d, (size_t)total * sizeof(u32), cudaMemcpyDeviceToHost, h->stream));
        }
    }
    RC_TRY(retire_slots(h, total, d, d.get() + total, events, cap, stats));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));  // slots_out is complete; the scratch buffers are freed on return
    return RCD_OK;
}

int rcd_halo_pack(rcd_handle h, int32_t n_peers, int32_t self, const float *slab_lo, const float *slab_hi, float halo,
                  void *out_records, uint64_t cap, uint64_t *counts) {
    if (!h || !slab_lo || !slab_hi || !counts || n_peers < 1 || n_peers > MAX_PEERS || self < 0 || self >= n_peers)
        return fail(h, RCD_EINVAL, "rcd_halo_pack: bad arguments");
    CUDA_TRY(h, cudaSetDevice(h->device));
    RC_TRY(wait_upload(h));
    for (int p = 0; p < n_peers; ++p) counts[p] = 0;
    if (h->n_owned == 0) return RCD_OK;
    SlabParams sp;
    sp.n_peers = n_peers; sp.self = self; sp.halo = halo;
    for (int p = 0; p < n_peers; ++p) { sp.lo[p] = slab_lo[p]; sp.hi[p] = slab_hi[p]; }
    DevBuf<unsigned long long> dcnt;  // [MAX_PEERS] counts, then [MAX_PEERS] bases
    CUDA_TRY(h, dcnt.alloc(2 * (size_t)MAX_PEERS));
    unsigned long long *const dbase = dcnt.get() + MAX_PEERS;
    unsigned long long host_cnt[MAX_PEERS] = {}, host_base[MAX_PEERS] = {};
    const unsigned blocks = (unsigned)((h->n_owned + 255) / 256);
    CUDA_TRY(h, cudaMemsetAsync(dcnt, 0, 2 * MAX_PEERS * sizeof(unsigned long long), h->stream));
    k_halo_pack<<<blocks, 256, 0, h->stream>>>((u32)h->n_owned, input_state(h), sp, 0, dcnt, dbase, nullptr, 0);
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaMemcpyAsync(host_cnt, dcnt, n_peers * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    u64 total = 0;
    for (int p = 0; p < n_peers; ++p) { host_base[p] = total; total += host_cnt[p]; counts[p] = host_cnt[p]; }
    if (!out_records && cap == 0) {  // counting pass only
        ++h->launches;
        return RCD_OK;
    }
    if (total > cap || (total && !out_records)) return fail(h, RCD_ECAPACITY, "rcd_halo_pack: record buffer too small");
    if (total) {
        CUDA_TRY(h, cudaMemsetAsync(dcnt, 0, MAX_PEERS * sizeof(unsigned long long), h->stream));
        CUDA_TRY(h, cudaMemcpyAsync(dbase, host_base, n_peers * sizeof(unsigned long long), cudaMemcpyHostToDevice, h->stream));
        k_halo_pack<<<blocks, 256, 0, h->stream>>>((u32)h->n_owned, input_state(h), sp, 1, dcnt, dbase,
                                                  static_cast<u32 *>(out_records), cap);
        CUDA_TRY(h, cudaGetLastError());
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    }
    h->launches += total ? 2 : 1;
    return RCD_OK;
}

int rcd_halo_pack_async(rcd_handle h, int32_t n_peers, int32_t self, const float *slab_lo, const float *slab_hi, float halo,
                        void *out_records, const uint64_t *peer_offset, uint64_t *counts_dev) {
    if (!h || !slab_lo || !slab_hi || !peer_offset || !counts_dev || !out_records || n_peers < 1 || n_peers > MAX_PEERS ||
        self < 0 || self >= n_peers)
        return fail(h, RCD_EINVAL, "rcd_halo_pack_async: bad arguments");
    CUDA_TRY(h, cudaSetDevice(h->device));
    RC_TRY(wait_upload(h));
    SlabParams sp;
    sp.n_peers = n_peers; sp.self = self; sp.halo = halo;
    SlabRegions rg;
    for (int p = 0; p < n_peers; ++p) {
        sp.lo[p] = slab_lo[p]; sp.hi[p] = slab_hi[p];
        rg.offset[p] = peer_offset[p];
        rg.cap[p] = peer_offset[p + 1] - peer_offset[p];
    }
    const u64 total = peer_offset[n_peers];
    // every slot starts as a ghost record (all bits set: NaN state, id 0xffffffff); the kernel overwrites the used ones
    if (total) CUDA_TRY(h, cudaMemsetAsync(out_records, 0xff, (size_t)total * HALO_WORDS * sizeof(u32), h->stream));
    CUDA_TRY(h, cudaMemsetAsync(counts_dev, 0, (size_t)n_peers * sizeof(unsigned long long), h->stream));
    if (h->n_owned) {
        k_halo_pack_regions<<<(unsigned)((h->n_owned + 255) / 256), 256, 0, h->stream>>>(
            (u32)h->n_owned, input_state(h), sp, rg, reinterpret_cast<unsigned long long *>(counts_dev), static_cast<u32 *>(out_records));
        KERNEL_CHECK(h);
    }
    return RCD_OK;
}

int rcd_halo_append(rcd_handle h, const void *records, uint64_t n_records) {
    if (!h || (n_records && !records)) return RCD_EINVAL;
    if (h->n + n_records > h->cap) return fail(h, RCD_ECAPACITY, "rcd_halo_append: exceeds max_objects");
    if (n_records == 0) return RCD_OK;
    CUDA_TRY(h, cudaSetDevice(h->device));
    RC_TRY(wait_upload(h));
    const MutableState st = mutable_state(h);
    k_halo_append<<<(unsigned)((n_records + 255) / 256), 256, 0, h->stream>>>(static_cast<const u32 *>(records),
                                                                             (u32)n_records, (u32)h->n, st);
    KERNEL_CHECK(h);
    RC_TRY(release_inputs(h));
    h->n += n_records;
    h->records_only = false;
    h->idx.valid = false;
    h->frame_done = false;
    return RCD_OK;
}

int rcd_get_stream(rcd_handle h, void **stream) {
    if (!h || !stream) return RCD_EINVAL;
    *stream = static_cast<void *>(h->stream);
    return RCD_OK;
}

int rcd_stage_ms(rcd_handle h, int32_t mode, float *ms) {
    if (!h || !ms || mode < 0 || mode > 2) return RCD_EINVAL;
    if (!(h->flags & RCD_FLAG_PROFILE)) return fail(h, RCD_ESTATE, "rcd_stage_ms: handle was created without RCD_FLAG_PROFILE");
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaStreamSynchronize(h->up_stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    for (int s = 0; s < RCD_NUM_STAGES; ++s) {
        ms[s] = 0.0f;
        const Stage &st = (s == RCD_STAGE_UPLOAD || s == RCD_STAGE_DOWNLOAD) ? h->stages[0][s] : h->stages[mode][s];
        if (st.used) {
            float t = 0.0f;
            if (cudaEventElapsedTime(&t, st.begin, st.end) == cudaSuccess) ms[s] = t;
            else (void)cudaGetLastError();
        }
    }
    return RCD_OK;
}

int rcd_pair_tests(rcd_handle h, uint64_t *n) {
    if (!h || !n) return RCD_EINVAL;
    if (!h->frame_done) return fail(h, RCD_ESTATE, "rcd_pair_tests: no frame has been stepped");
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaMemcpyAsync(h->counters_host, h->fb().counters, sizeof(Counters), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    *n = h->counters_host->n_tests;
    return RCD_OK;
}

int rcd_launch_count(rcd_handle h, uint64_t *n) {
    if (!h || !n) return RCD_EINVAL;
    *n = h->launches;
    return RCD_OK;
}

int rcd_sync(rcd_handle h) {
    if (!h) return RCD_EINVAL;
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaStreamSynchronize(h->up_stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (h->dl.alert_stream) CUDA_TRY(h, cudaStreamSynchronize(h->dl.alert_stream));
    return RCD_OK;
}

}  // extern "C"
