/*
 * TEST INFRASTRUCTURE ONLY -- CPU oracle for the src/collision hot path.
 *
 * Plain-C float64 restatement of the reference's algorithm (reference = pure Python, so there
 * is no reference binary to build: oracle/_ref does not apply; see DESIGN.md).  Only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load this
 * library, and only as the checker / the reported CPU baseline.  The product never links it.
 *
 * PARITY PIN: the reference ships no golden vectors (SURVEY.md 8c).  This restatement is pinned
 * against the reference's own bytecode executed under the documented shim (oracle/ref_shim.py)
 * by tests/test_oracle_vs_reference.py (runs where /root/reference exists) and against the
 * committed fixtures tests/golden/ (.npz) that the shim produced (tests/golden/make_golden.py).
 *
 * Every function cites the reference file:line (relative to /root/reference) it follows.
 * Arithmetic follows the Python evaluation order literally; `x ** 2` and `x ** 0.5` go through
 * libm pow() exactly as CPython's float_pow does (build with -fno-builtin -ffp-contract=off so
 * gcc neither folds pow(x,2) into x*x nor fuses multiply-adds).
 *
 * The uniform grid used to find neighbours is an accelerator only: at level 0 the reference's
 * 3x3x5 coarse-cell scan always covers the query ball (SURVEY.md appendix A.1), so the result
 * is "every indexed vehicle with dist <= R"; any grid with cell >= R and a full 27-cell stencil
 * followed by the same exact distance filter returns the identical set.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* ------------------------------------------------------------------------------------------
 * constants: src/collision/collision_detection.py:19-28, src/collision/warning_system.py:18-27
 * ---------------------------------------------------------------------------------------- */
#define SAFE_DISTANCE_DEFAULT 5.0
#define MAX_WARNING_TIME 10.0
#define MAX_RELATIVE_SPEED 50.0
#define WEIGHT_DISTANCE 0.3
#define WEIGHT_TIME 0.3
#define WEIGHT_SPEED 0.2
#define WEIGHT_ANGLE 0.1
#define WEIGHT_TYPE 0.1
#define RISK_LEVEL_LOW 0.3
#define RISK_LEVEL_MEDIUM 0.6
#define RISK_LEVEL_HIGH 0.8

typedef struct {
    int64_t n;
    const double *px, *py, *pz, *vx, *vy, *vz, *ax, *ay, *az, *size, *heading;
    const int32_t *type;
} orc_frame;

/* one emitted risk; layout mirrored by oracle/oracle.py (numpy structured dtype) */
typedef struct {
    int32_t i, j;
    double ttc;        /* time_to_collision: k*0.1 (detect) or k*0.1 + t_m (predict) */
    double distance;   /* distance at the first hit sample */
    double rel_speed;  /* |v_i - v_j| */
    double risk;       /* risk_level in [0,1] */
    double cx, cy, cz; /* collision_position = midpoint */
    int32_t offset;    /* predict: winning offset index m (0..19); detect: -1 */
    int32_t priority;  /* alert class: -1 (risk < 0.3, no alert), 0..3 */
} orc_risk;

typedef struct {
    int32_t i, j;
    double tc; /* time_to_closest */
    double cd; /* closest_distance */
} orc_potential;

/* ---- scalar helpers ------------------------------------------------------------------- */

/* collision_detection.py:391-406 / spatial_index.py:285-300: sqrt of pow()-squares */
static inline double dist3(double x1, double y1, double z1, double x2, double y2, double z2) {
    return sqrt(pow(x1 - x2, 2.0) + pow(y1 - y2, 2.0) + pow(z1 - z2, 2.0));
}
/* collision_detection.py:408-418 */
static inline double mag3(double x, double y, double z) {
    return sqrt(pow(x, 2.0) + pow(y, 2.0) + pow(z, 2.0));
}
/* src/common/models.py:17-21 (Position.distance_to) and :30-32 (Vector.magnitude): ** 0.5 */
static inline double dist3_B(double x1, double y1, double z1, double x2, double y2, double z2) {
    return pow(pow(x1 - x2, 2.0) + pow(y1 - y2, 2.0) + pow(z1 - z2, 2.0), 0.5);
}
/* collision_detection.py:433-449: p + v*t + 0.5*a*t*t, Python precedence */
static inline double pos1(double p, double v, double a, double t) {
    return p + v * t + 0.5 * a * t * t;
}
/* collision_detection.py:484-496 */
static inline double safe_dist(double s1, double s2) { return (s1 + s2) / 2 + SAFE_DISTANCE_DEFAULT; }

/* collision_detection.py:344-389 (+ :498-513 type factor) */
double orc_risk_level(double heading_i, double heading_j, int32_t type_i, int32_t type_j,
                      double collision_time, double distance, double safe, double rel_speed) {
    double heading_diff = fabs(heading_i - heading_j);
    double angle_factor = sin(heading_diff);
    double type_factor = (type_i == type_j) ? 0.5 : 0.8;
    double distance_factor = 1.0 - (distance / safe);
    double r = collision_time / MAX_WARNING_TIME;
    double time_factor = 1.0 - (r < 1.0 ? r : 1.0);           /* min(1.0, r) */
    double s = rel_speed / MAX_RELATIVE_SPEED;
    double speed_factor = (s < 1.0 ? s : 1.0);                /* min(1.0, s) */
    double risk = (WEIGHT_DISTANCE * distance_factor + WEIGHT_TIME * time_factor +
                   WEIGHT_SPEED * speed_factor + WEIGHT_ANGLE * angle_factor +
                   WEIGHT_TYPE * type_factor);
    double m = (risk < 1.0 ? risk : 1.0);                     /* min(1.0, risk) */
    return (m > 0.0) ? m : 0.0;                               /* max(0.0, m) */
}

/* warning_system.py:259-311: gate (risk < 0.3 -> no alert = -1) then priority 0..3 */
int32_t orc_priority(double risk, double ttc) {
    if (risk < RISK_LEVEL_LOW) return -1;
    if (risk >= RISK_LEVEL_HIGH && ttc < 3.0) return 3;
    if (risk >= RISK_LEVEL_HIGH || ttc < 5.0) return 2;
    if (risk >= RISK_LEVEL_MEDIUM) return 1;
    return 0;
}

/* spatial_index.py:97-112 / compute_node.py:34-39: int(p / cell) truncates toward zero */
void orc_grid_id(double x, double y, double z, double cx, double cy, double cz, int64_t *out) {
    out[0] = (int64_t)(x / cx);
    out[1] = (int64_t)(y / cy);
    out[2] = (int64_t)(z / cz);
}

/* collision_detection.py:623-711: trajectory pattern from <=100 (position, timestamp) samples.
 * returns 0 stationary, 1 constant_velocity, 2 accelerating, 3 unknown (< 2 samples). */
int32_t orc_pattern(int32_t n, const double *x, const double *y, const double *z, const double *t) {
    if (n < 2) return 3;
    /* sorted(history, key=timestamp): stable insertion sort of indices */
    int32_t *ord = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
    for (int32_t k = 0; k < n; ++k) {
        int32_t p = k;
        while (p > 0 && t[ord[p - 1]] > t[k]) { ord[p] = ord[p - 1]; --p; }
        ord[p] = k;
    }
    double *vxs = (double *)malloc(sizeof(double) * 4 * (size_t)n);
    double *vys = vxs + n, *vzs = vys + n, *vts = vzs + n;
    int32_t nv = 0;
    for (int32_t k = 1; k < n; ++k) {
        int32_t a = ord[k - 1], b = ord[k];
        double dt = t[b] - t[a];
        if (dt > 0) {
            vxs[nv] = (x[b] - x[a]) / dt;
            vys[nv] = (y[b] - y[a]) / dt;
            vzs[nv] = (z[b] - z[a]) / dt;
            vts[nv] = t[b];
            ++nv;
        }
    }
    int32_t cls;
    if (nv == 0) {
        cls = 0; /* "stationary" (:654-655) */
    } else {
        double sax = 0, say = 0, saz = 0;
        int32_t na = 0;
        for (int32_t k = 1; k < nv; ++k) {
            double dt = vts[k] - vts[k - 1];
            if (dt > 0) {
                sax += (vxs[k] - vxs[k - 1]) / dt;
                say += (vys[k] - vys[k - 1]) / dt;
                saz += (vzs[k] - vzs[k - 1]) / dt;
                ++na;
            }
        }
        double svx = 0, svy = 0, svz = 0;
        for (int32_t k = 0; k < nv; ++k) { svx += vxs[k]; svy += vys[k]; svz += vzs[k]; }
        svx /= nv; svy /= nv; svz /= nv;
        if (na) { sax /= na; say /= na; saz /= na; }
        double speed = mag3(svx, svy, svz);
        double accel = mag3(sax, say, saz);
        cls = (speed < 0.1) ? 0 : ((accel < 0.1) ? 1 : 2);
    }
    free(vxs);
    free(ord);
    return cls;
}

/* orc_pattern for n histories in one call: samples[i][k] = (x, y, z, t) of history i, k < min(count[i], stride),
 * in insertion order (each history is sorted by orc_pattern itself). */
void orc_patterns(int64_t n, int32_t stride, const double *samples, const uint32_t *count, uint8_t *out) {
#pragma omp parallel
    {
        double *buf = (double *)malloc(sizeof(double) * 4 * (size_t)(stride > 0 ? stride : 1));
        double *x = buf, *y = buf + stride, *z = y + stride, *t = z + stride;
#pragma omp for schedule(static)
        for (int64_t i = 0; i < n; ++i) {
            int32_t c = count[i] < (uint32_t)stride ? (int32_t)count[i] : stride;
            const double *h = samples + (size_t)i * (size_t)stride * 4;
            for (int32_t k = 0; k < c; ++k) { x[k] = h[4 * k]; y[k] = h[4 * k + 1]; z[k] = h[4 * k + 2]; t[k] = h[4 * k + 3]; }
            out[i] = (uint8_t)orc_pattern(c, x, y, z, t);
        }
        free(buf);
    }
}

/* ---- uniform grid accelerator (not part of the reference semantics) --------------------- */
typedef struct {
    double ox, oy, oz, cell;
    int64_t nx, ny, nz;
    int32_t *start; /* ncells + 1 */
    int32_t *items; /* n, object indices grouped by cell, ascending index inside a cell */
} grid_t;

static inline int64_t cell_of(double x, double o, double cell) { return (int64_t)floor((x - o) / cell); }

static int grid_build(grid_t *g, const orc_frame *f, double radius) {
    int64_t n = f->n;
    double lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0};
    for (int64_t i = 0; i < n; ++i) {
        double p[3] = {f->px[i], f->py[i], f->pz[i]};
        for (int d = 0; d < 3; ++d) {
            if (i == 0 || p[d] < lo[d]) lo[d] = p[d];
            if (i == 0 || p[d] > hi[d]) hi[d] = p[d];
        }
    }
    double cell = radius > 1e-9 ? radius : 1e-9;
    for (;;) {
        g->nx = (int64_t)floor((hi[0] - lo[0]) / cell) + 1;
        g->ny = (int64_t)floor((hi[1] - lo[1]) / cell) + 1;
        g->nz = (int64_t)floor((hi[2] - lo[2]) / cell) + 1;
        double total = (double)g->nx * (double)g->ny * (double)g->nz;
        if (total <= 3.2e7) break;
        cell *= 1.5;
    }
    g->ox = lo[0]; g->oy = lo[1]; g->oz = lo[2]; g->cell = cell;
    int64_t nc = g->nx * g->ny * g->nz;
    g->start = (int32_t *)calloc((size_t)nc + 1, sizeof(int32_t));
    g->items = (int32_t *)malloc(sizeof(int32_t) * (size_t)(n > 0 ? n : 1));
    if (!g->start || !g->items) return -1;
    int64_t *cid = (int64_t *)malloc(sizeof(int64_t) * (size_t)(n > 0 ? n : 1));
    for (int64_t i = 0; i < n; ++i) {
        int64_t cx = cell_of(f->px[i], g->ox, cell), cy = cell_of(f->py[i], g->oy, cell),
                cz = cell_of(f->pz[i], g->oz, cell);
        if (cx >= g->nx) cx = g->nx - 1;
        if (cy >= g->ny) cy = g->ny - 1;
        if (cz >= g->nz) cz = g->nz - 1;
        cid[i] = (cz * g->ny + cy) * g->nx + cx;
        g->start[cid[i] + 1]++;
    }
    for (int64_t c = 0; c < nc; ++c) g->start[c + 1] += g->start[c];
    int32_t *cur = (int32_t *)malloc(sizeof(int32_t) * (size_t)nc);
    memcpy(cur, g->start, sizeof(int32_t) * (size_t)nc);
    for (int64_t i = 0; i < n; ++i) g->items[cur[cid[i]]++] = (int32_t)i;
    free(cur);
    free(cid);
    return 0;
}
static void grid_free(grid_t *g) { free(g->start); free(g->items); }

/* growable per-thread output */
typedef struct { void *data; int64_t n, cap; size_t elem; } vec_t;
static void vec_init(vec_t *v, size_t elem) { v->data = NULL; v->n = 0; v->cap = 0; v->elem = elem; }
static void *vec_push(vec_t *v) {
    if (v->n == v->cap) {
        v->cap = v->cap ? v->cap * 2 : 256;
        v->data = realloc(v->data, v->elem * (size_t)v->cap);
    }
    return (char *)v->data + v->elem * (size_t)(v->n++);
}

static int cmp_risk(const void *a, const void *b) {
    const orc_risk *x = (const orc_risk *)a, *y = (const orc_risk *)b;
    if (x->i != y->i) return x->i < y->i ? -1 : 1;
    if (x->j != y->j) return x->j < y->j ? -1 : 1;
    return 0;
}
static int cmp_pot(const void *a, const void *b) {
    const orc_potential *x = (const orc_potential *)a, *y = (const orc_potential *)b;
    if (x->i != y->i) return x->i < y->i ? -1 : 1;
    if (x->j != y->j) return x->j < y->j ? -1 : 1;
    return 0;
}
static int cmp_i32(const void *a, const void *b) {
    int32_t x = *(const int32_t *)a, y = *(const int32_t *)b;
    return x < y ? -1 : (x > y);
}

/* visit every object in the 27 cells around point (x,y,z); cell >= radius so this is a superset */
#define FOR_NEIGHBOURS(g, x, y, z, J, ...)                                                      \
    do {                                                                                        \
        int64_t _cx = cell_of((x), (g)->ox, (g)->cell), _cy = cell_of((y), (g)->oy, (g)->cell), \
                _cz = cell_of((z), (g)->oz, (g)->cell);                                         \
        /* objects on the upper boundary were clamped into the last cell */                     \
        for (int64_t _z = _cz - 1; _z <= _cz + 1; ++_z) {                                       \
            if (_z < 0 || _z >= (g)->nz) continue;                                              \
            for (int64_t _y = _cy - 1; _y <= _cy + 1; ++_y) {                                   \
                if (_y < 0 || _y >= (g)->ny) continue;                                          \
                int64_t _x0 = _cx - 1 < 0 ? 0 : _cx - 1;                                        \
                int64_t _x1 = _cx + 1 >= (g)->nx ? (g)->nx - 1 : _cx + 1;                       \
                if (_x0 > _x1) continue;                                                        \
                int64_t _b = (_z * (g)->ny + _y) * (g)->nx;                                     \
                for (int32_t _s = (g)->start[_b + _x0]; _s < (g)->start[_b + _x1 + 1]; ++_s) {  \
                    int32_t J = (g)->items[_s];                                                 \
                    __VA_ARGS__                                                                 \
                }                                                                               \
            }                                                                                   \
        }                                                                                       \
    } while (0)

/* collision_detection.py:296-342: first sample k (t = k*step) with distance <= safe.
 * (pxi..) are the two start states; returns k or -1; dist_out / mid get the hit values. */
static int precise_hit(double pix, double piy, double piz, double vix, double viy, double viz,
                       double aix, double aiy, double aiz, double pjx, double pjy, double pjz,
                       double vjx, double vjy, double vjz, double ajx, double ajy, double ajz,
                       double safe, double time_window, double *dist_out, double *mid) {
    const double time_step = 0.1;
    int steps = (int)(time_window / time_step);
    for (int k = 0; k < steps; ++k) {
        double t = k * time_step;
        double xi = pos1(pix, vix, aix, t), yi = pos1(piy, viy, aiy, t), zi = pos1(piz, viz, aiz, t);
        double xj = pos1(pjx, vjx, ajx, t), yj = pos1(pjy, vjy, ajy, t), zj = pos1(pjz, vjz, ajz, t);
        double d = dist3(xi, yi, zi, xj, yj, zj);
        if (d <= safe) {
            *dist_out = d;
            mid[0] = (xi + xj) / 2; mid[1] = (yi + yj) / 2; mid[2] = (zi + zj) / 2;
            return k;
        }
    }
    return -1;
}

/* CollisionDetector._precise_collision_detection (collision_detection.py:296-342) for one pair of vehicles:
 * a, b = {px, py, pz, vx, vy, vz, ax, ay, az, size}.  Returns the index of the first sample inside the safe
 * distance (-1: None); out = {collision_time, distance, safe_distance, relative_speed, mid x, y, z}. */
int32_t orc_precise(const double *a, const double *b, double time_window, double *out) {
    const double safe = safe_dist(a[9], b[9]);
    double dist = 0.0, mid[3] = {0.0, 0.0, 0.0};
    const int k = precise_hit(a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], a[8], b[0], b[1], b[2], b[3], b[4], b[5],
                              b[6], b[7], b[8], safe, time_window, &dist, mid);
    out[0] = k * 0.1;
    out[1] = dist;
    out[2] = safe;
    out[3] = mag3(a[3] - b[3], a[4] - b[4], a[5] - b[5]);
    out[4] = mid[0]; out[5] = mid[1]; out[6] = mid[2];
    return k;
}

/* ------------------------------------------------------------------------------------------
 * detect(i) for one vehicle: collision_detection.py:110-191 (stages :208-389).
 * ---------------------------------------------------------------------------------------- */
static void detect_one(const orc_frame *f, const grid_t *g, int32_t i, double R, double T,
                       uint32_t *cand_count, vec_t *cands, vec_t *pots, vec_t *risks) {
    double pix = f->px[i], piy = f->py[i], piz = f->pz[i];
    uint32_t nc = 0;
    FOR_NEIGHBOURS(g, pix, piy, piz, j, {
        if (j == i) continue;                                  /* :224-225 */
        double cur0 = dist3(pix, piy, piz, f->px[j], f->py[j], f->pz[j]); /* spatial_index.py:266 */
        if (!(cur0 <= R)) continue;                            /* spatial_index.py:268 */
        ++nc;
        if (cands) { int32_t *c = (int32_t *)vec_push(cands); c[0] = i; c = (int32_t *)vec_push(cands); c[0] = j; }
        /* ---- stage 2, :244-292 ---- */
        double cur = dist3(pix, piy, piz, f->px[j], f->py[j], f->pz[j]);
        double rvx = f->vx[i] - f->vx[j], rvy = f->vy[i] - f->vy[j], rvz = f->vz[i] - f->vz[j];
        double rpx = f->px[j] - pix, rpy = f->py[j] - piy, rpz = f->pz[j] - piz;
        double rs = mag3(rvx, rvy, rvz);
        if (rs < 0.1) continue;
        double dot = rpx * rvx + rpy * rvy + rpz * rvz;
        if (dot > 0 && cur > SAFE_DISTANCE_DEFAULT) continue;
        double tc = -dot / (rs * rs);
        if (tc < 0 || tc > T) continue;
        double cd = dist3(pos1(pix, f->vx[i], f->ax[i], tc), pos1(piy, f->vy[i], f->ay[i], tc),
                          pos1(piz, f->vz[i], f->az[i], tc), pos1(f->px[j], f->vx[j], f->ax[j], tc),
                          pos1(f->py[j], f->vy[j], f->ay[j], tc), pos1(f->pz[j], f->vz[j], f->az[j], tc));
        double safe = safe_dist(f->size[i], f->size[j]);
        if (cd > safe) continue;
        if (pots) { orc_potential *p = (orc_potential *)vec_push(pots); p->i = i; p->j = j; p->tc = tc; p->cd = cd; }
        /* ---- stage 3, :296-342 ---- */
        double d, mid[3];
        int k = precise_hit(pix, piy, piz, f->vx[i], f->vy[i], f->vz[i], f->ax[i], f->ay[i], f->az[i],
                            f->px[j], f->py[j], f->pz[j], f->vx[j], f->vy[j], f->vz[j], f->ax[j],
                            f->ay[j], f->az[j], safe, T, &d, mid);
        if (k < 0) continue;
        double ct = k * 0.1;
        /* ---- stage 4, :344-389 ---- */
        double risk = orc_risk_level(f->heading[i], f->heading[j], f->type[i], f->type[j], ct, d, safe, rs);
        orc_risk *r = (orc_risk *)vec_push(risks);
        r->i = i; r->j = j; r->ttc = ct; r->distance = d; r->rel_speed = rs; r->risk = risk;
        r->cx = mid[0]; r->cy = mid[1]; r->cz = mid[2]; r->offset = -1;
        r->priority = orc_priority(risk, ct);
    });
    if (cand_count) cand_count[i] = nc;
}

/* ------------------------------------------------------------------------------------------
 * predict(i): collision_detection.py:572-865.  pattern: 0 stationary, 1 constant_velocity,
 * 2 accelerating / unknown.  (pattern 3 = history < 2 -> detect(i), handled by the caller.)
 * ---------------------------------------------------------------------------------------- */
static void predict_one(const orc_frame *f, const grid_t *g, int32_t i, int32_t pattern,
                        uint32_t *cand_count, vec_t *risks, vec_t *scratch) {
    int64_t first = risks->n;
    uint32_t nc = 0;
    (void)scratch;
    for (int m = 0; m < 20; ++m) {
        double t = 0.5 * m; /* np.arange(0, 10, 0.5)[m] is exactly m*0.5 */
        double cx, cy, cz;
        if (pattern == 0) {                        /* :728-731 */
            cx = f->px[i]; cy = f->py[i]; cz = f->pz[i];
        } else if (pattern == 1) {                 /* :733-741 */
            cx = f->px[i] + f->vx[i] * t; cy = f->py[i] + f->vy[i] * t; cz = f->pz[i] + f->vz[i] * t;
        } else {                                   /* :743-761 */
            cx = pos1(f->px[i], f->vx[i], f->ax[i], t);
            cy = pos1(f->py[i], f->vy[i], f->ay[i], t);
            cz = pos1(f->pz[i], f->vz[i], f->az[i], t);
        }
        FOR_NEIGHBOURS(g, cx, cy, cz, j, {
            if (j == i) continue;
            /* :801-803 + spatial_index.py:261-269: others at their CURRENT positions */
            double dq = dist3(cx, cy, cz, f->px[j], f->py[j], f->pz[j]);
            if (!(dq <= 100.0)) continue;
            ++nc;
            /* :814 other predicted position */
            double qx = pos1(f->px[j], f->vx[j], f->ax[j], t), qy = pos1(f->py[j], f->vy[j], f->ay[j], t),
                   qz = pos1(f->pz[j], f->vz[j], f->az[j], t);
            double safe = safe_dist(f->size[i], f->size[j]);
            double d, mid[3];
            int k = precise_hit(cx, cy, cz, f->vx[i], f->vy[i], f->vz[i], f->ax[i], f->ay[i], f->az[i],
                                qx, qy, qz, f->vx[j], f->vy[j], f->vz[j], f->ax[j], f->ay[j], f->az[j],
                                safe, 1.0, &d, mid);
            if (k < 0) continue;
            double ct = k * 0.1;
            double rs = mag3(f->vx[i] - f->vx[j], f->vy[i] - f->vy[j], f->vz[i] - f->vz[j]);
            double risk = orc_risk_level(f->heading[i], f->heading[j], f->type[i], f->type[j], ct, d, safe, rs);
            double ttc = ct + t;                   /* :835 */
            /* merge (:848-865): strict >, offsets ascending */
            orc_risk *slot = NULL;
            orc_risk *base = (orc_risk *)risks->data;
            for (int64_t q = first; q < risks->n; ++q) if (base[q].j == j) { slot = &base[q]; break; }
            if (!slot) {
                slot = (orc_risk *)vec_push(risks);
                slot->risk = -1.0;
            }
            if (risk > slot->risk) {
                slot->i = i; slot->j = j; slot->ttc = ttc; slot->distance = d; slot->rel_speed = rs;
                slot->risk = risk; slot->cx = mid[0]; slot->cy = mid[1]; slot->cz = mid[2];
                slot->offset = m; slot->priority = orc_priority(risk, ttc);
            }
        });
    }
    if (cand_count) cand_count[i] = nc;
}

/* ------------------------------------------------------------------------------------------
 * frame drivers.  mode 0: detect for all; mode 1: predict with per-vehicle pattern (3 -> detect).
 * Outputs are written sorted by (i, j).  Returns 0, or -1 if a capacity was exceeded (counts
 * still exact).  counts[0]=#directed candidates, [1]=#potentials, [2]=#risks, [3]=#risk>0.7.
 * ---------------------------------------------------------------------------------------- */
int orc_frame_A(int64_t n, const double *px, const double *py, const double *pz, const double *vx,
                const double *vy, const double *vz, const double *ax, const double *ay,
                const double *az, const double *size, const double *heading, const int32_t *type,
                int32_t mode, const uint8_t *pattern, double R, double T, int32_t threads,
                int64_t q_stride /* query only objects with i % q_stride == 0 (CPU-baseline sampling) */,
                uint32_t *cand_count /* n or NULL */, int32_t *cand_pairs /* 2*cand_cap or NULL */,
                int64_t cand_cap, orc_potential *pots_out, int64_t pot_cap, orc_risk *risks_out,
                int64_t risk_cap, int64_t *counts) {
    orc_frame f = {n, px, py, pz, vx, vy, vz, ax, ay, az, size, heading, type};
    grid_t g;
    counts[0] = counts[1] = counts[2] = counts[3] = 0;
    if (n <= 0) return 0;
    double gr = (mode == 1 && R < 100.0) ? 100.0 : R;
    if (grid_build(&g, &f, gr) != 0) return -2;
#ifdef _OPENMP
    int nt = threads > 0 ? threads : omp_get_max_threads();
#else
    int nt = 1;
    (void)threads;
#endif
    /* contiguous chunks of vehicles, many more than threads for balance under density skew */
    int64_t chunk = 256;
    int64_t nchunks = (n + chunk - 1) / chunk;
    vec_t *vc = (vec_t *)malloc(sizeof(vec_t) * (size_t)nchunks * 3);
    uint32_t *ccount = cand_count ? cand_count : (uint32_t *)calloc((size_t)n, sizeof(uint32_t));
#pragma omp parallel for schedule(dynamic, 1) num_threads(nt)
    for (int64_t c = 0; c < nchunks; ++c) {
        vec_t *cands = &vc[c * 3], *pots = &vc[c * 3 + 1], *risks = &vc[c * 3 + 2];
        vec_init(cands, sizeof(int32_t));
        vec_init(pots, sizeof(orc_potential));
        vec_init(risks, sizeof(orc_risk));
        int64_t lo = c * chunk, hi = lo + chunk < n ? lo + chunk : n;
        for (int64_t i = lo; i < hi; ++i) {
            if (q_stride > 1 && (i % q_stride) != 0) continue;
            int64_t r0 = risks->n, p0 = pots->n, c0 = cands->n;
            int pat = (mode == 1 && pattern) ? pattern[i] : (mode == 1 ? 2 : 3);
            if (mode == 0 || pat == 3)
                detect_one(&f, &g, (int32_t)i, mode == 0 ? R : 100.0, mode == 0 ? T : 10.0, ccount,
                           cand_pairs ? cands : NULL, pots, risks);
            else
                predict_one(&f, &g, (int32_t)i, pat, ccount, risks, NULL);
            /* canonical order inside one vehicle: ascending j */
            if (risks->n - r0 > 1)
                qsort((orc_risk *)risks->data + r0, (size_t)(risks->n - r0), sizeof(orc_risk), cmp_risk);
            if (pots->n - p0 > 1)
                qsort((orc_potential *)pots->data + p0, (size_t)(pots->n - p0), sizeof(orc_potential), cmp_pot);
            if (cands->n - c0 > 2) {
                /* pairs are (i, j) with constant i: sort the j's */
                int64_t m = (cands->n - c0) / 2;
                int32_t *tmp = (int32_t *)malloc(sizeof(int32_t) * (size_t)m);
                int32_t *cd = (int32_t *)cands->data + c0;
                for (int64_t q = 0; q < m; ++q) tmp[q] = cd[2 * q + 1];
                qsort(tmp, (size_t)m, sizeof(int32_t), cmp_i32);
                for (int64_t q = 0; q < m; ++q) cd[2 * q + 1] = tmp[q];
                free(tmp);
            }
        }
    }
    int rc = 0;
    int64_t nc = 0, np = 0, nr = 0, nh = 0;
    for (int64_t i = 0; i < n; ++i) nc += ccount[i];
    int64_t wc = 0;
    for (int64_t c = 0; c < nchunks; ++c) {
        vec_t *cands = &vc[c * 3], *pots = &vc[c * 3 + 1], *risks = &vc[c * 3 + 2];
        if (cand_pairs) {
            int64_t m = cands->n / 2;
            if (wc + m <= cand_cap) memcpy(cand_pairs + 2 * wc, cands->data, sizeof(int32_t) * 2 * (size_t)m);
            else rc = -1;
            wc += m;
        }
        if (pots_out) {
            if (np + pots->n <= pot_cap) memcpy(pots_out + np, pots->data, sizeof(orc_potential) * (size_t)pots->n);
            else rc = -1;
        }
        np += pots->n;
        if (risks_out) {
            if (nr + risks->n <= risk_cap) memcpy(risks_out + nr, risks->data, sizeof(orc_risk) * (size_t)risks->n);
            else rc = -1;
        }
        for (int64_t q = 0; q < risks->n; ++q) if (((orc_risk *)risks->data)[q].risk > 0.7) ++nh;
        nr += risks->n;
        free(cands->data); free(pots->data); free(risks->data);
    }
    counts[0] = nc; counts[1] = np; counts[2] = nr; counts[3] = nh;
    if (!cand_count) free(ccount);
    free(vc);
    grid_free(&g);
    return rc;
}

/* ------------------------------------------------------------------------------------------
 * impl. B frame (src/compute/compute_node.py:98-119 query_nearby + :229-321 detect_collisions;
 * VehicleState.predict_position :192-212 needs >= 2 samples -> has_history flag).
 * Output orc_risk: ttc = formula time_to_collision (quirk Q10), distance = future_distance,
 * offset = -1, priority = -1 (B has no alert stage).
 * ---------------------------------------------------------------------------------------- */
int orc_frame_B(int64_t n, const double *px, const double *py, const double *pz, const double *vx,
                const double *vy, const double *vz, const uint8_t *has_history, double radius,
                double prediction_time, double risk_threshold, int32_t threads,
                uint32_t *cand_count, orc_risk *risks_out, int64_t risk_cap, int64_t *counts) {
    orc_frame f = {n, px, py, pz, vx, vy, vz, NULL, NULL, NULL, NULL, NULL, NULL};
    grid_t g;
    counts[0] = counts[1] = counts[2] = counts[3] = 0;
    if (n <= 0) return 0;
    if (grid_build(&g, &f, radius) != 0) return -2;
#ifdef _OPENMP
    int nt = threads > 0 ? threads : omp_get_max_threads();
#else
    int nt = 1;
    (void)threads;
#endif
    const double vehicle_radius = 2.0;
    int64_t chunk = 256, nchunks = (n + chunk - 1) / chunk;
    vec_t *vc = (vec_t *)malloc(sizeof(vec_t) * (size_t)nchunks);
    uint32_t *ccount = cand_count ? cand_count : (uint32_t *)calloc((size_t)n, sizeof(uint32_t));
#pragma omp parallel for schedule(dynamic, 1) num_threads(nt)
    for (int64_t c = 0; c < nchunks; ++c) {
        vec_t *risks = &vc[c];
        vec_init(risks, sizeof(orc_risk));
        int64_t lo = c * chunk, hi = lo + chunk < n ? lo + chunk : n;
        for (int64_t ii = lo; ii < hi; ++ii) {
            int32_t i = (int32_t)ii;
            int64_t r0 = risks->n;
            uint32_t ncand = 0;
            FOR_NEIGHBOURS(&g, px[i], py[i], pz[i], j, {
                /* query_nearby (:112-117) returns self too (quirk Q8); counted as a candidate */
                double dq = dist3_B(px[i], py[i], pz[i], px[j], py[j], pz[j]);
                if (!(dq <= radius)) continue;
                ++ncand;
                if (j == i) continue;                                         /* :251-252 */
                double cur = dist3_B(px[i], py[i], pz[i], px[j], py[j], pz[j]); /* :259 */
                if (cur > 50.0) continue;                                     /* :262 */
                if (!has_history[i] || !has_history[j]) continue;            /* :266-270 */
                double fix = px[i] + vx[i] * prediction_time, fiy = py[i] + vy[i] * prediction_time,
                       fiz = pz[i] + vz[i] * prediction_time;
                double fjx = px[j] + vx[j] * prediction_time, fjy = py[j] + vy[j] * prediction_time,
                       fjz = pz[j] + vz[j] * prediction_time;
                double fut = dist3_B(fix, fiy, fiz, fjx, fjy, fjz);           /* :273 */
                double rvx = vx[i] - vx[j], rvy = vy[i] - vy[j], rvz = vz[i] - vz[j];
                double rs = pow(pow(rvx, 2.0) + pow(rvy, 2.0) + pow(rvz, 2.0), 0.5); /* :281 */
                if (fut > cur && cur > vehicle_radius * 2) continue;          /* :284 */
                double min_distance = fut > 0.1 ? fut : 0.1;                  /* max(0.1, fut) */
                double rl = (vehicle_radius * 2) / min_distance * rs / 10.0;  /* :289 */
                double risk = rl < 1.0 ? rl : 1.0;                           /* min(1.0, rl) */
                if (risk < risk_threshold) continue;                          /* :292 */
                double ttc = prediction_time;                                 /* :296-301 */
                if (fut < vehicle_radius * 2) {
                    if (cur > fut) {
                        double ratio = (cur - vehicle_radius * 2) / (cur - fut);
                        double v = prediction_time * ratio;
                        ttc = v > 0.1 ? v : 0.1;                              /* max(0.1, v) */
                    }
                }
                orc_risk *r = (orc_risk *)vec_push(risks);
                r->i = i; r->j = j; r->ttc = ttc; r->distance = fut; r->rel_speed = rs; r->risk = risk;
                r->cx = (fix + fjx) / 2; r->cy = (fiy + fjy) / 2; r->cz = (fiz + fjz) / 2;
                r->offset = -1; r->priority = -1;
            });
            ccount[i] = ncand;
            if (risks->n - r0 > 1)
                qsort((orc_risk *)risks->data + r0, (size_t)(risks->n - r0), sizeof(orc_risk), cmp_risk);
        }
    }
    int rc = 0;
    int64_t nc = 0, nr = 0;
    for (int64_t i = 0; i < n; ++i) nc += ccount[i];
    for (int64_t c = 0; c < nchunks; ++c) {
        vec_t *risks = &vc[c];
        if (risks_out) {
            if (nr + risks->n <= risk_cap) memcpy(risks_out + nr, risks->data, sizeof(orc_risk) * (size_t)risks->n);
            else rc = -1;
        }
        nr += risks->n;
        free(risks->data);
    }
    counts[0] = nc; counts[2] = nr;
    if (!cand_count) free(ccount);
    free(vc);
    grid_free(&g);
    return rc;
}

/* radius query for explicit points: spatial_index.py:229-271 (self NOT stripped, quirk Q8).
 * out_offsets has nq+1 entries; ids for query q are out_ids[out_offsets[q] .. out_offsets[q+1]),
 * ascending.  Returns 0 or -1 if cap exceeded (offsets still exact). */
int orc_query_radius(int64_t n, const double *px, const double *py, const double *pz, int64_t nq,
                     const double *qx, const double *qy, const double *qz, double radius,
                     int32_t variant_B, int64_t *out_offsets, int32_t *out_ids, int64_t cap) {
    orc_frame f = {n, px, py, pz, NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL};
    grid_t g;
    out_offsets[0] = 0;
    if (n <= 0) { for (int64_t q = 0; q < nq; ++q) out_offsets[q + 1] = 0; return 0; }
    if (grid_build(&g, &f, radius) != 0) return -2;
    int rc = 0;
    int64_t w = 0;
    for (int64_t q = 0; q < nq; ++q) {
        int64_t w0 = w;
        FOR_NEIGHBOURS(&g, qx[q], qy[q], qz[q], j, {
            double d = variant_B ? dist3_B(qx[q], qy[q], qz[q], px[j], py[j], pz[j])
                                 : dist3(qx[q], qy[q], qz[q], px[j], py[j], pz[j]);
            if (d <= radius) {
                if (w < cap) out_ids[w] = j; else rc = -1;
                ++w;
            }
        });
        if (rc == 0 && w - w0 > 1) qsort(out_ids + w0, (size_t)(w - w0), sizeof(int32_t), cmp_i32);
        out_offsets[q + 1] = w;
    }
    grid_free(&g);
    return rc;
}

int orc_max_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}
