// fcpp_plan.cu — the fused per-plan kernel: path sampling -> geofence tests -> curvature limit ->
// forward/backward min-plus scans -> kinematic validation -> path metrics.  One CTA per plan;
// the whole plan (x, y, u, class) lives in shared memory, only results go to HBM.
//
// Reference code replaced ("mlp3" = multi_layer_planner_v3.py):
//   A4  swaths + 20-pt half-circle turns            mlp3:720-830, rotate-back :709-714
//   A5  headland loops (straights, corner arcs)      mlp3:943-1011, :1013-1022, :1580-1608
//   A6  reverse fills                                mlp3:1066-1080, :1213-1216
//   A7  curvature limit + accel passes               mlp3:467-589
//   A8  lateral-acceleration validation              mlp3:1373-1424
//   A9  geofence / obstacle point tests              D3 (no reference code; README.md:24,200)
//   A13 path length / work time                      mlp3:1290-1311
//
// plan_gen_kernel: the plan is generated.  A plan is made of congruent pieces (fcpp_internal.cuh): the main work is a
// sequence of 22-point chains (turn + next swath) separated by zero-length segments that the acceleration passes do
// not cross, all but the first and the last congruent — they are speed-planned and validated ONCE per candidate and
// their points only generated, tested against the geofence / obstacles and written; the headland's straights,
// corner turns and reverse fills take segment length, curvature and speed limit from a per-candidate table; only
// the points where two pieces meet (~5 % of a plan) are evaluated from their coordinates (sqrt, atan2, divisions).
// path_kernel / path_big_kernel: A7/A8/A13 on caller-supplied paths (verify_curvature_constraints(path, speeds) of
// the drop-in API), every point evaluated from the coordinates.
#include "fcpp_internal.cuh"

namespace {

constexpr int T0 = FCPP_PLAN_THREADS;  // threads per CTA of the smallest variant; path_kernel also runs at 2x and 4x

// generated plans (plan_gen_kernel, plan_gen_omega_kernel)
struct PlanArgs {
    fcpp_batch b;
    const CandRec *recs;
    const TrigTables *trig;
    fcpp_outputs out;
    int obs_cap_verts; // smem capacity for obstacle vertices
    int obs_cap_polys;
    int ncap;          // smem capacity in staged points
};

// caller-supplied paths (path_kernel, path_big_kernel)
struct PathArgs {
    fcpp_vehicle veh;
    const double *in_path;
    const double *in_speeds;
    const int64_t *in_offsets;
    int do_speed_plan;
    double *speeds_kmh;
    double *curvature;
    fcpp_summary *summary;
    int ncap;          // smem capacity in points
    int nmin;          // this launch handles nmin < N <= ncap (tiers by path length, see launch_tiers)
    int defer;         // 1: a later launch with a larger staging handles N > ncap
    // paths longer than the shared-memory staging go through path_big_kernel (HBM/L2 staging)
    int big_enabled;          // regular kernel: leave paths with N > ncap to the big kernel
    int big_ncap;             // big kernel: point capacity of one CTA's scratch slice
    unsigned char *big_scratch;
    int64_t big_stride;       // bytes per CTA slice
    int64_t n_items;          // paths in the batch
};

// per-candidate table entry of a structure slot: segment length to the next point, curvature, curvature-limited
// speed (km/h) and its u = (v / 3.6)^2, time of the segment with the initial speeds
struct Tpl {
    double ds, kap, u, vl, tpre;
};
constexpr int TPL_PTS = 48;  // scratch points of the table set-up: 24 main + 15 turn samples

// staging of the caller-supplied-path kernels: x -> ds, y -> kappa, u per point + reduction scratch
struct Smem {
    double *X, *Y, *U;
    double *scratch;   // [SCRATCH]
};

__host__ __device__ inline size_t align16(size_t x) { return (x + 15) & ~size_t(15); }

constexpr int SCRATCH = 320;  // block reductions: 9 values x 32 warps
__host__ __device__ inline size_t plan_smem_bytes(int ncap)
{
    return 3 * align16(sizeof(double) * ncap) + align16(sizeof(double) * SCRATCH);
}

__device__ inline Smem carve(unsigned char *base, int ncap)
{
    Smem s;
    const size_t arr = align16(sizeof(double) * ncap);
    s.scratch = (double *)base;
    base += align16(sizeof(double) * SCRATCH);
    s.X = (double *)base;
    s.Y = (double *)(base + arr);
    s.U = (double *)(base + 2 * arr);
    return s;
}

// ---------------------------------------------------------------------------------------------
// min-plus scan element: the map u -> min(M, u + C)
// ---------------------------------------------------------------------------------------------
struct MP {
    double C, M;
};
__device__ __forceinline__ MP mp_combine(const MP &a, const MP &b)  // a first, then b
{
    MP r;
    r.C = a.C + b.C;
    r.M = fmin(b.M, a.M + b.C);
    return r;
}
__device__ __forceinline__ MP mp_shfl_up(const MP &v, int d)
{
    MP r;
    r.C = __shfl_up_sync(0xffffffffu, v.C, d);
    r.M = __shfl_up_sync(0xffffffffu, v.M, d);
    return r;
}

// exclusive block scan of per-thread aggregates in thread order; returns the carry-in value
// (the M of the composition of all earlier threads; +inf for thread 0)
__device__ __forceinline__ double mp_block_exclusive(MP agg, double *sh /*>= 2*NWARP*/, int tid)
{
    const int lane = tid & 31, warp = tid >> 5;
    MP inc = agg;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const MP o = mp_shfl_up(inc, d);
        if (lane >= d) inc = mp_combine(o, inc);
    }
    if (lane == 31) {
        sh[2 * warp] = inc.C;
        sh[2 * warp + 1] = inc.M;
    }
    __syncthreads();
    // composition of all earlier warps (serial over the few warps of the CTA)
    MP pre;
    pre.C = 0.0;
    pre.M = INFINITY;
    for (int w = 0; w < warp; ++w) {
        MP o;
        o.C = sh[2 * w];
        o.M = sh[2 * w + 1];
        pre = mp_combine(pre, o);
    }
    // exclusive within the warp
    MP ex = mp_shfl_up(inc, 1);
    if (lane == 0) {
        ex.C = 0.0;
        ex.M = INFINITY;
    }
    const MP tot = mp_combine(pre, ex);
    __syncthreads();
    return tot.M;
}

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    return v;
}
__device__ __forceinline__ double warp_max(double v)
{
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, d));
    return v;
}

// reduce NV sums / maxes across the CTA (deterministic order); result valid in thread 0
template <int NV, bool IS_MAX, int NWARP>
__device__ __forceinline__ void block_reduce(double (&v)[NV], double *sh, int tid)
{
    const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int k = 0; k < NV; ++k) v[k] = IS_MAX ? warp_max(v[k]) : warp_sum(v[k]);
    __syncthreads();
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < NV; ++k) sh[warp * NV + k] = v[k];
    }
    __syncthreads();
    if (tid == 0) {
#pragma unroll
        for (int k = 0; k < NV; ++k) {
            double a = sh[k];
            for (int w = 1; w < NWARP; ++w) a = IS_MAX ? fmax(a, sh[w * NV + k]) : a + sh[w * NV + k];
            v[k] = a;
        }
    }
}

__device__ __forceinline__ double cls_speed(const fcpp_vehicle &v, uint8_t c)
{
    return c == CLS_WORK ? v.max_work_speed_kmh
                         : (c == CLS_TURN ? v.headland_turn_speed_kmh
                                          : (c == CLS_HEAD ? v.max_headland_speed_kmh : v.reverse_speed_kmh));
}

// x / 3.6, correctly rounded, in three instructions instead of the generic FP64 division
// (Markstein: with r = RN(1/y) and q0 = RN(x r), RN(q0 + r RN(x - y q0)) = RN(x / y) whenever the
// significand of y is not all ones; checked here against the division on 1.5e9 random doubles).
// The km/h <-> m/s conversions of the reference (mlp3:498, :564-566, :580-582, :1306, :1389) are
// the most frequent divisions of this kernel; the result is bit-identical to `x / 3.6`.
__device__ __forceinline__ double div36(double x)
{
    if (!(fabs(x) < 1e150)) return x / 3.6;  // inf / nan / absurd magnitudes: the generic path
    const double r = 1.0 / 3.6;
    const double q0 = x * r;
    return fma(fma(-q0, 3.6, x), r, q0);
}

// FP64 sqrt and division take a ~70-instruction slow path when the radicand / numerator is zero,
// and one zero lane (a zero-length segment, a straight joint) drags its whole warp through it.
// The zero lanes are fed a harmless operand and get their exact result (0) by a select.
// (the substitution is opaque inline PTX: written as a C++ select the compiler proves
// sqrt(0) == 0 and 0 / den == 0, folds the select away and the slow path is back)
__device__ __forceinline__ double one_if_zero(double x)
{
    double r;
    asm("{\n\t.reg .pred p;\n\tsetp.eq.f64 p, %1, 0d0000000000000000;\n\t"
        "selp.f64 %0, 0d3FF0000000000000, %1, p;\n\t}"
        : "=d"(r)
        : "d"(x));
    return r;
}
__device__ __forceinline__ double sqrt_z(double q)
{
    const double r = sqrt(one_if_zero(q));
    return (q == 0.0) ? 0.0 : r;
}
__device__ __forceinline__ double div_z(double num, double den)  // den > 0
{
    const double r = one_if_zero(num) / den;
    return (num == 0.0) ? 0.0 : r;
}

// mlp3:513-536 with the three atan2 folded into one: dtheta = atan2(d1 x d2, d1 . d2)
__device__ __forceinline__ double curvature3(double dx1, double dy1, double ds1, double dx2, double dy2,
                                             double ds2)
{
    if (ds1 < FCPP_ZERO_LEN || ds2 < FCPP_ZERO_LEN) return 0.0;
    const double cr = dx1 * dy2 - dy1 * dx2;
    const double dt = dx1 * dx2 + dy1 * dy2;
    // collinear joints (cr == 0): atan2(+-0, dt) is 0 for dt > 0 and +-pi for dt < 0; only |dtheta| is used
    const bool col = (cr == 0.0);
    const double at = atan2(one_if_zero(cr), dt);
    const double dth = col ? (dt < 0.0 ? 3.141592653589793 : 0.0) : at;
    return fabs(div_z(2 * dth, ds1 + ds2));
}

// curvature speed limit in km/h (mlp3:496-503)
__device__ __forceinline__ double vlimit(double v0, double kappa, const fcpp_vehicle &v)
{
    if (kappa > FCPP_KAPPA_EPS) {
        const double vmax = sqrt(v.max_lateral_accel / kappa) * v.safety_factor * 3.6;
        if (v0 > vmax) return vmax;
    }
    return v0;
}

// ---------------------------------------------------------------------------------------------
// GEN: one generated plan per CTA
// ---------------------------------------------------------------------------------------------
#ifndef FCPP_PLAN_GEN_THREADS
#define FCPP_PLAN_GEN_THREADS 128
#endif
constexpr int TG = FCPP_PLAN_GEN_THREADS;
#ifndef FCPP_PLAN_GEN_MIN_CTAS
// CTAs of 128 threads per SM the register allocation aims at.  Measured (tools/cover_ab.py, plan kernel of config
// 2 / 5 / 3): 8 CTAs (64 registers, 308 B of spills) 0.207 / 0.624 / 4.50 ms, 7 (72 registers) 0.193 / 0.602 / 4.20,
// 6 (80) 0.203 / 0.598 / 4.25, 5 (96) 0.220 / 0.641 / 4.36, 4 (120, no spills) 0.240 / 0.680 / 4.80.
#define FCPP_PLAN_GEN_MIN_CTAS 7
#endif
static_assert(TG >= 128 && TG % 32 == 0, "the table set-up uses threads 0 .. 96 + 4 * FCPP_MAX_LOOPS - 1 in two rounds");

// shared memory of the generated-plan kernel: fixed part (compile-time offsets) + obstacle tables + the staging of
// the `ncap` staged points (first 2 + last 22 main points + headland): ds, kappa, u (FP64) and the structure tag
constexpr int MIXED_CAP = 510;  // listed passes; a pass beyond the list is tested by the thread that classified it
struct GenFixed {
    CandRec rec;
    TrigTables tt;
    Tpl tbl[N_SLOTS];
    double tpts[2 * TPL_PTS];
    double geo[20];              // [4][5] field edges of the geofence test: ax, ay, ex, ey, threshold
    double gelen[4];             // |e| of the four edges
    uint16_t mixed[MIXED_CAP];   // main passes whose turn samples need the per-point tests (phase 0c)
    int32_t n_mixed;
    double gvl[N_GENERIC];       // curvature-limited speed of the generic points
    double scratch[9 * (FCPP_PLAN_GEN_THREADS / 32) + 8];  // block reductions: 9 values per warp; scans: 2 per warp
    union {
        struct {
            double chain_v[CHAIN_POINTS];  // final speed (km/h) of the regular chain's points
            double chain_sum[8];           // per regular chain: length, time (initial speeds), time (final speeds),
                                           // accel violations, max kappa, max a_lat, max kappa jump
        };
        double omega_part[8 * (FCPP_PLAN_GEN_THREADS / 32)];  // Ω pattern (no regular chain): the same sums of all
                                                              // chains, per warp
    };
    int32_t glist[N_GENERIC];    // point index of generic ordinal g (-1: none)
    uint64_t bar;
};
struct GenSmem {
    GenFixed *f;
    double *obs_xy;    // [obs_cap_verts][2]
    double *obs_bb;    // [obs_cap_polys][4] bbox of each obstacle grown by W/2 + 1e-6 (early reject)
    int32_t *obs_vs;   // [obs_cap_polys + 1], relative to the field's first vertex
    double *X, *Y, *U;
    uint8_t *TAG;
};
__host__ __device__ inline size_t gen_smem_bytes(int ncap, int obs_verts, int obs_polys)
{
    size_t s = align16(sizeof(GenFixed));
    s += align16(sizeof(double) * 2 * (obs_verts > 0 ? obs_verts : 1));
    s += align16(sizeof(double) * 4 * (obs_polys > 0 ? obs_polys : 1));
    s += align16(sizeof(int32_t) * (obs_polys + 1));
    s += 3 * align16(sizeof(double) * ncap) + align16(ncap);
    return s;
}
__device__ __forceinline__ GenSmem gen_carve(unsigned char *base, int ncap, int obs_verts, int obs_polys)
{
    GenSmem s;
    s.f = reinterpret_cast<GenFixed *>(base);
    size_t o = align16(sizeof(GenFixed));
    s.obs_xy = (double *)(base + o);
    o += align16(sizeof(double) * 2 * (obs_verts > 0 ? obs_verts : 1));
    s.obs_bb = (double *)(base + o);
    o += align16(sizeof(double) * 4 * (obs_polys > 0 ? obs_polys : 1));
    s.obs_vs = (int32_t *)(base + o);
    o += align16(sizeof(int32_t) * (obs_polys + 1));
    const size_t arr = align16(sizeof(double) * ncap);
    s.X = (double *)(base + o);
    s.Y = (double *)(base + o + arr);
    s.U = (double *)(base + o + 2 * arr);
    s.TAG = (uint8_t *)(base + o + 3 * arr);
    return s;
}

// a / b for a finite a >= 0 and a normal b > 0 (speeds >= 0.1 m/s): reciprocal seed + two Newton steps + one
// residual correction — correctly rounded in all but the rarest cases (the sums it feeds are compared at 1e-9),
// a third of the instructions of the generic division and no slow path
__device__ __forceinline__ double div_pos(double a, double b)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(b));
    r = fma(fma(-b, r, 1.0), r, r);
    r = fma(fma(-b, r, 1.0), r, r);
    const double q = a * r;
    return fma(fma(-b, q, a), r, q);
}

// final speed of a point from its scanned u (mlp3:558-587): the km/h limit comes back verbatim when the scans
// left it alone, else 3.6 sqrt(u); the square root only runs in warps where some lane needs it.
// Must be called by all 32 lanes of the warp.
__device__ __forceinline__ double final_speed(bool act, double u, double u_lim, double vl)
{
    const bool need = act && (u != u_lim);
    double v = vl;
    if (__any_sync(0xffffffffu, need)) {
        const double sq = sqrt(need ? u : 1.0);
        if (need) v = 3.6 * sq;
    }
    return v;
}

// geofence (D3) and obstacle (D2/D3) point tests of one generated point (point_tests_impl, fcpp_internal.cuh)
__device__ __forceinline__ void point_tests(const GenSmem &s, int n_obs_poly, double r2, double x, double y, int &n_bviol,
                                            int &n_oviol)
{
    const int m = point_tests_impl(s.f->geo, s.obs_xy, s.obs_bb, s.obs_vs, n_obs_poly, r2, x, y);
    n_bviol += m & 1;
    n_oviol += m >> 1;
}


// One generated plan by the TG threads of a CTA (tid = 0 .. TG-1).
template <bool OMEGA = false>
__device__ __forceinline__ void plan_gen_body(const PlanArgs &a, unsigned char *smem, const int tid, const int64_t cand)
{
    constexpr int T = TG;
    const GenSmem s = gen_carve(smem, a.ncap, a.obs_cap_verts, a.obs_cap_polys);
    GenFixed &f = *s.f;
    const int lane = tid & 31;
    const fcpp_vehicle &veh = a.b.vehicle;
    fcpp_summary *sum = a.out.summary ? a.out.summary + cand : nullptr;
    if (tid == 0) mbar_init(&f.bar, 1);
    __syncthreads();

    int n_obs_poly = 0;
    {
        // stage the candidate record (and the field's obstacle vertices) with TMA bulk copies
        if (tid == 0) {
            const int fi = a.recs[cand].field;
            uint32_t bytes = sizeof(CandRec);
            int v0 = 0, nv = 0;
            if (a.b.obs_poly_start) {
                const int p0 = a.b.obs_poly_start[fi], p1 = a.b.obs_poly_start[fi + 1];
                v0 = a.b.obs_vert_start[p0];
                nv = a.b.obs_vert_start[p1] - v0;
                if (nv > a.obs_cap_verts) nv = a.obs_cap_verts;
                bytes += nv * 16;
            }
            mbar_expect_tx(&f.bar, bytes);
            bulk_g2s(&f.rec, a.recs + cand, sizeof(CandRec), &f.bar);
            if (nv > 0) bulk_g2s(s.obs_xy, a.b.obs_verts + 2 * (int64_t)v0, nv * 16, &f.bar);
        }
        // trig tables through the ordinary path meanwhile; the generic-point list starts empty
        for (int k = tid; k < (int)(sizeof(TrigTables) / sizeof(double)); k += T)
            ((double *)&f.tt)[k] = ((const double *)a.trig)[k];
        for (int k = tid; k < N_GENERIC; k += T) f.glist[k] = -1;
        // ONE thread polls the mbarrier, the CTA barrier releases the rest, and every thread then observes the
        // completed phase itself (acquire of the async-proxy writes)
        if (tid == 0)
            while (!mbar_try_wait(&f.bar, 0)) {
            }
        __syncthreads();
        while (!mbar_try_wait(&f.bar, 0)) {
        }
    }
    const CandRec &r = f.rec;
    if (a.b.obs_poly_start) {
        const int p0 = a.b.obs_poly_start[r.field], p1 = a.b.obs_poly_start[r.field + 1];
        n_obs_poly = min(p1 - p0, a.obs_cap_polys);
        const int base = a.b.obs_vert_start[p0];
        for (int k = tid; k <= n_obs_poly; k += T) s.obs_vs[k] = a.b.obs_vert_start[p0 + k] - base;
    }
    const int N = r.n_total, n_main = r.n_main;
    FCPP_ASSERT(gen_smem_bytes(a.ncap, a.obs_cap_verts, a.obs_cap_polys) <= fcpp_dynamic_smem_bytes() + 0u);
    const int n_skip = main_skip(n_main);  // regular chain points: i in [2, 2 + n_skip)
    const int NS = N - n_skip;             // staged points
    const int64_t off = a.out.offsets ? a.out.offsets[cand] : 0;
    if (sum && tid == 0) {
        sum->n_passes = r.P;
        sum->n_loops = r.K;
        sum->n_main = r.n_main;
        sum->n_head = r.n_head;
        sum->n_rev[0] = r.n_rev[0];
        sum->n_rev[1] = r.n_rev[1];
        sum->n_rev[2] = r.n_rev[2];
        sum->corner_g = r.corner_g;
    }
    {
        int st = r.status;
        if (NS > a.ncap) st |= FCPP_CAND_TOO_LARGE;
        // the paths of this plan would not fit the caller's buffers (sized from an earlier batch)
        if (a.out.path_capacity > 0 && off + N > a.out.path_capacity) st |= FCPP_CAND_TOO_LARGE;
        if (st != 0 || N == 0) {
            if (sum && tid == 0) {
                sum->status = st;
                sum->n_accel_viol = sum->n_boundary_viol = sum->n_obstacle_viol = 0;
                sum->len_main = sum->len_head = sum->time_main = sum->time_head = 0.0;
                sum->time_main_pre = sum->time_head_pre = 0.0;
                sum->max_curvature = sum->max_lateral_accel = sum->max_jump = 0.0;
                sum->reserved = 0.0;
                if (!a.b.do_coverage) {
                    sum->cov_cells = sum->cov_total = 0;
                    for (int k = 0; k < 4; ++k) sum->corner_before[k] = sum->corner_after[k] = 0;
                }
            }
            return;
        }
    }
    __syncthreads();  // obs_vs is complete
    const double W = veh.working_width;
    TurnModel tm;
    tm.model = a.b.turn_model;
    tm.lam = a.b.clothoid_share;
    const double rr = W / 2;
    const double r2 = rr * rr;
    const double two_a = 2 * veh.max_longitudinal_accel;
    const bool do_scan = N >= 3;

    // ------------------------------------------------------------------------------------
    // phase 0: per-candidate tables.  Scratch points of the first main pass (+ the first two points of the
    // second) in the swath frame and of one corner turn; geofence edges; obstacle boxes.
    // ------------------------------------------------------------------------------------
    if (tid < 24) {
        if (r.P >= 2) {
            double px, py;
            main_local_pt<OMEGA>(r, f.tt, tm, W, tid < 22 ? 0 : 1, tid < 22 ? tid : tid - 22, px, py);
            f.tpts[2 * tid] = px;
            f.tpts[2 * tid + 1] = py;
        }
    } else if (tid >= 32 && tid < 32 + FCPP_CORNER_POINTS) {
        double px, py;
        corner_arc_pt(f.tt, tm, 0.0, 0.0, r.R, 0, tid - 32, px, py);
        f.tpts[2 * (tid - 8)] = px;  // scratch points 24 .. 38
        f.tpts[2 * (tid - 8) + 1] = py;
    } else if (tid >= 64 && tid < 68) {
        // field edges for the D3 test: cross(e, p - v) < -eps*|e|
        const int k = tid - 64, k1 = (k + 1) & 3;
        const double ax = a.b.field_verts[(int64_t)r.field * 8 + 2 * k], ay = a.b.field_verts[(int64_t)r.field * 8 + 2 * k + 1];
        const double ex = a.b.field_verts[(int64_t)r.field * 8 + 2 * k1] - ax;
        const double ey = a.b.field_verts[(int64_t)r.field * 8 + 2 * k1 + 1] - ay;
        f.geo[5 * k] = ax;
        f.geo[5 * k + 1] = ay;
        f.geo[5 * k + 2] = ex;
        f.geo[5 * k + 3] = ey;
        const double el = sqrt(ex * ex + ey * ey);
        f.geo[5 * k + 4] = -FCPP_GEOFENCE_EPS * el;
        f.gelen[k] = el;
    }
    // early-reject boxes: a point outside an obstacle's bbox grown by W/2 (+1e-6 m, far above any rounding of the
    // exact test) can neither be inside it nor within W/2 of an edge
    for (int p = tid - 96; p < n_obs_poly; p += T) {
        if (p < 0) continue;
        double x0 = 1e300, y0 = 1e300, x1 = -1e300, y1 = -1e300;
        for (int q = s.obs_vs[p]; q < s.obs_vs[p + 1]; ++q) {
            x0 = fmin(x0, s.obs_xy[2 * q]);
            x1 = fmax(x1, s.obs_xy[2 * q]);
            y0 = fmin(y0, s.obs_xy[2 * q + 1]);
            y1 = fmax(y1, s.obs_xy[2 * q + 1]);
        }
        s.obs_bb[4 * p] = x0 - rr - 1e-6;
        s.obs_bb[4 * p + 1] = y0 - rr - 1e-6;
        s.obs_bb[4 * p + 2] = x1 + rr + 1e-6;
        s.obs_bb[4 * p + 3] = y1 + rr + 1e-6;
    }
    __syncthreads();
    // one thread per table slot (two rounds when the CTA has fewer threads than slots' thread ids)
    for (int vt = tid; vt < 96 + 4 * FCPP_MAX_LOOPS; vt += T) {
        int slot = -1;
        double ds = 0.0, kap = 0.0, v0 = 0.0, v1 = 0.0;
        if (vt < CHAIN_POINTS) {
            if (r.P >= 2) {
                // chain point c = scratch point c + 2: turn samples of pass 0, then the two ends of swath 1
                const int c = vt;
                slot = SLOT_CHAIN + c;
                const double *p = f.tpts + 2 * (c + 2);
                const double d1x = p[0] - p[-2], d1y = p[1] - p[-1];
                if (c < CHAIN_POINTS - 1) {
                    const double d2x = p[2] - p[0], d2y = p[3] - p[1];
                    ds = sqrt_z(d2x * d2x + d2y * d2y);
                    kap = curvature3(d1x, d1y, sqrt_z(d1x * d1x + d1y * d1y), d2x, d2y, ds);
                }  // the chain's last point is followed by its own copy (the next turn's first sample): ds = kappa = 0
                v0 = (c < FCPP_UTURN_POINTS) ? veh.headland_turn_speed_kmh : veh.max_work_speed_kmh;
                v1 = (c < FCPP_UTURN_POINTS - 1) ? veh.headland_turn_speed_kmh : veh.max_work_speed_kmh;
            }
        } else if (vt >= 32 && vt < 32 + FCPP_CORNER_POINTS) {
            const int aI = vt - 32;
            if (aI >= 1 && aI <= FCPP_CORNER_POINTS - 2) {
                slot = SLOT_ARC + aI;
                const double *p = f.tpts + 2 * 24;
                const double d1x = p[2 * aI] - p[2 * (aI - 1)], d1y = p[2 * aI + 1] - p[2 * (aI - 1) + 1];
                const double d2x = p[2 * (aI + 1)] - p[2 * aI], d2y = p[2 * (aI + 1) + 1] - p[2 * aI + 1];
                ds = sqrt_z(d2x * d2x + d2y * d2y);
                kap = curvature3(d1x, d1y, sqrt_z(d1x * d1x + d1y * d1y), d2x, d2y, ds);
                v0 = v1 = veh.headland_turn_speed_kmh;
            }
        } else if (vt >= 64 && vt < 67) {
            const int t = vt - 64;
            if (r.n_rev[t] >= 2) {  // points ex + (m step) d: equally spaced, collinear (mlp3:1214-1216)
                slot = SLOT_REV + t;
                const double step = r.rev[t][4] / (r.n_rev[t] - 1);
                const double sx = step * r.rev[t][2], sy = step * r.rev[t][3];
                ds = sqrt_z(sx * sx + sy * sy);
                v0 = v1 = veh.reverse_speed_kmh;
            }
        } else if (vt >= 96 && vt < 96 + 4 * r.K) {
            const int kt = vt - 96, k = kt >> 2, t = kt & 3;
            const int sc = r.flags & FCPP_FLAG_CORNER_MASK, ci = (sc + t) & 3, ni = (sc + t + 1) & 3;
            slot = SLOT_STRAIGHT + kt;
            constexpr double DIV = FCPP_STRAIGHT_POINTS - 1;
            const double sx = div_const(r.corners[k][ni][0] - r.corners[k][ci][0], DIV, 1.0 / DIV);
            const double sy = div_const(r.corners[k][ni][1] - r.corners[k][ci][1], DIV, 1.0 / DIV);
            ds = sqrt_z(sx * sx + sy * sy);
            v0 = v1 = veh.max_headland_speed_kmh;
        }
        if (slot >= 0) {
            const double vl = vlimit(v0, kap, veh);
            const double vms = div36(vl);
            Tpl e;
            e.ds = ds;
            e.kap = kap;
            e.vl = vl;
            e.u = vms * vms;
            e.tpre = div_z(ds, fmax(div36((v0 + v1) / 2), FCPP_MIN_SPEED_MS));
            f.tbl[slot] = e;
        }
    }
    __syncthreads();

    // ------------------------------------------------------------------------------------
    // phase 0c (summary-only batches): the turns of the regular main passes, classified per PASS.  The 20 turn samples
    // of main pass idx and the swath end they start from lie on the circle of radius R around (min_x or max_x, y of
    // the pass) in the swath frame (mlp3:815-823).  When that disc, grown by 1e-6 m (six orders of magnitude above
    // the rounding of either test), misses every obstacle's grown box and
    //   * is inside all four field edges (cross(e, c - v) >= (R + 1e-6) |e|): none of the 21 points fails a test;
    //   * is outside one edge (cross <= -(R + 1e-6) |e|): every one of them is a boundary violation, nothing else
    //     (swaths span the bounding box of the rotated work area, mlp3:736-737, so on sheared or rotated fields most
    //     turns are of this kind);
    // either way the points are only COUNTED.  Every other pass goes on a list and phase 1b generates and tests the
    // points of the listed passes only — a dense index space, so warps stay full.  The swaths' far ends are always
    // tested.  (Clothoid turns are wider than the disc, and with materialised paths every point is generated
    // anyway: no classification then.)
    // ------------------------------------------------------------------------------------
    constexpr bool omega = OMEGA;  // the Ω pattern has its own kernel instance (launch: turn_model == FCPP_TURN_OMEGA)
    const bool cull = n_skip > 0 && !a.out.path_xy && !a.out.speeds_kmh && !a.out.curvature &&
                      tm.model == FCPP_TURN_ARC;
    const int i_end = 2 + n_skip;  // regular chain points: i in [2, i_end)
    int n_bviol = 0, n_oviol = 0;
    auto main_pt = [&](int idx, int j, double &x, double &y) {
        double px, py;
        main_local_pt<OMEGA>(r, f.tt, tm, W, idx, j, px, py);
        if (r.flags & FCPP_FLAG_ROTATED)
            rotate_pt(px, py, r.cos_a, r.sin_a, r.cx, r.cy, x, y);  // mlp3:709-714
        else {
            x = px;
            y = py;
        }
    };
    if (cull) {
        if (tid == 0) f.n_mixed = 0;
        __syncthreads();
        const double rad = r.R + 1e-6;
        for (int idx = tid; idx * CHAIN_POINTS + 1 < i_end; idx += T) {
            // the pass's points j >= 1 inside the regular range (pass 0: its two ends are staged)
            const int lo = idx == 0 ? 2 : 1, hi = min(CHAIN_POINTS, i_end - idx * CHAIN_POINTS);
            if (hi <= lo) continue;
            const int pi = (r.flags & FCPP_FLAG_REVERSE_ORDER) ? (r.P - 1 - idx) : idx;
            const double py = r.min_y + pi * W;
            const bool go_left = (r.flags & FCPP_FLAG_START_FROM_RIGHT) ? ((idx & 1) == 0) : ((idx & 1) == 1);
            const double px = go_left ? r.min_x : r.max_x;
            double x = px, y = py;
            if (r.flags & FCPP_FLAG_ROTATED) rotate_pt(px, py, r.cos_a, r.sin_a, r.cx, r.cy, x, y);
            bool clear = true;
            for (int p = 0; p < n_obs_poly && clear; ++p)
                clear = x + rad < s.obs_bb[4 * p] || y + rad < s.obs_bb[4 * p + 1] || x - rad > s.obs_bb[4 * p + 2] ||
                        y - rad > s.obs_bb[4 * p + 3];
            bool in = clear, out = false;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const double cr = f.geo[5 * k + 2] * (y - f.geo[5 * k + 1]) - f.geo[5 * k + 3] * (x - f.geo[5 * k]);
                const double lim = rad * f.gelen[k];
                in = in && (cr >= lim);
                out = out || (cr <= -lim);
            }
            if (in) continue;
            if (out && clear) {
                n_bviol += hi - lo;
                continue;
            }
            const int pos = idx < 65536 ? atomicAdd(&f.n_mixed, 1) : MIXED_CAP;
            if (pos < MIXED_CAP) {
                FCPP_ASSERT(pos >= 0 && idx >= 0 && idx < r.P);
                f.mixed[pos] = (uint16_t)idx;
            } else {  // (a plan with more than MIXED_CAP unclassifiable passes, or more than 65 535 passes)
                for (int j = lo; j < hi; ++j) {
                    double qx, qy;
                    main_pt(idx, j, qx, qy);
                    point_tests(s, n_obs_poly, r2, qx, qy, n_bviol, n_oviol);
                }
            }
        }
    }

    // ------------------------------------------------------------------------------------
    // phase 0b (warp 0): the regular chain once — acceleration passes over its 22 points (a zero-length segment
    // precedes and follows it, so it is a closed system, mlp3:560, :576), final speeds, validation, sums
    // ------------------------------------------------------------------------------------
    if (tid < 32 && n_skip > 0 && !omega) {
        const bool on = lane < CHAIN_POINTS;
        const Tpl e = f.tbl[SLOT_CHAIN + (on ? lane : 0)];
        const double ds_prev = __shfl_up_sync(0xffffffffu, e.ds, 1);
        // forward: element c = (increment from c-1, U_c); the chain starts behind a zero-length segment
        MP inc;
        inc.C = (on && lane > 0 && !(ds_prev < FCPP_ZERO_LEN)) ? two_a * ds_prev : INFINITY;
        inc.M = on ? e.u : INFINITY;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const MP o = mp_shfl_up(inc, d);
            if (lane >= d) inc = mp_combine(o, inc);
        }
        const double fwd = inc.M;
        // backward over the mirrored lanes: lane l holds chain point 21 - l
        const int src = CHAIN_POINTS - 1 - lane;  // valid for lane < 22
        const double f_m = __shfl_sync(0xffffffffu, fwd, src & 31);
        const double ds_m = __shfl_sync(0xffffffffu, e.ds, src & 31);  // ds of the mirrored point = increment to ITS successor
        MP b;
        b.C = (on && !(ds_m < FCPP_ZERO_LEN)) ? two_a * ds_m : INFINITY;  // applied when coming from the successor
        b.M = on ? f_m : INFINITY;
        // scan element for the mirrored order: value_l = min(M_l, value_{l-1} + C_l) with C_l = increment between
        // point (21-l) and its successor (21-l+1) = ds of point 21-l
        if (lane == 0) b.C = INFINITY;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const MP o = mp_shfl_up(b, d);
            if (lane >= d) b = mp_combine(o, b);
        }
        const double u_fin = __shfl_sync(0xffffffffu, b.M, src & 31);  // back to chain order
        const double v = do_scan ? final_speed(on, u_fin, e.u, e.vl) : e.vl;
        const double v_next = __shfl_down_sync(0xffffffffu, v, 1);
        const double k_next = __shfl_down_sync(0xffffffffu, e.kap, 1);
        double t_adj = 0.0, alat = 0.0, jump = 0.0;
        if (on) {
            f.chain_v[lane] = v;
            if (lane < CHAIN_POINTS - 1) {
                t_adj = div_pos(e.ds, fmax(div36((v + v_next) / 2), FCPP_MIN_SPEED_MS));
                jump = fabs(k_next - e.kap);
            }
            const double vm = div36(v);
            alat = vm * vm * e.kap;
        }
        const double s_len = warp_sum(on ? e.ds : 0.0), s_tpre = warp_sum(on ? e.tpre : 0.0), s_tadj = warp_sum(t_adj);
        const double s_av = warp_sum((on && alat > veh.max_lateral_accel) ? 1.0 : 0.0);
        const double m_k = warp_max(on ? e.kap : 0.0), m_a = warp_max(alat), m_j = warp_max(jump);
        if (lane == 0) {
            f.chain_sum[0] = s_len;
            f.chain_sum[1] = s_tpre;
            f.chain_sum[2] = s_tadj;
            f.chain_sum[3] = s_av;
            f.chain_sum[4] = m_k;
            f.chain_sum[5] = m_a;
            f.chain_sum[6] = m_j;
        }
    }

    // ------------------------------------------------------------------------------------
    // phase 1: the staged points (first 2 + last 22 main points, headland): points -> HBM (when paths are
    // materialised) + point tests; ds / kappa / U of every point inside a congruent headland piece from the
    // table; the generic points are listed by their fixed ordinal
    // ------------------------------------------------------------------------------------
    double acc_len_m = 0.0, acc_len_h = 0.0, acc_tpre_m = 0.0, acc_tpre_h = 0.0;
    double2 *gp = a.out.path_xy ? reinterpret_cast<double2 *>(a.out.path_xy) + off : nullptr;
    double *gs = a.out.speeds_kmh ? a.out.speeds_kmh + off : nullptr;
    double *gk = a.out.curvature ? a.out.curvature + off : nullptr;
    for (int q = tid; q < NS; q += T) {
        const int i = q < 2 ? q : q + n_skip;
        double x, y;
        uint8_t c;
        int tag, gord;
        gen_point_tag<OMEGA>(r, f.tt, tm, W, i, x, y, c, tag, gord);
        FCPP_ASSERT(q >= 0 && q < a.ncap && i >= 0 && i < N && gord < N_GENERIC && (gord >= 0 || (tag >= 0 && tag < N_SLOTS)));
        if (gp) gp[i] = make_double2(x, y);
        s.TAG[q] = (uint8_t)tag;
        if (gord >= 0) {
            f.glist[gord] = i;
        } else {
            const Tpl e = f.tbl[tag];
            s.X[q] = e.ds;
            s.Y[q] = e.kap;
            s.U[q] = e.u;
            acc_len_h += e.ds;  // table slots of staged points are headland pieces
            acc_tpre_h += e.tpre;
        }
        point_tests(s, n_obs_poly, r2, x, y, n_bviol, n_oviol);
    }
    __syncthreads();  // glist, chain_v
    // ------------------------------------------------------------------------------------
    // phase 1b: the regular chains' points (most of a plan): generated, tested, written with the chain's speeds
    // ------------------------------------------------------------------------------------
    if constexpr (OMEGA) {
        // Ω pattern: the chains (turn + next swath) are not congruent — the gap between consecutive rows varies —
        // so every regular chain is evaluated from its coordinates, ONE WARP PER CHAIN (lane = chain point): segment
        // lengths, curvature, limit, the two acceleration passes by shuffles (the chain is a closed system: a
        // zero-length segment precedes and follows it), validation, sums, outputs
        double o_len = 0.0, o_tpre = 0.0, o_t = 0.0, o_av = 0.0, o_k = 0.0, o_a = 0.0, o_j = 0.0;
        for (int c = tid >> 5; c < n_skip / CHAIN_POINTS; c += T / 32) {
            const bool on = lane < CHAIN_POINTS;
            const int i = 2 + c * CHAIN_POINTS + (on ? lane : 0);
            const int idx = i / CHAIN_POINTS, j = i - idx * CHAIN_POINTS;
            double x, y;
            main_pt(idx, j, x, y);
            const double xp = __shfl_up_sync(0xffffffffu, x, 1), yp = __shfl_up_sync(0xffffffffu, y, 1);
            const double xn = __shfl_down_sync(0xffffffffu, x, 1), yn = __shfl_down_sync(0xffffffffu, y, 1);
            // the chain's first point repeats the swath end before it, its last point is repeated by the next turn
            const double dx1 = lane > 0 ? x - xp : 0.0, dy1 = lane > 0 ? y - yp : 0.0;
            const double dx2 = lane < CHAIN_POINTS - 1 ? xn - x : 0.0, dy2 = lane < CHAIN_POINTS - 1 ? yn - y : 0.0;
            const double ds1 = sqrt_z(dx1 * dx1 + dy1 * dy1), ds = sqrt_z(dx2 * dx2 + dy2 * dy2);
            const double kap = curvature3(dx1, dy1, ds1, dx2, dy2, ds);
            const double v0 = (lane < FCPP_UTURN_POINTS) ? veh.headland_turn_speed_kmh : veh.max_work_speed_kmh;
            const double vl = vlimit(v0, kap, veh);
            const double vms = div36(vl);
            const double u_lim = vms * vms;
            const double v0n = __shfl_down_sync(0xffffffffu, v0, 1);
            MP inc;
            inc.C = (on && lane > 0 && !(ds1 < FCPP_ZERO_LEN)) ? two_a * ds1 : INFINITY;
            inc.M = on ? u_lim : INFINITY;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const MP o = mp_shfl_up(inc, d);
                if (lane >= d) inc = mp_combine(o, inc);
            }
            const double fwd = inc.M;
            const int src = CHAIN_POINTS - 1 - lane;  // backward pass over the mirrored lanes
            const double f_m = __shfl_sync(0xffffffffu, fwd, src & 31);
            const double ds_m = __shfl_sync(0xffffffffu, ds, src & 31);
            MP bk;
            bk.C = (on && lane > 0 && !(ds_m < FCPP_ZERO_LEN)) ? two_a * ds_m : INFINITY;
            bk.M = on ? f_m : INFINITY;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const MP o = mp_shfl_up(bk, d);
                if (lane >= d) bk = mp_combine(o, bk);
            }
            const double u_fin = __shfl_sync(0xffffffffu, bk.M, src & 31);
            const double v = do_scan ? final_speed(on, u_fin, u_lim, vl) : vl;
            const double v_next = __shfl_down_sync(0xffffffffu, v, 1);
            const double k_next = __shfl_down_sync(0xffffffffu, kap, 1);
            if (on) {
                if (gp) gp[i] = make_double2(x, y);
                if (gs) gs[i] = v;
                if (gk) gk[i] = kap;
                point_tests(s, n_obs_poly, r2, x, y, n_bviol, n_oviol);
                if (lane < CHAIN_POINTS - 1) {
                    o_len += ds;
                    o_tpre += div_z(ds, fmax(div36((v0 + v0n) / 2), FCPP_MIN_SPEED_MS));
                    o_t += div_z(ds, fmax(div36((v + v_next) / 2), FCPP_MIN_SPEED_MS));
                    o_j = fmax(o_j, fabs(k_next - kap));
                }
                const double vm = div36(v);
                const double alat = vm * vm * kap;
                o_av += (alat > veh.max_lateral_accel) ? 1.0 : 0.0;
                o_k = fmax(o_k, kap);
                o_a = fmax(o_a, alat);
            }
        }
        // per-warp partials in a fixed order (deterministic sums); thread 0 adds them to the plan's totals
        o_len = warp_sum(o_len), o_tpre = warp_sum(o_tpre), o_t = warp_sum(o_t), o_av = warp_sum(o_av);
        o_k = warp_max(o_k), o_a = warp_max(o_a), o_j = warp_max(o_j);
        if (lane == 0) {
            double *part = f.omega_part + 8 * (tid >> 5);
            part[0] = o_len, part[1] = o_tpre, part[2] = o_t, part[3] = o_av, part[4] = o_k, part[5] = o_a, part[6] = o_j;
        }
    }
    if (!omega && !cull) {
        for (int i = 2 + tid; i < i_end; i += T) {
            const int idx = i / CHAIN_POINTS;
            const int j = i - idx * CHAIN_POINTS;
            double x, y;
            main_pt(idx, j, x, y);
            const int c = j >= 2 ? j - 2 : j + FCPP_UTURN_POINTS;  // position in its chain
            if (gp) gp[i] = make_double2(x, y);
            if (gs) gs[i] = f.chain_v[c];
            if (gk) gk[i] = f.tbl[SLOT_CHAIN + c].kap;
            point_tests(s, n_obs_poly, r2, x, y, n_bviol, n_oviol);
        }
    } else if (!omega) {
        // the swaths' far ends (j = 0) of passes 1 ...; then the points of the listed passes, densely indexed
        for (int idx = 1 + tid; idx * CHAIN_POINTS < i_end; idx += T) {
            double x, y;
            main_pt(idx, 0, x, y);
            point_tests(s, n_obs_poly, r2, x, y, n_bviol, n_oviol);
        }
        const int n_listed = min(f.n_mixed, MIXED_CAP);
        for (int k = tid; k < n_listed * (CHAIN_POINTS - 1); k += T) {
            const int m = k / (CHAIN_POINTS - 1);
            const int idx = f.mixed[m], j = 1 + (k - m * (CHAIN_POINTS - 1));
            if ((idx == 0 && j < 2) || idx * CHAIN_POINTS + j >= i_end) continue;
            double x, y;
            main_pt(idx, j, x, y);
            point_tests(s, n_obs_poly, r2, x, y, n_bviol, n_oviol);
        }
    }
    // ------------------------------------------------------------------------------------
    // phase 2: the generic points (where two pieces meet, the irregular main points) from their coordinates
    // (mlp3:490-504): the point and its two neighbours are regenerated
    // ------------------------------------------------------------------------------------
    const int n_gslots = MAIN_STAGED + GEN_PER_LOOP * r.K;
    for (int g = tid; g < n_gslots; g += T) {
        const int i = f.glist[g];
        if (i < 0) continue;
        double P3[3][2] = {{0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}};
        uint8_t C3[3] = {0, 0, 0};
#pragma unroll 1
        for (int d = 0; d < 3; ++d) {
            const int qq = i - 1 + d;
            if (qq >= 0 && qq < N) gen_point<OMEGA>(r, f.tt, tm, W, qq, P3[d][0], P3[d][1], C3[d]);
        }
        const double dx1 = P3[1][0] - P3[0][0], dy1 = P3[1][1] - P3[0][1];
        const double dx2 = P3[2][0] - P3[1][0], dy2 = P3[2][1] - P3[1][1];
        double ds1 = 0.0, ds2 = 0.0;
        if (i > 0) ds1 = sqrt_z(dx1 * dx1 + dy1 * dy1);
        if (i + 1 < N) ds2 = sqrt_z(dx2 * dx2 + dy2 * dy2);
        double kap = 0.0;
        if (i >= 1 && i + 1 < N) kap = curvature3(dx1, dy1, ds1, dx2, dy2, ds2);
        const double v0 = cls_speed(veh, C3[1]);
        const double vl = vlimit(v0, kap, veh);
        const double vms = div36(vl);
        const int q = i < 2 ? i : i - n_skip;
        FCPP_ASSERT(q >= 0 && q < NS && NS <= a.ncap && g < N_GENERIC);
        s.X[q] = ds2;
        s.Y[q] = kap;
        s.U[q] = vms * vms;
        f.gvl[g] = vl;
        // per-layer length and pre-adjustment time (mlp3:616-617, :882-883)
        if (i + 1 < N && i != n_main - 1) {
            const double t = div_z(ds2, fmax(div36((v0 + cls_speed(veh, C3[2])) / 2), FCPP_MIN_SPEED_MS));
            if (i < n_main) {
                acc_len_m += ds2;
                acc_tpre_m += t;
            } else {
                acc_len_h += ds2;
                acc_tpre_h += t;
            }
        }
    }
    __syncthreads();

    // ------------------------------------------------------------------------------------
    // phases 3 / 4 over the staged sequence (the zero-length segment after point 1 separates the two staged ends
    // of the main work): forward f = min(U, f_prev + 2a ds_prev) (mlp3:558-571), backward (mlp3:574-587)
    // ------------------------------------------------------------------------------------
    const int chunk = (NS + T - 1) / T;
    const int cs = min(NS, tid * chunk);
    const int ce = min(NS, cs + chunk);
    if (do_scan) {
        {
            MP agg;
            agg.C = 0.0;
            agg.M = INFINITY;
            for (int q = cs; q < ce; ++q) {
                const double dsp = (q > 0) ? s.X[q - 1] : 0.0;
                const double c = (q > 0 && !(dsp < FCPP_ZERO_LEN)) ? two_a * dsp : INFINITY;
                agg.M = fmin(s.U[q], agg.M + c);
                agg.C = agg.C + c;
            }
            double carry = mp_block_exclusive(agg, f.scratch, tid);
            for (int q = cs; q < ce; ++q) {
                const double dsp = (q > 0) ? s.X[q - 1] : 0.0;
                const double c = (q > 0 && !(dsp < FCPP_ZERO_LEN)) ? two_a * dsp : INFINITY;
                carry = fmin(s.U[q], carry + c);
                s.U[q] = carry;
            }
        }
        __syncthreads();
        {
            const int rt = T - 1 - tid;
            const int rs = min(NS, rt * chunk);
            const int re = min(NS, rs + chunk);
            MP agg;
            agg.C = 0.0;
            agg.M = INFINITY;
            for (int q = re - 1; q >= rs; --q) {
                const double dsn = s.X[q];  // ds to the successor (0 for the last point)
                const double c = (q + 1 < NS && !(dsn < FCPP_ZERO_LEN)) ? two_a * dsn : INFINITY;
                agg.M = fmin(s.U[q], agg.M + c);
                agg.C = agg.C + c;
            }
            double carry = mp_block_exclusive(agg, f.scratch, tid);
            for (int q = re - 1; q >= rs; --q) {
                const double dsn = s.X[q];
                const double c = (q + 1 < NS && !(dsn < FCPP_ZERO_LEN)) ? two_a * dsn : INFINITY;
                carry = fmin(s.U[q], carry + c);
                s.U[q] = carry;
            }
        }
        __syncthreads();
    }

    // ------------------------------------------------------------------------------------
    // phase 5a: final speeds (km/h) of the staged points -> U[q] and HBM; lateral-acceleration validation
    // (mlp3:1383-1410)
    // ------------------------------------------------------------------------------------
    int n_aviol = 0;
    double mx[3] = {0.0, 0.0, 0.0};  // max kappa, max a_lat, max |kappa jump|
    auto finish_point = [&](bool act, int q, double u_lim, double vl) {
        const double kap = act ? s.Y[q] : 0.0;
        const double u = act ? s.U[q] : 0.0;
        const double v = do_scan ? final_speed(act, u, u_lim, vl) : vl;
        if (!act) return;
        const int i = q < 2 ? q : q + n_skip;
        if (gs) gs[i] = v;
        if (gk) gk[i] = kap;
        if (i >= 1 && i + 1 < N) {
            const double vm = div36(v);
            const double alat = vm * vm * kap;  // mlp3:1389-1390
            n_aviol += (alat > veh.max_lateral_accel);
            mx[0] = fmax(mx[0], kap);
            mx[1] = fmax(mx[1], alat);
            // the successor in the staged order is the successor in the plan except after point 1, where both
            // curvatures are 0 (a zero-length segment on either side)
            if (i + 2 < N) mx[2] = fmax(mx[2], fabs(s.Y[q + 1] - kap));
        }
        s.U[q] = v;  // safe: U[q] is read only by its owner in this phase
    };
    for (int base = 0; base < NS; base += T) {  // warp-uniform trip count (final_speed votes)
        const int q = base + tid;
        const int tag = (q < NS) ? s.TAG[q] : TAG_GENERIC;
        const bool act = tag < TAG_GENERIC;
        double u_lim = 0.0, vl = 0.0;
        if (act) {
            u_lim = f.tbl[tag].u;
            vl = f.tbl[tag].vl;
        }
        finish_point(act, q, u_lim, vl);
    }
    for (int base = 0; base < n_gslots; base += T) {
        const int g = base + tid;
        const int i = (g < n_gslots) ? f.glist[g] : -1;
        const bool act = i >= 0;
        double vl = 0.0, u_lim = 0.0;
        if (act) {
            vl = f.gvl[g];
            const double vms = div36(vl);
            u_lim = vms * vms;
        }
        finish_point(act, act ? (i < 2 ? i : i - n_skip) : 0, u_lim, vl);
    }
    __syncthreads();
    // ------------------------------------------------------------------------------------
    // phase 5b: work time with the adjusted speeds (mlp3:423-431, :1298-1311)
    // ------------------------------------------------------------------------------------
    double acc_t_m = 0.0, acc_t_h = 0.0;
    for (int q = tid; q + 1 < NS; q += T) {
        const int i = q < 2 ? q : q + n_skip;
        if (i == n_main - 1) continue;
        // (after point 1 the staged successor is not the plan's, but that segment has zero length: t = 0)
        const double t = div_pos(s.X[q], fmax(div36((s.U[q] + s.U[q + 1]) / 2), FCPP_MIN_SPEED_MS));
        if (i < n_main)
            acc_t_m += t;
        else
            acc_t_h += t;
    }
    double sums[9] = {acc_len_m, acc_len_h, acc_tpre_m, acc_tpre_h, acc_t_m,
                      acc_t_h,   (double)n_aviol, (double)n_bviol, (double)n_oviol};
    block_reduce<9, false, T / 32>(sums, f.scratch, tid);
    block_reduce<3, true, T / 32>(mx, f.scratch, tid);
    if (tid == 0 && sum) {
        // the regular chains: one chain's sums times their number
        const double nreg = (double)(n_skip / CHAIN_POINTS);
        const bool reg = n_skip > 0 && !omega;  // (the Ω pattern's chains went into the sums one by one)
        if (omega && n_skip > 0) {
            for (int w = 0; w < T / 32; ++w) {
                const double *part = f.omega_part + 8 * w;
                sums[0] += part[0], sums[2] += part[1], sums[4] += part[2], sums[6] += part[3];
                mx[0] = fmax(mx[0], part[4]), mx[1] = fmax(mx[1], part[5]), mx[2] = fmax(mx[2], part[6]);
            }
        }
        sum->status = 0;
        sum->len_main = sums[0] + (reg ? nreg * f.chain_sum[0] : 0.0);
        sum->len_head = sums[1];
        sum->time_main_pre = sums[2] + (reg ? nreg * f.chain_sum[1] : 0.0);
        sum->time_head_pre = sums[3];
        sum->time_main = sums[4] + (reg ? nreg * f.chain_sum[2] : 0.0);
        sum->time_head = sums[5];
        sum->n_accel_viol = (int)(sums[6] + (reg ? nreg * f.chain_sum[3] : 0.0));
        sum->n_boundary_viol = (int)sums[7];
        sum->n_obstacle_viol = (int)sums[8];
        sum->max_curvature = reg ? fmax(mx[0], f.chain_sum[4]) : mx[0];
        sum->max_lateral_accel = reg ? fmax(mx[1], f.chain_sum[5]) : mx[1];
        sum->max_jump = reg ? fmax(mx[2], f.chain_sum[6]) : mx[2];
        sum->reserved = 0.0;
        if (!a.b.do_coverage) {
            sum->cov_cells = sum->cov_total = 0;
            for (int k = 0; k < 4; ++k) sum->corner_before[k] = sum->corner_after[k] = 0;
        }
    }
}

__global__ void __launch_bounds__(TG, FCPP_PLAN_GEN_MIN_CTAS) plan_gen_omega_kernel(const PlanArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    plan_gen_body<true>(a, smem_raw, threadIdx.x, blockIdx.x);
}

__global__ void __launch_bounds__(TG, FCPP_PLAN_GEN_MIN_CTAS) plan_gen_kernel(const PlanArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    plan_gen_body(a, smem_raw, threadIdx.x, blockIdx.x);
}

// One caller-supplied path (A7 / A8 / A13 of the drop-in API): every point from its coordinates.
template <bool BIG, int T>
__device__ __forceinline__ void plan_body_path(const PathArgs &a, const Smem &s, const int64_t cand, const int cap)
{
    const int tid = threadIdx.x;
    const fcpp_vehicle &veh = a.veh;
    fcpp_summary *sum = a.summary ? a.summary + cand : nullptr;
    const int64_t off = a.in_offsets[cand];
    const int N = (int)(a.in_offsets[cand + 1] - off);
    const int n_main = N;
    if (N > cap && !BIG && a.big_enabled) return;
    if (N > cap || N == 0) {
        if (sum && tid == 0) {
            sum->status = N ? FCPP_CAND_TOO_LARGE : 0;
            sum->n_main = N;
            sum->n_head = 0;
            sum->n_accel_viol = 0;
            sum->len_main = sum->time_main = sum->time_main_pre = 0.0;
            sum->max_curvature = sum->max_lateral_accel = sum->max_jump = 0.0;
        }
        return;
    }
    {
        const double2 *gp = reinterpret_cast<const double2 *>(a.in_path) + off;
        for (int i = tid; i < N; i += T) {
            const double2 p = gp[i];
            s.X[i] = p.x;
            s.Y[i] = p.y;
        }
    }
    __syncthreads();

    // per-thread contiguous chunk: ds_i -> X[i], kappa_i -> Y[i], U_i = (vlim/3.6)^2
    const int chunk = (N + T - 1) / T;
    const int cs = min(N, tid * chunk);
    const int ce = min(N, cs + chunk);
    double hpx = 0.0, hpy = 0.0, hnx = 0.0, hny = 0.0;
    if (cs < ce) {
        if (cs > 0) {
            hpx = s.X[cs - 1];
            hpy = s.Y[cs - 1];
        }
        if (ce < N) {
            hnx = s.X[ce];
            hny = s.Y[ce];
        }
    }
    __syncthreads();
    double acc_len_m = 0.0, acc_tpre_m = 0.0;
    if (cs < ce) {
        double px = hpx, py = hpy;
        double cx = s.X[cs], cy = s.Y[cs];
        double dx1 = cx - px, dy1 = cy - py;
        double ds1 = (cs > 0) ? sqrt_z(dx1 * dx1 + dy1 * dy1) : 0.0;
        for (int i = cs; i < ce; ++i) {
            double nx, ny;
            if (i + 1 < ce) {
                nx = s.X[i + 1];
                ny = s.Y[i + 1];
            } else {
                nx = hnx;
                ny = hny;
            }
            double dx2 = 0.0, dy2 = 0.0, ds2 = 0.0;
            if (i + 1 < N) {
                dx2 = nx - cx;
                dy2 = ny - cy;
                ds2 = sqrt_z(dx2 * dx2 + dy2 * dy2);
            }
            double kap = 0.0;
            if (i >= 1 && i + 1 < N) kap = curvature3(dx1, dy1, ds1, dx2, dy2, ds2);
            const double v0 = a.in_speeds[off + i];
            const double v1 = (i + 1 < N) ? a.in_speeds[off + i + 1] : 0.0;
            const double vl = a.do_speed_plan ? vlimit(v0, kap, veh) : v0;
            const double vms = div36(vl);
            s.X[i] = ds2;
            s.Y[i] = kap;
            s.U[i] = vms * vms;
            if (i + 1 < N) {  // length and pre-adjustment time (mlp3:1290-1311)
                acc_len_m += ds2;
                acc_tpre_m += div_z(ds2, fmax(div36((v0 + v1) / 2), FCPP_MIN_SPEED_MS));
            }
            dx1 = dx2;
            dy1 = dy2;
            ds1 = ds2;
            cx = nx;
            cy = ny;
        }
    }
    __syncthreads();

    const bool do_scan = a.do_speed_plan && N >= 3;
    const double two_a = 2 * veh.max_longitudinal_accel;
    if (do_scan) {
        {
            MP agg;
            agg.C = 0.0;
            agg.M = INFINITY;
            for (int i = cs; i < ce; ++i) {
                const double dsp = (i > 0) ? s.X[i - 1] : 0.0;
                const double c = (i > 0 && !(dsp < FCPP_ZERO_LEN)) ? two_a * dsp : INFINITY;
                agg.M = fmin(s.U[i], agg.M + c);
                agg.C = agg.C + c;
            }
            double carry = mp_block_exclusive(agg, s.scratch, tid);
            for (int i = cs; i < ce; ++i) {
                const double dsp = (i > 0) ? s.X[i - 1] : 0.0;
                const double c = (i > 0 && !(dsp < FCPP_ZERO_LEN)) ? two_a * dsp : INFINITY;
                carry = fmin(s.U[i], carry + c);
                s.U[i] = carry;
            }
        }
        __syncthreads();
        {
            const int rt = T - 1 - tid;
            const int rs = min(N, rt * chunk);
            const int re = min(N, rs + chunk);
            MP agg;
            agg.C = 0.0;
            agg.M = INFINITY;
            for (int i = re - 1; i >= rs; --i) {
                const double dsn = s.X[i];
                const double c = (i + 1 < N && !(dsn < FCPP_ZERO_LEN)) ? two_a * dsn : INFINITY;
                agg.M = fmin(s.U[i], agg.M + c);
                agg.C = agg.C + c;
            }
            double carry = mp_block_exclusive(agg, s.scratch, tid);
            for (int i = re - 1; i >= rs; --i) {
                const double dsn = s.X[i];
                const double c = (i + 1 < N && !(dsn < FCPP_ZERO_LEN)) ? two_a * dsn : INFINITY;
                carry = fmin(s.U[i], carry + c);
                s.U[i] = carry;
            }
        }
        __syncthreads();
    }

    int n_aviol = 0;
    double mx[3] = {0.0, 0.0, 0.0};
    {
        double *gs = a.speeds_kmh ? a.speeds_kmh + off : nullptr;
        double *gk = a.curvature ? a.curvature + off : nullptr;
        for (int i = tid; i < N; i += T) {
            const double kap = s.Y[i];
            const double v0 = a.in_speeds[off + i];
            double v;
            if (do_scan) {
                const double vl = vlimit(v0, kap, veh);
                const double vms = div36(vl);
                const double u = s.U[i];
                v = (u == vms * vms) ? vl : 3.6 * sqrt(u);
            } else {
                v = v0;
            }
            if (gs) gs[i] = v;
            if (gk) gk[i] = kap;
            if (i >= 1 && i + 1 < N) {
                const double vm = div36(v);
                const double alat = vm * vm * kap;  // mlp3:1389-1390
                n_aviol += (alat > veh.max_lateral_accel);
                mx[0] = fmax(mx[0], kap);
                mx[1] = fmax(mx[1], alat);
                if (i + 2 < N) mx[2] = fmax(mx[2], fabs(s.Y[i + 1] - kap));
            }
            s.U[i] = v;
        }
    }
    __syncthreads();
    double acc_t_m = 0.0;
    for (int i = tid; i + 1 < N; i += T)
        acc_t_m += div_z(s.X[i], fmax(div36((s.U[i] + s.U[i + 1]) / 2), FCPP_MIN_SPEED_MS));
    double sums[4] = {acc_len_m, acc_tpre_m, acc_t_m, (double)n_aviol};
    block_reduce<4, false, T / 32>(sums, s.scratch, tid);
    block_reduce<3, true, T / 32>(mx, s.scratch, tid);
    if (tid == 0 && sum) {
        sum->status = 0;
        sum->n_passes = 0;
        sum->n_loops = 0;
        sum->n_main = n_main;
        sum->n_head = 0;
        sum->len_main = sums[0];
        sum->len_head = 0.0;
        sum->time_main_pre = sums[1];
        sum->time_head_pre = 0.0;
        sum->time_main = sums[2];
        sum->time_head = 0.0;
        sum->n_accel_viol = (int)sums[3];
        sum->n_boundary_viol = 0;
        sum->n_obstacle_viol = 0;
        sum->max_curvature = mx[0];
        sum->max_lateral_accel = mx[1];
        sum->max_jump = mx[2];
        sum->reserved = 0.0;
        sum->cov_cells = sum->cov_total = 0;
        for (int k = 0; k < 4; ++k) sum->corner_before[k] = sum->corner_after[k] = 0;
    }
}

#ifndef FCPP_PLAN_MIN_CTAS
#define FCPP_PLAN_MIN_CTAS 4
#endif
// Caller-supplied paths.  T threads per CTA: T0 (256) when four or more CTAs fit an SM, 2*T0 / 4*T0 when the
// staging of long paths leaves room for only two / one: the SM keeps ~32 resident warps either way
template <int T>
__global__ void __launch_bounds__(T, (T0 * FCPP_PLAN_MIN_CTAS) / T) path_kernel(const PathArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    if (a.nmin >= 0 || a.defer) {  // tiered launch: is this path in this tier's length range?
        const int n = (int)(a.in_offsets[blockIdx.x + 1] - a.in_offsets[blockIdx.x]);
        if (n <= a.nmin || (a.defer && n > a.ncap)) return;
    }
    const Smem s = carve(smem_raw, a.ncap);
    plan_body_path<false, T>(a, s, blockIdx.x, a.ncap);
}

// Paths that do not fit the shared-memory staging (N > ~9000 points): a few persistent CTAs walk the batch and
// run the same body with x/y/u staged in a per-CTA slice of library-owned HBM (L2-resident in practice).
__global__ void __launch_bounds__(T0, 3) path_big_kernel(const PathArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem s = carve(smem_raw, 0);
    unsigned char *slice = a.big_scratch + (int64_t)blockIdx.x * a.big_stride;
    const size_t arr = align16(sizeof(double) * (size_t)a.big_ncap);
    s.X = (double *)slice;
    s.Y = (double *)(slice + arr);
    s.U = (double *)(slice + 2 * arr);
    for (int64_t c = blockIdx.x; c < a.n_items; c += gridDim.x) {
        const int n = (int)(a.in_offsets[c + 1] - a.in_offsets[c]);
        if (n <= a.ncap) continue;  // handled by path_kernel
        plan_body_path<true, T0>(a, s, c, a.big_ncap);
        __syncthreads();
    }
}

template <int T>
cudaError_t launch_variant(const PathArgs &a, int64_t n, size_t bytes, cudaStream_t st)
{
    cudaError_t e = cudaFuncSetAttribute(path_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return e;
    path_kernel<T><<<(unsigned)n, T, bytes, st>>>(a);
    return cudaGetLastError();
}
// largest point capacity whose staging lets `ctas` CTAs share one SM (1 KB reserved per CTA)
int capacity_for_ctas(fcpp_handle *h, int ctas)
{
    size_t budget = (size_t)h->max_smem_sm / ctas - 1024;
    if (budget > (size_t)h->max_smem_optin) budget = (size_t)h->max_smem_optin;
    const size_t fixed = plan_smem_bytes(0);
    if (budget <= fixed) return 0;
    return (int)((budget - fixed) / 24) / 64 * 64;
}

// One launch when the longest path of the batch leaves room for four CTAs per SM.  A batch of mixed lengths is cut
// into up to three TIERS by length — N <= cap4 at T0 threads and four CTAs per SM, cap4 < N <= cap2 at 2*T0 and
// two, longer at 4*T0 and one — so that short paths do not inherit the occupancy of the longest.  Every tier
// launches one CTA per path; CTAs outside the tier's range exit on one read.
cudaError_t launch_tiers(fcpp_handle *h, PathArgs &a, int64_t n, int want, int cap_max, bool big, cudaStream_t st)
{
    const int cap4 = capacity_for_ctas(h, 4);
    const int cap2 = capacity_for_ctas(h, 2);
    const int last = (want > 0 && want < cap_max) ? want : cap_max;
    int caps[3], nt = 0;
    if (last > cap4 && cap4 >= 256) caps[nt++] = cap4;
    if (last > cap2 && cap2 > cap4) caps[nt++] = cap2;
    caps[nt++] = last;
    int prev = -1;
    for (int t = 0; t < nt; ++t) {
        a.ncap = caps[t];
        a.nmin = prev;
        a.defer = (t + 1 < nt) ? 1 : 0;
        a.big_enabled = (t + 1 == nt && big) ? 1 : 0;
        const size_t bytes = plan_smem_bytes(a.ncap);
        if (bytes > (size_t)h->max_smem_optin) return cudaErrorInvalidValue;
        const int fit = (int)((size_t)h->max_smem_sm / (bytes + 1024));
        h->launches++;
        cudaError_t e = fit >= 4   ? launch_variant<T0>(a, n, bytes, st)
                        : fit >= 2 ? launch_variant<2 * T0>(a, n, bytes, st)
                                   : launch_variant<4 * T0>(a, n, bytes, st);
        if (e != cudaSuccess) return e;
        prev = caps[t];
    }
    return cudaSuccess;
}

// launch path_big_kernel when the longest path exceeds the shared-memory capacity.  The HBM staging (h->d_big) is
// owned and resized here only.
cudaError_t launch_big(fcpp_handle *h, PathArgs &a, int64_t n_items, int max_points, cudaStream_t st)
{
    const int big_ncap = (max_points + 255) / 256 * 256;
    const int64_t stride = (int64_t)(3 * align16(sizeof(double) * (size_t)big_ncap));
    int64_t ctas = n_items < 2 * h->sm_count ? n_items : 2 * h->sm_count;
    while (ctas > 1 && ctas * stride > ((int64_t)8 << 30)) ctas /= 2;  // at most 8 GiB of scratch
    if (ctas * stride > h->big_cap) {
        if (h->d_big) cudaFree(h->d_big);
        h->d_big = nullptr;
        h->big_cap = 0;
        cudaError_t e = cudaMalloc(&h->d_big, (size_t)(ctas * stride));
        if (e != cudaSuccess) return e;
        h->big_cap = ctas * stride;
    }
    a.big_ncap = big_ncap;
    a.big_scratch = (unsigned char *)h->d_big;
    a.big_stride = stride;
    a.n_items = n_items;
    path_big_kernel<<<(unsigned)ctas, T0, plan_smem_bytes(0), st>>>(a);
    h->launches++;
    return cudaGetLastError();
}

}  // namespace

// Generated plans: one CTA per candidate.  Only the first 2 + last 22 main points and the headland are staged in
// shared memory (~25 B per point), so the staging depends on the longest HEADLAND of the batch, not on the plan
// length: no length tiers, no HBM staging, 7-8 CTAs of 128 threads per SM at every field size.
cudaError_t fcpp_launch_plan(fcpp_handle *h, const fcpp_batch &b, const fcpp_outputs &o, cudaStream_t st)
{
    if (b.n_cand == 0) return cudaSuccess;
    PlanArgs a{};
    a.b = b;
    a.recs = h->d_rec;
    a.trig = h->d_trig;
    a.out = o;
    a.obs_cap_verts = b.obs_poly_start ? b.max_obs_verts : 0;
    a.obs_cap_polys = b.obs_poly_start ? b.max_obs_polys : 0;
    a.ncap = (MAIN_STAGED + (h->cover_pcap > 0 ? h->cover_pcap : 0) + 63) / 64 * 64;
    const size_t bytes = gen_smem_bytes(a.ncap, a.obs_cap_verts, a.obs_cap_polys);
    if (bytes > (size_t)h->max_smem_optin) return cudaErrorInvalidValue;  // obstacle tables / headland beyond shared memory
    const bool omega = b.turn_model == FCPP_TURN_OMEGA;  // its own instance: the default patterns do not carry its code
    cudaError_t e = cudaFuncSetAttribute(omega ? plan_gen_omega_kernel : plan_gen_kernel,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return e;
    if (omega)
        plan_gen_omega_kernel<<<(unsigned)b.n_cand, TG, bytes, st>>>(a);
    else
        plan_gen_kernel<<<(unsigned)b.n_cand, TG, bytes, st>>>(a);
    h->launches++;
    return cudaGetLastError();
}

cudaError_t fcpp_launch_speed_verify(fcpp_handle *h, const fcpp_vehicle &veh, const double *d_path,
                                     const double *d_speeds_in, const int64_t *d_offsets, int64_t n_paths,
                                     int64_t max_len, int do_speed_plan, double *d_speeds_out, double *d_curv,
                                     fcpp_summary *d_summary, cudaStream_t st)
{
    if (n_paths == 0) return cudaSuccess;
    PathArgs a{};
    a.veh = veh;
    a.in_path = d_path;
    a.in_speeds = d_speeds_in;
    a.in_offsets = d_offsets;
    a.do_speed_plan = do_speed_plan;
    a.summary = d_summary;
    a.speeds_kmh = d_speeds_out;
    a.curvature = d_curv;
    const int cap_max = capacity_for_ctas(h, 1);
    const int want = max_len > 0 ? (int)((max_len + 255) / 256 * 256) : 0;
    a.ncap = (want > 0 && want < cap_max) ? want : cap_max;
    const bool big = want > a.ncap;
    a.big_enabled = big ? 1 : 0;
    a.n_items = n_paths;
    cudaError_t e = launch_tiers(h, a, n_paths, want > 0 ? want : a.ncap, a.ncap, big, st);
    if (e == cudaSuccess && big) e = launch_big(h, a, n_paths, want, st);
    return e;
}
