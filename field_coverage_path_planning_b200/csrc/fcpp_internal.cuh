// fcpp_internal.cuh — shared device-side definitions of libfcpp (sm_100a only).
//
// Numerics contract (DESIGN.md §4): every expression that feeds an INTEGER output (point
// counts, violation counts, coverage cells) is evaluated in FP64 in the operation order of the
// reference's numpy code with FMA contraction disabled (this library is compiled with
// -fmad=false); sin/cos never run on the device for geometry — the arc tables and the heading
// rotation come from the host — so generated path points are bit-identical to numpy's.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/fcpp.h"

#define FCPP_PLAN_THREADS 256
#ifndef FCPP_COVER_THREADS
#define FCPP_COVER_THREADS 512
#endif
#ifndef FCPP_COVER_RECT
#define FCPP_COVER_RECT 1  // vertical chains as rectangles + end discs (fcpp_cover.cu: setup_entries)
#endif

// speed classes of a path point (initial speeds, SURVEY.md App. A Q5)
enum : uint8_t { CLS_WORK = 0, CLS_TURN = 1, CLS_HEAD = 2, CLS_REVERSE = 3 };

// reference constants (SURVEY.md §5)
#define FCPP_ZERO_LEN 1e-6        // mlp3:526, :560, :576
#define FCPP_KAPPA_EPS 1e-6       // mlp3:496
#define FCPP_GEOFENCE_EPS 1e-9    // D3
#define FCPP_MIN_SPEED_MS 0.1     // mlp3:1308
#define FCPP_REV_SPACING 0.5      // mlp3:1214
#define FCPP_REV_MIN_PTS 10       // mlp3:1214
#define FCPP_REV_CAP 3.0          // mlp3:1279
#define FCPP_CORNER_GRID_H 0.1    // mlp3:1452

struct TrigTables {
    double cos20[FCPP_UTURN_POINTS], sin20[FCPP_UTURN_POINTS];
    double cos15[FCPP_CORNER_POINTS], sin15[FCPP_CORNER_POINTS];
};

// Per-candidate geometry record written by the layout kernel (A2-A6 scalar part) and consumed
// by the plan and coverage kernels through one bulk (TMA) copy.  Size is a multiple of 16 B.
struct __align__(16) CandRec {
    int32_t status, P, K, n_main;
    int32_t n_head, n_total, flags, field;
    int32_t n_rev[3], corner_g;
    int32_t vn_rev[4];
    double R;
    double min_x, min_y, max_x, max_y;  // swath-frame bounds of the work area (mlp3:731-732)
    double cx, cy;                      // rotation centre (work-area centroid, mlp3:690, :710)
    double cos_a, sin_a;                // rotate-back (mlp3:709-714)
    uint64_t cover_key[2];              // hashes of the fields A10 (corner windows) / A11 (band) read (de-duplication)
    int32_t band_group;                 // 1: every headland straight is axis-aligned on the 1e-4 m lattice (de-duplicated
                                        // batches only): the bands of all four start corners are evaluated together
                                        // (fcpp_cover.cu: band_grouped)
    int32_t pad1;
    double main_quad[4][2];             // R-inset of the field (mlp3:594-595), D1
    double rev[3][5];                   // loop-0 reverse fills: ex, ey, dx, dy, length (mlp3:1154-1218)
    double vrev[4][5];                  // verification corners (mlp3:1531-1554)
    double corners[FCPP_MAX_LOOPS][4][2];  // inset rings of the K headland loops (mlp3:964-972)
};
static_assert(sizeof(CandRec) % 16 == 0, "CandRec must be bulk-copyable");

struct fcpp_handle {
    int device;
    TrigTables *d_trig;
    CandRec *d_rec;
    int64_t rec_cap;
    void *d_scan_tmp;
    void *d_big;             // HBM staging of caller-supplied paths that do not fit shared memory
    int64_t big_cap;
    int64_t scan_tmp_cap;
    int64_t launches;
    int *d_maxn;             // device: [max n_total, max n_head] of the last layout pass
    int *h_maxn;             // pinned host mirror
    int max_smem_optin;
    int max_smem_sm;         // shared memory per SM
    int sm_count;
    bool layout_valid;
    bool rec_valid;          // the candidate records belong to the batch of layout_id (kept after fcpp_plan_batch)
    bool profiling;
    cudaEvent_t ev[4];       // layout start, plan start, cover start, end
    int last_maxn;
    int last_maxhead;
    int64_t last_total;      // total points of the last synchronous layout pass with offsets (-1: unknown)
    int cover_pcap;          // point capacity of the coverage kernel's staging for the next launch
    int cover_mode;          // diagnostics (fcpp_set_cover_mode): bit 0 = never use the zoned band evaluation,
                             // bit 1 = no coverage de-duplication, bits 6 / 7 = de-duplicated batches: force one
                             // coverage CTA per listed task / the persistent grid over the task list
    void *d_dedupe;          // coverage de-duplication: hash table, hashes, representatives
    size_t dedupe_bytes;
    uint32_t dedupe_cap;     // slots of the (currently zeroed) table inside d_dedupe; 0 = not initialised
    int64_t layout_ncand;
    const void *layout_id[4]; // identity of the batch the valid layout belongs to: cand_R, cand_flags, field_verts, stream
    void *d_ga;              // GA workspace (two populations, lengths, fitness, ranks, state, best route)
    size_t ga_bytes;
    void *h_ga_state;        // pinned host copy of the GA state
    cudaStream_t ga_stream;  // capture stream of the generation graph
    void *d_sel;             // top-k selection workspace (fcpp_select.cu): field counts, keys sorted by field, unit lists
    size_t sel_bytes;
    void *d_pcov;            // path coverage (fcpp_cover.cu): per-path first slab [n + 1], the slab counter
    size_t pcov_bytes;
    char err[512];
};

__device__ __forceinline__ uint64_t mix64(uint64_t h, uint64_t w)
{
    h = (h ^ w) * 0x9E3779B97F4A7C15ull;
    return h ^ (h >> 29);
}
__device__ __forceinline__ uint64_t dbits(double x) { return (uint64_t)__double_as_longlong(x); }

constexpr int COVER_FLAG_MASK = FCPP_FLAG_CORNER_MASK | FCPP_FLAG_GAP_GATE;

// hashes of the CandRec fields the coverage kernel reads (fcpp_cover.cu: coverage de-duplication).
// part 0 = A10, the four corner windows: field, R, window size, verification reverse fills — NOT the
// start corner; part 1 = A11, the headland band: field, R, loops, rings, reverse fills and the start corner,
// except for records with band_group set: their four start corners share one key and one CTA evaluates the
// bands of all of them.  Their reverse fills are left out: the fill at a corner is a function of the field,
// R, the gap gate and the first ring (reverse_fill), all of which are in the key
__device__ __forceinline__ bool cover_dead(const CandRec &r) { return r.status != 0 || r.n_total == 0; }
__device__ __forceinline__ uint64_t cover_key(const CandRec &r, int part)
{
    uint64_t h = part ? 0x243F6A8885A308D3ull : 0x13198A2E03707344ull;
    const bool dead = cover_dead(r);
    h = mix64(h, ((uint64_t)(uint32_t)r.status << 32) | (uint32_t)r.field);
    h = mix64(h, dead ? 1u : 0u);
    if (dead) return h | 1ull;  // all dead candidates of a field share zero counts
    h = mix64(h, dbits(r.R));
    if (part == 0) {
        h = mix64(h, (uint32_t)r.corner_g);
        for (int k = 0; k < 4; ++k) h = mix64(h, (uint32_t)r.vn_rev[k]);
        for (int k = 0; k < 20; ++k) h = mix64(h, dbits((&r.vrev[0][0])[k]));
    } else if (r.band_group) {
        h = mix64(h, ((uint64_t)(uint32_t)r.K << 32) | 0x80000000u);
        h = mix64(h, (uint32_t)(r.flags & FCPP_FLAG_GAP_GATE));
        for (int k = 0; k < 8; ++k) h = mix64(h, dbits((&r.main_quad[0][0])[k]));
        for (int k = 0; k < 8 * r.K; ++k) h = mix64(h, dbits((&r.corners[0][0][0])[k]));
    } else {
        h = mix64(h, ((uint64_t)(uint32_t)r.K << 32) | (uint32_t)r.n_head);
        h = mix64(h, (uint32_t)(r.flags & COVER_FLAG_MASK));
        for (int k = 0; k < 3; ++k) h = mix64(h, (uint32_t)r.n_rev[k]);
        for (int k = 0; k < 8; ++k) h = mix64(h, dbits((&r.main_quad[0][0])[k]));
        for (int k = 0; k < 15; ++k) h = mix64(h, dbits((&r.rev[0][0])[k]));
        for (int k = 0; k < 8 * r.K; ++k) h = mix64(h, dbits((&r.corners[0][0][0])[k]));
    }
    return h | 1ull;  // 0 marks an empty slot
}
__device__ __forceinline__ bool cover_same(const CandRec &a, const CandRec &b, int part)
{
    const bool da = cover_dead(a), db = cover_dead(b);
    if (a.status != b.status || a.field != b.field || da != db) return false;
    if (da) return true;
    bool same = dbits(a.R) == dbits(b.R);
    if (part == 0) {
        same = same && a.corner_g == b.corner_g;
        for (int k = 0; k < 4; ++k) same = same && a.vn_rev[k] == b.vn_rev[k];
        for (int k = 0; k < 20; ++k) same = same && dbits((&a.vrev[0][0])[k]) == dbits((&b.vrev[0][0])[k]);
        return same;
    }
    same = same && a.K == b.K && a.band_group == b.band_group;
    if (a.band_group) {
        same = same && (a.flags & FCPP_FLAG_GAP_GATE) == (b.flags & FCPP_FLAG_GAP_GATE);
    } else {
        same = same && a.n_head == b.n_head && (a.flags & COVER_FLAG_MASK) == (b.flags & COVER_FLAG_MASK);
        for (int k = 0; k < 3; ++k) same = same && a.n_rev[k] == b.n_rev[k];
        for (int k = 0; k < 15; ++k) same = same && dbits((&a.rev[0][0])[k]) == dbits((&b.rev[0][0])[k]);
    }
    for (int k = 0; k < 8; ++k) same = same && dbits((&a.main_quad[0][0])[k]) == dbits((&b.main_quad[0][0])[k]);
    for (int k = 0; same && k < 8 * a.K; ++k)
        same = dbits((&a.corners[0][0][0])[k]) == dbits((&b.corners[0][0][0])[k]);
    return same;
}

// ---------------------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------------------
// Bounds-checked debug build (make VARIANT=bounds DEFS=-DFCPP_BOUNDS_DEBUG): device asserts at the shared-memory
// indexers of the hot kernels.  compute-sanitizer is closed on the GPU pool, so the parity tests are run once per
// round through this build instead (a failed assert traps the kernel and surfaces as a CUDA error in the test).
#ifdef FCPP_BOUNDS_DEBUG
#include <assert.h>
#define FCPP_ASSERT(c) assert(c)
__device__ __forceinline__ uint32_t fcpp_dynamic_smem_bytes()
{
    uint32_t n;
    asm("mov.u32 %0, %%dynamic_smem_size;" : "=r"(n));
    return n;
}
#else
#define FCPP_ASSERT(c) ((void)0)
#endif

// doubles as unsigned keys with the same order (per-field argmin and top-k selection)
__device__ __forceinline__ unsigned long long order_bits(double x)
{
    const unsigned long long b = (unsigned long long)__double_as_longlong(x);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double unorder_bits(unsigned long long o)
{
    const unsigned long long b = (o >> 63) ? (o & 0x7fffffffffffffffull) : ~o;
    return __longlong_as_double((long long)b);
}

__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}

// TMA 1-D bulk copy global -> shared, completion on an mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t phase)
{
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(phase)
        : "memory");
    return ok != 0;
}

// Block-wide wait for a TMA completion: ONE thread polls the mbarrier (256 spinning threads cost
// 14 % of the plan kernel's instructions), the block barrier releases the rest, and every thread
// then observes the completed phase itself (acquire of the async-proxy writes).
__device__ __forceinline__ void mbar_wait_block(uint64_t *bar, uint32_t phase)
{
    if (threadIdx.x == 0)
        while (!mbar_try_wait(bar, phase)) {
        }
    __syncthreads();
    while (!mbar_try_wait(bar, phase)) {
    }
}

// D1: mitred inset of a convex CCW quad (oracle/geom.py inset_convex — same operation order).
__device__ inline bool inset4(const double (*v)[2], double d, double (*out)[2])
{
    double nx[4], ny[4], c[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int k1 = (k + 1) & 3;
        const double ex = v[k1][0] - v[k][0];
        const double ey = v[k1][1] - v[k][1];
        const double ln = sqrt(ex * ex + ey * ey);
        nx[k] = -ey / ln;
        ny[k] = ex / ln;
        c[k] = (nx[k] * v[k][0] + ny[k] * v[k][1]) + d;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int a = (i + 3) & 3, b = i;
        const double det = nx[a] * ny[b] - ny[a] * nx[b];
        out[i][0] = (c[a] * ny[b] - c[b] * ny[a]) / det;
        out[i][1] = (nx[a] * c[b] - nx[b] * c[a]) / det;
    }
    bool ok = true;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int k1 = (k + 1) & 3;
        const double ex = v[k1][0] - v[k][0], ey = v[k1][1] - v[k][1];
        const double fx = out[k1][0] - out[k][0], fy = out[k1][1] - out[k][1];
        ok = ok && (ex * fx + ey * fy > 0.0);
    }
    return ok;
}

__device__ inline double signed_area4(const double (*v)[2])
{
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int j = (i + 1) & 3;
        s += v[i][0] * v[j][1] - v[j][0] * v[i][1];
    }
    return 0.5 * s;
}

// oracle/geom.py centroid (shifted to vertex 0)
__device__ inline void centroid4(const double (*v)[2], double &cx, double &cy)
{
    const double ox = v[0][0], oy = v[0][1];
    double a2 = 0.0, sx = 0.0, sy = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int j = (i + 1) & 3;
        const double x0 = v[i][0] - ox, y0 = v[i][1] - oy;
        const double x1 = v[j][0] - ox, y1 = v[j][1] - oy;
        const double cr = x0 * y1 - x1 * y0;
        a2 += cr;
        sx += (x0 + x1) * cr;
        sy += (y0 + y1) * cr;
    }
    cx = ox + sx / (3.0 * a2);
    cy = oy + sy / (3.0 * a2);
}

// D3 geofence and obstacle (D2/D3) tests of one point, shared by the plan kernel and the path coverage kernels:
// bit 0 = outside the field by more than 1e-9 m (geo [4][5]: edge start ax, ay, edge ex, ey, -1e-9 |e|), bit 1 = inside
// an obstacle polygon or closer than r to one of its edges (obs_bb [n][4]: the polygons' boxes grown by r + 1e-6;
// obs_vs [n + 1]: their vertex ranges in obs_xy).  The tables are handed over as four __restrict__ pointers instead
// of through the plan kernel's shared-memory struct: measured 2-5 % on the plan kernel (a non-inlined single copy,
// tried against the instruction-fetch stalls, cost 15-30 %).
__device__ __forceinline__ int point_tests_impl(const double *__restrict__ geo, const double *__restrict__ obs_xy,
                                                const double *__restrict__ obs_bb, const int32_t *__restrict__ obs_vs,
                                                int n_obs_poly, double r2, double x, double y)
{
    bool outb = false;
#pragma unroll
    for (int k = 0; k < 4; ++k)
        outb = outb || (geo[5 * k + 2] * (y - geo[5 * k + 1]) - geo[5 * k + 3] * (x - geo[5 * k]) < geo[5 * k + 4]);
    bool hit = false;
    for (int p = 0; p < n_obs_poly && !hit; ++p) {
        if (x < obs_bb[4 * p] || y < obs_bb[4 * p + 1] || x > obs_bb[4 * p + 2] || y > obs_bb[4 * p + 3]) continue;
        const int vs = obs_vs[p], ve = obs_vs[p + 1];
        bool inside = false;
        for (int q = vs; q < ve; ++q) {
            const int q1 = (q + 1 < ve) ? q + 1 : vs;
            const double ax = obs_xy[2 * q], ay = obs_xy[2 * q + 1];
            const double bx = obs_xy[2 * q1], by = obs_xy[2 * q1 + 1];
            // even-odd crossing (oracle/geom.py point_in_polygon_crossing)
            if ((ay > y) != (by > y)) {
                const double xi = ax + (y - ay) * (bx - ax) / (by - ay);
                if (x < xi) inside = !inside;
            }
            // D2 distance test (oracle/geom.py dist2_point_segment)
            const double dx = bx - ax, dy = by - ay, wx = x - ax, wy = y - ay;
            const double dd = dx * dx + dy * dy;
            const double tt_ = wx * dx + wy * dy;
            double u = dd > 0.0 ? tt_ / dd : 0.0;
            u = fmin(fmax(u, 0.0), 1.0);
            const double qx = wx - u * dx, qy = wy - u * dy;
            hit = hit || (qx * qx + qy * qy < r2);
        }
        hit = hit || inside;
    }
    return (outb ? 1 : 0) | (hit ? 2 : 0);
}

// x / y for a compile-time constant y, correctly rounded, in three instructions instead of the generic FP64
// division and its ~70-instruction slow path for a zero numerator (Markstein: with r = RN(1/y) and q0 = RN(x r),
// RN(q0 + r RN(x - y q0)) = RN(x / y) whenever the significand of y is not all ones; checked against the division
// on 1.5e9 random doubles for y = 3.6 and y = 19).  The result is bit-identical to `x / y`.
__device__ __forceinline__ double div_const(double x, double y, double r /* = 1.0 / y */)
{
    if (!(fabs(x) < 1e150)) return x / y;  // inf / nan / absurd magnitudes: the generic path
    const double q0 = x * r;
    return fma(fma(-q0, y, x), r, q0);
}

// mlp3:265-284
__device__ __forceinline__ void rotate_pt(double px, double py, double ca, double sa, double cx, double cy,
                                          double &ox, double &oy)
{
    const double x = px - cx, y = py - cy;
    const double xn = x * ca - y * sa;
    const double yn = x * sa + y * ca;
    ox = xn + cx;
    oy = yn + cy;
}

// Turn model of a batch (fcpp_batch.turn_model / clothoid_share)
struct TurnModel {
    int model;   // FCPP_TURN_ARC | FCPP_TURN_CLOTHOID
    double lam;  // clothoid share of the deflection
};

// Fresnel integrals S(t) = int_0^t sin(pi u^2/2) du, C(t) = int_0^t cos(pi u^2/2) du by their power
// series; |t| <= 1 here (a clothoid never deflects more than pi/2), 14 terms give < 4e-16.
__device__ __forceinline__ void fresnel_sc(double t, double &S, double &C)
{
    const double x = 1.5707963267948966 * t * t;
    const double x2 = x * x;
    double tc = 1.0, ts = x, sc = 1.0, ss = x / 3.0;
#pragma unroll
    for (int k = 1; k < 14; ++k) {
        tc *= -x2 / (double)((2 * k - 1) * (2 * k));
        ts *= -x2 / (double)((2 * k) * (2 * k + 1));
        sc += tc / (double)(4 * k + 1);
        ss += ts / (double)(4 * k + 3);
    }
    C = t * sc;
    S = t * ss;
}

// Unit-radius clothoid -> arc -> clothoid turn of total deflection phi sampled at n equal
// arc-length steps: local coordinates of sample i (xi along the entry heading, eta to the
// turning side).  oracle/clothoid.py cac_unit is the scipy.special.fresnel restatement.
static __device__ __noinline__ void cac_unit(double phi, int n, int i, double lam, double &xi, double &eta)
{
    const double alpha = lam * phi / 2, Lc = 2 * alpha, La = phi - 2 * alpha, Lt = 2 * Lc + La;
    const double s = (i == n - 1) ? Lt : i * (Lt / (n - 1));
    if (!(Lc > 0.0)) {
        double sn, cs;
        sincos(s, &sn, &cs);
        xi = sn;
        eta = 1 - cs;
        return;
    }
    const double a = sqrt(3.141592653589793 * Lc);
    if (s <= Lc) {
        double S, C;
        fresnel_sc(s / a, S, C);
        xi = a * C;
        eta = a * S;
        return;
    }
    double S1, C1, sa, ca;
    fresnel_sc(Lc / a, S1, C1);
    sincos(alpha, &sa, &ca);
    const double p1x = a * C1, p1y = a * S1;
    if (s <= Lc + La) {
        double sf, cf;
        sincos(alpha + (s - Lc), &sf, &cf);
        xi = p1x - sa + sf;
        eta = p1y + ca - cf;
        return;
    }
    double s2, c2, sp, cp;
    sincos(alpha + La, &s2, &c2);
    sincos(phi, &sp, &cp);
    const double p2x = p1x - sa + s2, p2y = p1y + ca - c2;
    const double cb = -cp, sb = -sp;  // rotation by phi + pi
    const double m1x = a * C1, m1y = -a * S1;
    const double ex = p2x - (cb * m1x - sb * m1y), ey = p2y - (sb * m1x + cb * m1y);
    double S, C;
    fresnel_sc((Lt - s) / a, S, C);
    const double mx = a * C, my = -a * S;
    xi = ex + (cb * mx - sb * my);
    eta = ey + (sb * mx + cb * my);
}

// 15-point quarter turn sample j at ring corner ci (mlp3:1049-1060, :1592-1603)
__device__ __forceinline__ void corner_arc_pt(const TrigTables &tt, const TurnModel &tm, double x, double y, double R,
                                              int ci, int j, double &ox, double &oy)
{
    if (tm.model == FCPP_TURN_CLOTHOID) {
        // same start pose and (clockwise) turning sense as the reference's arc, clothoid-arc-clothoid
        double xi, eta;
        cac_unit(1.5707963267948966, FCPP_CORNER_POINTS, j, tm.lam, xi, eta);
        if (ci == 0) {
            ox = x + R * eta;
            oy = y + R * xi;
        } else if (ci == 1) {
            ox = x - R * xi;
            oy = y + R * eta;
        } else if (ci == 2) {
            ox = x - R * eta;
            oy = y - R * xi;
        } else {
            ox = x + R * xi;
            oy = y - R * eta;
        }
        return;
    }
    const double c = tt.cos15[j], s = tt.sin15[j];
    if (ci == 0) {
        ox = x + R * (1 - c);
        oy = y + R * s;
    } else if (ci == 1) {
        ox = x - R * s;
        oy = y + R * (1 - c);
    } else if (ci == 2) {
        ox = x - R * (1 - c);
        oy = y - R * s;
    } else {
        ox = x + R * s;
        oy = y - R * (1 - c);
    }
}

// 1e-4 m fixed point (D5): one FP64 multiply, round-half-even
__device__ __forceinline__ int64_t qfix(double x) { return __double2ll_rn(x * FCPP_FIXED_UNIT); }

// ---- reverse fills (layout kernel; the coverage kernel for the start corner of another candidate) ----
// mlp3:1220-1288 — ray to the bbox lines x=0, x=field_length, y=0, y=field_width
__device__ inline double distance_to_boundary(double x, double y, double dx, double dy, double fl, double fw, double R)
{
    double best = -1.0;
    if (fabs(dx) > 1e-6) {
        double t = (0.0 - x) / dx;
        if (t > 0 && (best < 0 || t < best)) best = t;
        t = (fl - x) / dx;
        if (t > 0 && (best < 0 || t < best)) best = t;
    }
    if (fabs(dy) > 1e-6) {
        double t = (0.0 - y) / dy;
        if (t > 0 && (best < 0 || t < best)) best = t;
        t = (fw - y) / dy;
        if (t > 0 && (best < 0 || t < best)) best = t;
    }
    if (best < 0) return 2.0 * R;
    const double cap = FCPP_REV_CAP * R;
    return best < cap ? best : cap;
}

// mlp3:1154-1218: chord direction of the last two arc samples, length, sample count
__device__ inline int reverse_fill(const TrigTables &tt, const TurnModel &tm, double cx, double cy, int ci, double R,
                            double fl, double fw, double *rev /*[5]*/)
{
    double ex, ey, sx, sy;
    corner_arc_pt(tt, tm, cx, cy, R, ci, FCPP_CORNER_POINTS - 1, ex, ey);
    corner_arc_pt(tt, tm, cx, cy, R, ci, FCPP_CORNER_POINTS - 2, sx, sy);
    const double tx = ex - sx, ty = ey - sy;
    const double nrm = sqrt(tx * tx + ty * ty);
    double dx, dy;
    if (nrm > 1e-6) {
        dx = -tx / nrm;
        dy = -ty / nrm;
    } else {
        dx = -1.0;
        dy = 0.0;
    }
    const double len = distance_to_boundary(ex, ey, dx, dy, fl, fw, R);
    int n = (int)(len / FCPP_REV_SPACING);
    if (n < FCPP_REV_MIN_PTS) n = FCPP_REV_MIN_PTS;
    rev[0] = ex;
    rev[1] = ey;
    rev[2] = dx;
    rev[3] = dy;
    rev[4] = len;
    return n;
}

// ---------------------------------------------------------------------------------------------
// point generation: index -> (x, y, speed class, structure tag)
// ---------------------------------------------------------------------------------------------
// A plan is made of a few CONGRUENT pieces: every main pass (2 swath ends + 20 turn samples) is a
// translate / mirror image of the first one, every corner turn is the same 15-sample arc turned by a
// multiple of 90 degrees, the interior of a straight or of a reverse fill is equally spaced and
// collinear.  The structure tag of a point names its piece and its position in it, so that the plan
// kernel takes the segment length, the curvature and the curvature speed limit of such a point from a
// per-candidate table instead of recomputing sqrt / atan2 / divisions for every point; the first and
// last point of every piece (where two pieces meet) are GENERIC and are evaluated from the coordinates.
constexpr int SLOT_CHAIN = 0;      // + c: position in a regular main chain (0 .. 19 = turn samples, 20, 21 = the next swath's ends)
constexpr int SLOT_ARC = 22;       // + a: corner-turn sample a (1 .. 13)
constexpr int SLOT_REV = 37;       // + t: interior of the reverse fill after turn t of loop 0
constexpr int SLOT_STRAIGHT = 40;  // + 4 k + t: interior of straight t of headland loop k
constexpr int N_SLOTS = SLOT_STRAIGHT + 4 * FCPP_MAX_LOOPS;
constexpr int TAG_GENERIC = 252;   // + speed class
// The main work is a sequence of CHAINS separated by zero-length segments (a turn starts on the swath end it
// follows, mlp3:773-778, and the acceleration passes do not cross a zero-length segment, mlp3:560, :576): the
// first chain is the first swath, every further chain is one turn (20 samples) + the next swath (2 ends) = 22
// points.  All chains but the first and the last are congruent — same lengths, curvatures, limits, hence the same
// speed profile — and are evaluated ONCE per candidate (fcpp_plan.cu); only the first 2 and the last 22 main
// points are staged point by point together with the headland.
constexpr int CHAIN_POINTS = 2 + FCPP_UTURN_POINTS;
constexpr int MAIN_STAGED = 2 + CHAIN_POINTS;
__host__ __device__ __forceinline__ int main_skip(int n_main) { return n_main > MAIN_STAGED ? n_main - MAIN_STAGED : 0; }
// generic points (evaluated from their coordinates) get a fixed ordinal (deterministic summation order): the staged
// main points first, then 21 per headland loop: 0 = loop start, 1 + 2 t / 2 + 2 t = ends of straight t,
// 9 + 2 t / 10 + 2 t = ends of turn t, 15 + 2 t / 16 + 2 t = ends of reverse fill t
constexpr int GEN_PER_LOOP = 21;
constexpr int N_GENERIC = MAIN_STAGED + GEN_PER_LOOP * FCPP_MAX_LOOPS;

// ---- Ω (skip-row) pattern, FCPP_TURN_OMEGA: build-defined, restated in oracle/ref_planner.py (omega_*) ----
__device__ __forceinline__ int omega_skip(double R, double W)
{
    const int s = (int)ceil(2.0 * R / W - 1e-9);
    return s < 1 ? 1 : s;
}
// row of visit idx: blocks of 2 s rows, inside a block of m rows the lower and the upper half alternate
__device__ __forceinline__ int omega_row(int idx, int P, int s)
{
    const int base = (idx / (2 * s)) * (2 * s);
    const int m = min(2 * s, P - base);
    const int h = (m + 1) >> 1;
    const int k = idx - base;
    return base + (k >> 1) + ((k & 1) ? h : 0);
}
// sample a of the connecting turn between two rows d_abs apart, in the turn's frame (u outwards, v towards the next
// row): half circle of radius d_abs / 2 (table angles) or, below 2 R, the bulb turn of three radius-R arcs
__device__ __forceinline__ void omega_turn_local(const TrigTables &tt, double d_abs, double R, int a, double &u, double &v)
{
    if (d_abs >= 2.0 * R) {
        const double rho = d_abs / 2.0;
        u = rho * tt.sin20[a];
        v = rho - rho * tt.cos20[a];
        return;
    }
    const double xc = sqrt(4.0 * R * R - (R + d_abs / 2.0) * (R + d_abs / 2.0));
    const double alpha = atan2(xc, R + d_abs / 2.0);
    const double pi = 3.141592653589793;
    const double total = pi + 4.0 * alpha;
    const double phi = (a == FCPP_UTURN_POINTS - 1) ? total : a * (total / (FCPP_UTURN_POINTS - 1));
    if (phi <= alpha) {
        u = R * sin(phi);
        v = -R + R * cos(phi);
    } else if (phi <= pi + 3.0 * alpha) {
        const double hd = -alpha + (phi - alpha);
        u = 2.0 * R * sin(alpha) + R * sin(hd);
        v = (-R + 2.0 * R * cos(alpha)) - R * cos(hd);
    } else {
        const double hd = pi + alpha - (phi - (pi + 3.0 * alpha));
        u = -R * sin(hd);
        v = d_abs + R + R * cos(hd);
    }
}

// main-work point of the Ω pattern (visit index idx, position j in the pass) in the swath frame
static __device__ __noinline__ void omega_main_local_pt(const CandRec &r, const TrigTables &tt, double W, int idx, int j,
                                                        double &px, double &py)
{
    const int os = omega_skip(r.R, W);
    const int row = omega_row(idx, r.P, os);
    const int pi = (r.flags & FCPP_FLAG_REVERSE_ORDER) ? (r.P - 1 - row) : row;
    const double yy = r.min_y + pi * W;
    const bool go_left = (r.flags & FCPP_FLAG_START_FROM_RIGHT) ? ((idx & 1) == 0) : ((idx & 1) == 1);
    if (j < 2) {
        const double xs = r.min_x + r.R, xe = r.max_x - r.R;
        px = (go_left == (j == 0)) ? xe : xs;
        py = yy;
        return;
    }
    const int row2 = omega_row(idx + 1, r.P, os);
    const int pi2 = (r.flags & FCPP_FLAG_REVERSE_ORDER) ? (r.P - 1 - row2) : row2;
    const double d = (r.min_y + pi2 * W) - yy;
    double u, v;
    omega_turn_local(tt, fabs(d), r.R, j - 2, u, v);
    const double xe = go_left ? r.min_x + r.R : r.max_x - r.R;
    px = xe + (go_left ? -1.0 : 1.0) * u;
    py = yy + (d >= 0.0 ? 1.0 : -1.0) * v;
}

// main-work point (visit index idx, position j in the pass) in the swath frame, before the rotate-back.
// OMEGA is a compile-time switch (the plan kernel has an instance per pattern): a run-time test with an out-of-line
// call at every inlined copy cost the default patterns 5-9 % (measured).
template <bool OMEGA = false>
__device__ __forceinline__ void main_local_pt(const CandRec &r, const TrigTables &tt, const TurnModel &tm, double W,
                                              int idx, int j, double &px, double &py)
{
    // mlp3:744-780: visit index idx, pass index pi, 2 endpoints + 20 arc samples per pass
    if constexpr (OMEGA) {
        omega_main_local_pt(r, tt, W, idx, j, px, py);
        return;
    }
    const int pi = (r.flags & FCPP_FLAG_REVERSE_ORDER) ? (r.P - 1 - idx) : idx;
    const double yy = r.min_y + pi * W;  // mlp3:751
    const bool go_left = (r.flags & FCPP_FLAG_START_FROM_RIGHT) ? ((idx & 1) == 0) : ((idx & 1) == 1);
    if (j < 2) {
        const double xs = r.min_x + r.R, xe = r.max_x - r.R;  // mlp3:736-737
        px = (go_left == (j == 0)) ? xe : xs;                  // mlp3:761-764
        py = yy;
    } else {
        const int a = j - 2;
        if (tm.model == FCPP_TURN_CLOTHOID) {
            // clothoid-arc-clothoid U-turn leaving the swath end tangentially towards the next swath
            double xi, eta;
            cac_unit(3.141592653589793, FCPP_UTURN_POINTS, a, tm.lam, xi, eta);
            const double xe = go_left ? r.min_x + r.R : r.max_x - r.R;
            const double dir_x = go_left ? -1.0 : 1.0;
            const double dir_y = (r.flags & FCPP_FLAG_REVERSE_ORDER) ? -1.0 : 1.0;
            px = xe + dir_x * (r.R * xi);
            py = yy + dir_y * (r.R * eta);
        } else {
            const bool turn_right = !go_left;  // mlp3:776
            px = turn_right ? (r.max_x - r.R * tt.cos20[a]) : (r.min_x + r.R * tt.cos20[a]);  // mlp3:815, :822
            py = yy + r.R * tt.sin20[a];                                                       // mlp3:816, :823
        }
    }
}

template <bool OMEGA = false>
__device__ __forceinline__ void gen_point_tag(const CandRec &r, const TrigTables &tt, const TurnModel &tm, double W,
                                              int i, double &x, double &y, uint8_t &cls, int &tag, int &gord)
{
    gord = -1;
    if (i < r.n_main) {
        const int per = 2 + FCPP_UTURN_POINTS;
        const int idx = i / per;
        const int j = i - idx * per;
        double px, py;
        main_local_pt<OMEGA>(r, tt, tm, W, idx, j, px, py);
        cls = (j < 2) ? CLS_WORK : CLS_TURN;
        if (r.flags & FCPP_FLAG_ROTATED)
            rotate_pt(px, py, r.cos_a, r.sin_a, r.cx, r.cy, x, y);  // mlp3:709-714
        else {
            x = px;
            y = py;
        }
        tag = TAG_GENERIC + cls;  // staged main points (the first 2 and the last 22) are all generic
        gord = i < 2 ? i : i - main_skip(r.n_main);
        return;
    }
    // ---- headland (mlp3:943-1011) ----
    int hI = i - r.n_main;
    const int l0 = FCPP_POINTS_PER_LOOP + r.n_rev[0] + r.n_rev[1] + r.n_rev[2];
    int k, m;
    if (hI < l0) {
        k = 0;
        m = hI;
    } else {
        hI -= l0;
        k = 1 + hI / FCPP_POINTS_PER_LOOP;
        m = hI - (k - 1) * FCPP_POINTS_PER_LOOP;
    }
    const int sc = r.flags & FCPP_FLAG_CORNER_MASK;
    const int g0 = MAIN_STAGED + GEN_PER_LOOP * k;
    if (m == 0) {  // mlp3:978-980
        x = r.corners[k][sc][0];
        y = r.corners[k][sc][1];
        cls = CLS_HEAD;
        tag = TAG_GENERIC + CLS_HEAD;
        gord = g0;
        return;
    }
    m -= 1;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const int ci = (sc + t) & 3, ni = (sc + t + 1) & 3;
        if (m < FCPP_STRAIGHT_POINTS) {  // np.linspace(cur, nxt, 20), mlp3:1013-1022
            const double ax = r.corners[k][ci][0], ay = r.corners[k][ci][1];
            const double bx = r.corners[k][ni][0], by = r.corners[k][ni][1];
            if (m == FCPP_STRAIGHT_POINTS - 1) {
                x = bx;
                y = by;
            } else {
                // np.linspace: step = delta / 19 (an axis-aligned straight has a zero delta: no slow path here)
                constexpr double DIV = FCPP_STRAIGHT_POINTS - 1;
                const double sx = div_const(bx - ax, DIV, 1.0 / DIV);
                const double sy = div_const(by - ay, DIV, 1.0 / DIV);
                x = m * sx + ax;
                y = m * sy + ay;
            }
            cls = CLS_HEAD;
            tag = SLOT_STRAIGHT + 4 * k + t;
            if (m == 0 || m == FCPP_STRAIGHT_POINTS - 1) {
                tag = TAG_GENERIC + CLS_HEAD;
                gord = g0 + 1 + 2 * t + (m ? 1 : 0);
            }
            return;
        }
        m -= FCPP_STRAIGHT_POINTS;
        if (t < 3) {
            if (m < FCPP_CORNER_POINTS) {
                corner_arc_pt(tt, tm, r.corners[k][ni][0], r.corners[k][ni][1], r.R, ni, m, x, y);
                cls = CLS_TURN;
                tag = SLOT_ARC + m;
                if (m == 0 || m == FCPP_CORNER_POINTS - 1) {
                    tag = TAG_GENERIC + CLS_TURN;
                    gord = g0 + 9 + 2 * t + (m ? 1 : 0);
                }
                return;
            }
            m -= FCPP_CORNER_POINTS;
            const int nr = (k == 0) ? r.n_rev[t] : 0;
            if (m < nr) {  // mlp3:1214-1216
                const double len = r.rev[t][4];
                const double tt_ = (m == nr - 1) ? len : m * (len / (nr - 1));
                x = r.rev[t][0] + tt_ * r.rev[t][2];
                y = r.rev[t][1] + tt_ * r.rev[t][3];
                cls = CLS_REVERSE;
                tag = SLOT_REV + t;
                if (m == 0 || m == nr - 1) {
                    tag = TAG_GENERIC + CLS_REVERSE;
                    gord = g0 + 15 + 2 * t + (m ? 1 : 0);
                }
                return;
            }
            m -= nr;
        }
    }
    x = 0.0;
    y = 0.0;
    cls = CLS_HEAD;  // unreachable
    tag = TAG_GENERIC + CLS_HEAD;
    gord = 0;
}

template <bool OMEGA = false>
__device__ __forceinline__ void gen_point(const CandRec &r, const TrigTables &tt, const TurnModel &tm, double W, int i,
                                          double &x, double &y, uint8_t &cls)
{
    int tag, gord;
    gen_point_tag<OMEGA>(r, tt, tm, W, i, x, y, cls, tag, gord);
}


// launchers (defined in the .cu files, called from fcpp_api.cu)
cudaError_t fcpp_launch_layout(fcpp_handle *h, const fcpp_batch &b, int32_t *d_n_pts, int64_t *d_offsets,
                               cudaStream_t st);
cudaError_t fcpp_launch_plan(fcpp_handle *h, const fcpp_batch &b, const fcpp_outputs &o, cudaStream_t st);
cudaError_t fcpp_launch_cover(fcpp_handle *h, const fcpp_batch &b, const fcpp_outputs &o, cudaStream_t st);
cudaError_t fcpp_launch_speed_verify(fcpp_handle *h, const fcpp_vehicle &veh, const double *d_path,
                                     const double *d_speeds_in, const int64_t *d_offsets, int64_t n_paths,
                                     int64_t max_len, int do_speed_plan, double *d_speeds_out, double *d_curv,
                                     fcpp_summary *d_summary, cudaStream_t st);
cudaError_t fcpp_launch_raster_window(fcpp_handle *h, const double *d_path, int32_t n_pts, double radius,
                                      double ox, double oy, double hc, int32_t g, uint32_t *d_bits,
                                      int64_t *d_count, cudaStream_t st);
cudaError_t fcpp_launch_tours(fcpp_handle *h, const double *d_D, int32_t n, const int32_t *d_pop,
                              int64_t pop_size, double *d_out, double *d_fit, cudaStream_t st);
void fcpp_ga_sizes(const fcpp_ga_config &cfg, int m_in, int &keep, int &e_take, int &m_out);
cudaError_t fcpp_launch_ga_init(fcpp_handle *h, const fcpp_ga_config &cfg, int n, int32_t *d_pop, cudaStream_t st);
cudaError_t fcpp_launch_ga_generation(fcpp_handle *h, const fcpp_ga_config &cfg, int gen, int n,
                                      const int32_t *d_pop_in, const double *d_fit, int m_in, int32_t *d_pop_out,
                                      int *d_rank, int32_t *d_trace, const void *d_state, cudaStream_t st);
cudaError_t fcpp_launch_ga_track(fcpp_handle *h, const double *d_fit, const double *d_len, const int32_t *d_pop,
                                 int m, int n, int threshold, int initial, void *d_state, int32_t *d_best_route,
                                 double *d_history, cudaStream_t st);
cudaError_t fcpp_launch_ga_rotate(fcpp_handle *h, const int32_t *d_route, int n, int32_t *d_out, cudaStream_t st);
size_t fcpp_ga_state_bytes();
void fcpp_ga_read_state(const void *host_copy, int &gen, int &stagnant, int &done, int &last_gen, double &best_fit,
                        double &best_len);
cudaError_t fcpp_launch_winner_records(fcpp_handle *h, const fcpp_summary *d_summary, int64_t lo, int64_t hi,
                                       const int64_t *d_best_cand, int32_t n_fields, void *d_out, cudaStream_t st);
cudaError_t fcpp_launch_distance_matrix(fcpp_handle *h, const double *d_pos, int32_t n, double *d_D, cudaStream_t st);
cudaError_t fcpp_launch_connection_matrix(fcpp_handle *h, const double *d_verts, int32_t n_fields, double depot_x,
                                          double depot_y, double *d_C, int32_t *d_arg, cudaStream_t st);
cudaError_t fcpp_launch_status_count(fcpp_handle *h, const fcpp_summary *d_summary, int64_t n, int mask, int32_t *d_count,
                                     cudaStream_t st);
cudaError_t fcpp_launch_select(fcpp_handle *h, const fcpp_summary *d_summary, const int32_t *d_cand_field,
                               int64_t n_cand, int32_t n_fields, const fcpp_selection &sel, int64_t cand_base,
                               double *d_cost, int64_t *d_cand, cudaStream_t st);
cudaError_t fcpp_launch_select_merge(fcpp_handle *h, const int64_t *d_gathered, int world, int32_t n_fields, int k,
                                     double *d_cost, int64_t *d_cand, cudaStream_t st);
cudaError_t fcpp_launch_sweep(fcpp_handle *h, const fcpp_batch &b, fcpp_sweep *d_out, cudaStream_t st);
cudaError_t fcpp_launch_sweep_paths(fcpp_handle *h, const double *d_path, const int64_t *d_offsets, int64_t n_paths,
                                    const int32_t *d_n_main, const int32_t *d_vert_start, const double *d_verts,
                                    int32_t n_polys, double radius, fcpp_sweep *d_out, cudaStream_t st);
// whole-field / headland-band coverage and D3 counts of polylines in device memory (fcpp_cover.cu)
struct PathCoverSrc {
    const double *path;           // [total][2]
    const int64_t *offsets;       // [n + 1]
    int64_t n;
    // caller paths: per path its field, headland width and main-work points (n_main NULL: 0)
    const int32_t *path_field;
    const double *headland_width;
    const int32_t *n_main;
    // materialised plans (recs != NULL): field, R and n_main from the candidate records; a record with a status, no
    // points, or whose summary has FCPP_CAND_TOO_LARGE (its path was not written) is skipped
    const CandRec *recs;
    const fcpp_summary *summary;
    int32_t n_fields;
    const double *field_verts;    // [F][4][2]
    const int32_t *obs_poly_start, *obs_vert_start;  // fcpp_batch layout; obs_poly_start NULL: no obstacles
    const double *obs_verts;
    double radius, grid_h;
};
cudaError_t fcpp_launch_path_cover(fcpp_handle *h, const PathCoverSrc &src, fcpp_path_cover *d_out, cudaStream_t st);
