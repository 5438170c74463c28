// fcpp_sweep.cu — segment-level obstacle sweep (DESIGN.md §3.9): how many segments of a plan, and how many metres,
// drive through the obstacle region O, the set of points D3's per-point test counts (inside an obstacle polygon, or
// closer than W/2 to one of its edges).  oracle/sweep.py states the rule; the expressions here are the same, in the
// same order (-fmad=false), so the per-segment measures are the same doubles.
//
// sweep_gen_kernel: generated plans, one CTA per candidate, points regenerated from the candidate records with the
// plan kernel's own point code (fcpp_internal.cuh).  A plan is cut into PIECES (a swath, a U-turn, a headland
// straight, a corner arc, a reverse fill) that tile its points in order; the segment from a piece's last point to the
// next piece's first point is its JOIN.  Joins are always swept; a piece's inner segments only when a conservative
// world-frame bound of the piece meets an obstacle's box grown by W/2 + 1e-6 m.  The swept segments of a round of
// pieces get a dense index (block scan), so warps stay full.
// sweep_path_kernel: caller-supplied paths, one CTA per path, every segment.
// Both sum each layer's hit measures left to right in segment order (hits are listed per round and added by one
// thread), so the two forms give the same bytes on the same points.
#include "fcpp_internal.cuh"

namespace {

constexpr int TS_GEN = 128;            // threads per CTA, generated plans
constexpr int TS_PATH = 256;           // threads per CTA, caller-supplied paths
constexpr int SW_MAX_VERTS = 1024;     // obstacle vertices staged in shared memory; a field with more is read from
constexpr int SW_MAX_POLYS = 256;      // global memory (same results: the staged boxes only skip empty contributions)
constexpr int SW_IVL = 12;             // capsule intervals of one segment listed in shared memory
constexpr double SW_PI = 3.141592653589793;

__host__ __device__ inline size_t al16(size_t x) { return (x + 15) & ~size_t(15); }

// one field's obstacles: vertices and polygon ranges in shared memory with their boxes grown by r + 1e-6 (bb), or
// the caller's global arrays (bb == nullptr: no box rejects)
struct ObsView {
    const double *xy;
    const int32_t *vs;  // [n + 1]
    const double *bb;   // [n][4] or nullptr
    int n;
    double ux0, uy0, ux1, uy1;  // union of the grown boxes (+-inf without boxes)
};

__device__ __forceinline__ bool box_meets(const ObsView &o, double x0, double y0, double x1, double y1)
{
    if (!o.bb) return true;
    if (x1 < o.ux0 || y1 < o.uy0 || x0 > o.ux1 || y0 > o.uy1) return false;
    for (int p = 0; p < o.n; ++p)
        if (!(x1 < o.bb[4 * p] || y1 < o.bb[4 * p + 1] || x0 > o.bb[4 * p + 2] || y0 > o.bb[4 * p + 3])) return true;
    return false;
}

// the D3 obstacle predicate at one point (fcpp_plan.cu point_tests_impl, oracle/sweep.py in_region)
__device__ bool in_region(const ObsView &o, double r2, double x, double y)
{
    for (int p = 0; p < o.n; ++p) {
        if (o.bb && (x < o.bb[4 * p] || y < o.bb[4 * p + 1] || x > o.bb[4 * p + 2] || y > o.bb[4 * p + 3])) continue;
        const int vs = o.vs[p], ve = o.vs[p + 1];
        bool inside = false, hit = false;
        for (int q = vs; q < ve; ++q) {
            const int q1 = (q + 1 < ve) ? q + 1 : vs;
            const double ax = o.xy[2 * q], ay = o.xy[2 * q + 1];
            const double bx = o.xy[2 * q1], by = o.xy[2 * q1 + 1];
            if ((ay > y) != (by > y)) {
                const double xi = ax + (y - ay) * (bx - ax) / (by - ay);
                if (x < xi) inside = !inside;
            }
            const double dx = bx - ax, dy = by - ay, wx = x - ax, wy = y - ay;
            const double dd = dx * dx + dy * dy;
            const double tt_ = wx * dx + wy * dy;
            double u = dd > 0.0 ? tt_ / dd : 0.0;
            u = fmin(fmax(u, 0.0), 1.0);
            const double qx = wx - u * dx, qy = wy - u * dy;
            hit = hit || (qx * qx + qy * qy < r2);
        }
        if (hit || inside) return true;
    }
    return false;
}

// parameter interval of a + t d (t in [0, 1]) within r of the edge p q: the hull of the two vertex-disc intervals and
// the strip interval, clipped; false when empty or a single point (oracle/sweep.py capsule_interval)
__device__ __forceinline__ bool capsule(double ax, double ay, double dx, double dy, double A, double px, double py,
                                        double qx, double qy, double r, double r2, double &lo_out, double &hi_out)
{
    double lo = INFINITY, hi = -INFINITY;
#pragma unroll
    for (int v = 0; v < 2; ++v) {
        const double cx = v ? qx : px, cy = v ? qy : py;
        const double wx = ax - cx, wy = ay - cy;
        const double B = dx * wx + dy * wy;
        const double Cc = (wx * wx + wy * wy) - r2;
        const double disc = B * B - A * Cc;
        if (disc >= 0.0) {
            const double s = sqrt(disc);
            lo = fmin(lo, (-B - s) / A);
            hi = fmax(hi, (-B + s) / A);
        }
    }
    const double ex = qx - px, ey = qy - py;
    const double ee = ex * ex + ey * ey;
    if (ee > 0.0) {
        const double wx = ax - px, wy = ay - py;
        double s_lo = -INFINITY, s_hi = INFINITY;
        const double w0 = wx * ex + wy * ey, w1 = dx * ex + dy * ey;
        const double h0 = ex * wy - ey * wx, h1 = ex * dy - ey * dx;
        const double rl = r * sqrt(ee);
        bool ok = true;
        if (w1 == 0.0) {
            ok = 0.0 <= w0 && w0 <= ee;
        } else {
            double ta = (0.0 - w0) / w1, tb = (ee - w0) / w1;
            if (w1 < 0.0) {
                const double t = ta;
                ta = tb;
                tb = t;
            }
            s_lo = fmax(s_lo, ta);
            s_hi = fmin(s_hi, tb);
        }
        if (h1 == 0.0) {
            ok = ok && fabs(h0) <= rl;
        } else {
            double ta = (-rl - h0) / h1, tb = (rl - h0) / h1;
            if (h1 < 0.0) {
                const double t = ta;
                ta = tb;
                tb = t;
            }
            s_lo = fmax(s_lo, ta);
            s_hi = fmin(s_hi, tb);
        }
        if (ok && s_lo <= s_hi) {
            lo = fmin(lo, s_lo);
            hi = fmax(hi, s_hi);
        }
    }
    lo = fmax(lo, 0.0);
    hi = fmin(hi, 1.0);
    lo_out = lo;
    hi_out = hi;
    return lo < hi;
}

// the capsule intervals of every edge near the segment: the smallest interval end above `cur` (1 when none); with
// `ivl` (a thread's column of SW_IVL interval slots, stride T) the intervals are also listed, their number in nv
template <int T>
__device__ __forceinline__ double edge_scan(const ObsView &o, double r, double r2, double ax, double ay, double dx,
                                            double dy, double A, double sx0, double sy0, double sx1, double sy1,
                                            double cur, double *ivl, int &nv)
{
    const double g = r + 1e-6;
    double nxt = 1.0;
    for (int p = 0; p < o.n; ++p) {
        if (o.bb && (sx1 < o.bb[4 * p] || sy1 < o.bb[4 * p + 1] || sx0 > o.bb[4 * p + 2] || sy0 > o.bb[4 * p + 3]))
            continue;
        const int vs = o.vs[p], ve = o.vs[p + 1];
        for (int q = vs; q < ve; ++q) {
            const int q1 = (q + 1 < ve) ? q + 1 : vs;
            const double px = o.xy[2 * q], py = o.xy[2 * q + 1];
            const double qx = o.xy[2 * q1], qy = o.xy[2 * q1 + 1];
            // an edge whose box grown by r + 1e-6 misses the segment's box has an empty interval
            if (sx1 < fmin(px, qx) - g || sx0 > fmax(px, qx) + g || sy1 < fmin(py, qy) - g || sy0 > fmax(py, qy) + g)
                continue;
            double lo, hi;
            if (capsule(ax, ay, dx, dy, A, px, py, qx, qy, r, r2, lo, hi)) {
                if (lo > cur) nxt = fmin(nxt, lo);
                if (hi > cur) nxt = fmin(nxt, hi);
                if (ivl) {
                    if (nv < SW_IVL) {
                        ivl[(2 * nv) * T] = lo;
                        ivl[(2 * nv + 1) * T] = hi;
                    }
                    ++nv;
                }
            }
        }
    }
    return nxt;
}

// metres of the segment a -> b inside O.  The breakpoints are visited in ascending order: each step takes the
// smallest interval end above the current one (equal ends are one breakpoint, as in the oracle's set).  The
// intervals are computed once and listed in shared memory; a segment near more than SW_IVL edges recomputes them
// at every step instead (same breakpoints).
template <int T>
__device__ double seg_measure(const ObsView &o, double r, double r2, double ax, double ay, double bx, double by,
                              double *ivl)
{
    const double dx = bx - ax, dy = by - ay;
    const double A = dx * dx + dy * dy;
    if (A == 0.0) return 0.0;
    const double sx0 = fmin(ax, bx), sx1 = fmax(ax, bx), sy0 = fmin(ay, by), sy1 = fmax(ay, by);
    if (!box_meets(o, sx0, sy0, sx1, sy1)) return 0.0;
    int nv = 0;
    double cur = 0.0, s = 0.0;
    double nxt = edge_scan<T>(o, r, r2, ax, ay, dx, dy, A, sx0, sy0, sx1, sy1, cur, ivl, nv);
    while (true) {
        const double tm = 0.5 * (cur + nxt);
        if (in_region(o, r2, ax + tm * dx, ay + tm * dy)) s += nxt - cur;
        cur = nxt;
        if (!(cur < 1.0)) break;
        if (nv <= SW_IVL) {
            nxt = 1.0;
            for (int k = 0; k < nv; ++k) {
                FCPP_ASSERT(k < SW_IVL);
                const double lo = ivl[(2 * k) * T], hi = ivl[(2 * k + 1) * T];
                if (lo > cur) nxt = fmin(nxt, lo);
                if (hi > cur) nxt = fmin(nxt, hi);
            }
        } else {
            int unused = 0;
            nxt = edge_scan<T>(o, r, r2, ax, ay, dx, dy, A, sx0, sy0, sx1, sy1, cur, nullptr, unused);
        }
    }
    return s * sqrt(A);
}

// shared memory of both kernels besides the obstacle tables
template <int T>
struct SweepShared {
    double m[T];             // measure of this round's segment of each thread
    uint8_t layer[T];        // 0 main, 1 headland, 2 none
    uint32_t hits[T / 32];   // per-warp ballots of m > 0
    int32_t scan[T / 32];
    int32_t poff[T];         // gen: dense offset of the round's piece j
    int32_t pseg[T];         // gen: first swept segment of piece j
    double ivl[2 * SW_IVL][T];  // the capsule intervals of each thread's segment (column = thread)
};

template <int T>
__device__ __forceinline__ int block_excl_scan(int v, int32_t *sh, int &total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += o;
    }
    if (lane == 31) sh[warp] = inc;
    __syncthreads();
    int pre = 0;
    total = 0;
#pragma unroll
    for (int w = 0; w < T / 32; ++w) {
        const int t = sh[w];
        if (w < warp) pre += t;
        total += t;
    }
    __syncthreads();
    return pre + inc - v;
}

// one round: every thread's (m, layer); thread 0 adds the hits in thread order (= segment order), left to right
template <int T>
__device__ __forceinline__ void ordered_add(SweepShared<T> &sh, double m, int layer, fcpp_sweep &acc)
{
    const int tid = threadIdx.x;
    FCPP_ASSERT(tid < T);
    sh.m[tid] = m;
    sh.layer[tid] = (uint8_t)layer;
    const unsigned bal = __ballot_sync(0xffffffffu, m > 0.0 && layer < 2);
    if ((tid & 31) == 0) sh.hits[tid >> 5] = bal;
    __syncthreads();
    if (tid == 0) {
        for (int w = 0; w < T / 32; ++w) {
            unsigned bits = sh.hits[w];
            while (bits) {
                const int k = 32 * w + __ffs(bits) - 1;
                bits &= bits - 1;
                FCPP_ASSERT(k < T && sh.layer[k] < 2);
                if (sh.layer[k] == 0) {
                    acc.n_seg_main += 1;
                    acc.len_main += sh.m[k];
                } else {
                    acc.n_seg_head += 1;
                    acc.len_head += sh.m[k];
                }
            }
        }
    }
    __syncthreads();
}

// stage one obstacle set (polygons p0 .. p0 + np of the global tables) in shared memory when it fits, and build the
// view; the caller synchronises before use
__device__ ObsView stage_obstacles(const int32_t *vert_start, const double *verts, int p0, int np, int cap_v,
                                   int cap_p, double *s_xy, double *s_bb, int32_t *s_vs, double r, int tid, int T)
{
    ObsView o;
    o.n = np;
    const int v0 = vert_start[p0], nv = vert_start[p0 + np] - v0;
    if (np <= cap_p && nv <= cap_v) {
        for (int k = tid; k < 2 * nv; k += T) {
            FCPP_ASSERT(k < 2 * cap_v);
            s_xy[k] = verts[2 * (int64_t)v0 + k];
        }
        for (int k = tid; k <= np; k += T) {
            FCPP_ASSERT(k <= cap_p);
            s_vs[k] = vert_start[p0 + k] - v0;
        }
        __syncthreads();
        const double g = r + 1e-6;
        for (int p = tid; p < np; p += T) {
            double x0 = 1e300, y0 = 1e300, x1 = -1e300, y1 = -1e300;
            for (int q = s_vs[p]; q < s_vs[p + 1]; ++q) {
                FCPP_ASSERT(q >= 0 && q < cap_v);
                x0 = fmin(x0, s_xy[2 * q]);
                x1 = fmax(x1, s_xy[2 * q]);
                y0 = fmin(y0, s_xy[2 * q + 1]);
                y1 = fmax(y1, s_xy[2 * q + 1]);
            }
            FCPP_ASSERT(p < cap_p);
            s_bb[4 * p] = x0 - g;
            s_bb[4 * p + 1] = y0 - g;
            s_bb[4 * p + 2] = x1 + g;
            s_bb[4 * p + 3] = y1 + g;
        }
        __syncthreads();
        o.xy = s_xy;
        o.vs = s_vs;
        o.bb = s_bb;
        o.ux0 = o.uy0 = INFINITY;
        o.ux1 = o.uy1 = -INFINITY;
        for (int p = 0; p < np; ++p) {  // every thread, from shared memory: a few polygons
            o.ux0 = fmin(o.ux0, s_bb[4 * p]);
            o.uy0 = fmin(o.uy0, s_bb[4 * p + 1]);
            o.ux1 = fmax(o.ux1, s_bb[4 * p + 2]);
            o.uy1 = fmax(o.uy1, s_bb[4 * p + 3]);
        }
    } else {
        o.xy = verts;
        o.vs = vert_start + p0;
        o.bb = nullptr;
        o.ux0 = o.uy0 = -INFINITY;
        o.ux1 = o.uy1 = INFINITY;
    }
    return o;
}

template <int T>
__host__ __device__ inline size_t sweep_smem_bytes(size_t fixed, int cap_v, int cap_p)
{
    return al16(fixed) + al16(sizeof(double) * 2 * (cap_v > 0 ? cap_v : 1)) + al16(sizeof(double) * 4 * (cap_p > 0 ? cap_p : 1)) +
           al16(sizeof(int32_t) * (cap_p + 1));
}

// ---------------------------------------------------------------------------------------------------------------------
// generated plans
// ---------------------------------------------------------------------------------------------------------------------
struct GenShared {
    CandRec rec;
    TrigTables tt;
    SweepShared<TS_GEN> s;
};

struct SweepArgs {
    fcpp_batch b;
    const CandRec *recs;
    const TrigTables *trig;
    fcpp_sweep *out;
    int cap_v, cap_p;
};

constexpr int HEAD_SLOTS = 11;  // per headland loop: start point, S0, A0, R0, S1, A1, R1, S2, A2, R2, S3

// Piece j of a layer: its first point p0 (layer-relative), its point count np, and whether its inner segments can
// meet an obstacle.  Bounds: a swath is swept directly (its one segment's own box test is the cheapest reject); a
// U-turn lies in the disc around its first sample whose radius is the turn's arc length; a headland straight and a
// reverse fill in the box of their end points; a corner arc in the disc around the ring corner it starts on.  Every
// bound is grown by 1e-6 m.
template <bool OMEGA>
__device__ void gen_piece(const CandRec &r, const TrigTables &tt, const TurnModel &tm, double W, const ObsView &o,
                          int head, int j, int &p0, int &np, bool &listed)
{
    const double lam = tm.model == FCPP_TURN_CLOTHOID ? tm.lam : 0.0;
    double x0, y0, x1, y1;
    if (!head) {
        const int idx = j >> 1;
        if ((j & 1) == 0) {
            p0 = CHAIN_POINTS * idx;
            np = 2;
            listed = true;
            return;
        }
        p0 = CHAIN_POINTS * idx + 2;
        np = FCPP_UTURN_POINTS;
        double cx, cy;
        uint8_t cls;
        gen_point<OMEGA>(r, tt, tm, W, p0, cx, cy, cls);
        double rho;
        if constexpr (OMEGA) {
            const int os = omega_skip(r.R, W);
            const double d = fabs((double)(omega_row(idx + 1, r.P, os) - omega_row(idx, r.P, os))) * W;
            rho = SW_PI * fmax(d, 3.0 * r.R);  // half circle of radius d / 2, or the bulb's three arcs (< 3 pi R)
        } else {
            rho = SW_PI * (1.0 + lam) * r.R;
        }
        rho += 1e-6;
        x0 = cx - rho, y0 = cy - rho, x1 = cx + rho, y1 = cy + rho;
    } else {
        const int k = j / HEAD_SLOTS, s = j - k * HEAD_SLOTS;
        const int l0 = FCPP_POINTS_PER_LOOP + r.n_rev[0] + r.n_rev[1] + r.n_rev[2];
        int p = k == 0 ? 0 : l0 + (k - 1) * FCPP_POINTS_PER_LOOP;
        int sz = 1;
        for (int u = 1; u <= s; ++u) {
            p += sz;
            const int t = (u - 1) / 3, kind = (u - 1) % 3;  // 0 straight, 1 arc, 2 reverse fill
            sz = kind == 0 ? FCPP_STRAIGHT_POINTS : kind == 1 ? FCPP_CORNER_POINTS : (k == 0 ? r.n_rev[t] : 0);
        }
        p0 = p;
        np = sz;
        listed = false;
        if (s == 0 || np < 2) return;
        const int t = (s - 1) / 3, kind = (s - 1) % 3;
        const int sc = r.flags & FCPP_FLAG_CORNER_MASK, ci = (sc + t) & 3, ni = (sc + t + 1) & 3;
        if (kind == 0) {
            const double ax = r.corners[k][ci][0], ay = r.corners[k][ci][1];
            const double bx = r.corners[k][ni][0], by = r.corners[k][ni][1];
            x0 = fmin(ax, bx), y0 = fmin(ay, by), x1 = fmax(ax, bx), y1 = fmax(ay, by);
        } else if (kind == 1) {
            const double rho = 0.5 * SW_PI * (1.0 + lam) * r.R;
            const double cx = r.corners[k][ni][0], cy = r.corners[k][ni][1];
            x0 = cx - rho, y0 = cy - rho, x1 = cx + rho, y1 = cy + rho;
        } else {
            const double *v = r.rev[t];
            const double ex = v[0] + v[4] * v[2], ey = v[1] + v[4] * v[3];
            x0 = fmin(v[0], ex), y0 = fmin(v[1], ey), x1 = fmax(v[0], ex), y1 = fmax(v[1], ey);
        }
        x0 -= 1e-6, y0 -= 1e-6, x1 += 1e-6, y1 += 1e-6;
    }
    listed = box_meets(o, x0, y0, x1, y1);
}

template <bool OMEGA>
__device__ __forceinline__ void sweep_gen_body(const SweepArgs &a, unsigned char *smem, int64_t cand)
{
    constexpr int T = TS_GEN;
    const int tid = threadIdx.x;
    GenShared &g = *reinterpret_cast<GenShared *>(smem);
    size_t off = al16(sizeof(GenShared));
    double *s_xy = (double *)(smem + off);
    off += al16(sizeof(double) * 2 * (a.cap_v > 0 ? a.cap_v : 1));
    double *s_bb = (double *)(smem + off);
    off += al16(sizeof(double) * 4 * (a.cap_p > 0 ? a.cap_p : 1));
    int32_t *s_vs = (int32_t *)(smem + off);
    FCPP_ASSERT(sweep_smem_bytes<T>(sizeof(GenShared), a.cap_v, a.cap_p) <= fcpp_dynamic_smem_bytes() + 0u);

    for (int k = tid; k < (int)(sizeof(CandRec) / 16); k += T)
        reinterpret_cast<int4 *>(&g.rec)[k] = reinterpret_cast<const int4 *>(a.recs + cand)[k];
    for (int k = tid; k < (int)(sizeof(TrigTables) / sizeof(double)); k += T)
        ((double *)&g.tt)[k] = ((const double *)a.trig)[k];
    __syncthreads();
    const CandRec &r = g.rec;
    int p0 = 0, npoly = 0;
    if (a.b.obs_poly_start) {
        p0 = a.b.obs_poly_start[r.field];
        npoly = a.b.obs_poly_start[r.field + 1] - p0;
    }
    if (r.status != 0 || r.n_total == 0 || npoly <= 0) {  // dead candidates and fields without obstacles
        if (tid == 0) a.out[cand] = fcpp_sweep{0, 0, 0.0, 0.0};
        return;
    }
    const double W = a.b.vehicle.working_width;
    const double rr = W / 2, r2 = rr * rr;
    const ObsView o = stage_obstacles(a.b.obs_vert_start, a.b.obs_verts, p0, npoly, a.cap_v, a.cap_p, s_xy, s_bb, s_vs,
                                      rr, tid, T);
    TurnModel tm;
    tm.model = a.b.turn_model;
    tm.lam = a.b.clothoid_share;
    fcpp_sweep acc{0, 0, 0.0, 0.0};  // thread 0's
    for (int head = 0; head < 2; ++head) {
        const int n_layer = head ? r.n_head : r.n_main;
        const int base_pt = head ? r.n_main : 0;
        const int n_pieces = head ? HEAD_SLOTS * r.K : (n_layer > 0 ? 2 * r.P - 1 : 0);
        for (int j0 = 0; j0 < n_pieces; j0 += T) {
            const int j = j0 + tid;
            int cnt = 0, seg0 = 0;
            if (j < n_pieces) {
                int q0, np;
                bool listed;
                gen_piece<OMEGA>(r, g.tt, tm, W, o, head, j, q0, np, listed);
                if (np > 0) {
                    const int inner = listed ? np - 1 : 0;
                    const int join = (q0 + np < n_layer) ? 1 : 0;
                    cnt = inner + join;
                    seg0 = listed ? q0 : q0 + np - 1;
                }
            }
            int total;
            const int pos = block_excl_scan<T>(cnt, g.s.scan, total);
            g.s.poff[tid] = pos;
            g.s.pseg[tid] = seg0;
            __syncthreads();
            for (int q0 = 0; q0 < total; q0 += T) {
                const int q = q0 + tid;
                double m = 0.0;
                if (q < total) {
                    int lo = 0, hi = T - 1;  // the last piece whose offset is <= q (empty pieces share offsets)
                    while (lo < hi) {
                        const int mid = (lo + hi + 1) >> 1;
                        if (g.s.poff[mid] <= q)
                            lo = mid;
                        else
                            hi = mid - 1;
                    }
                    FCPP_ASSERT(lo >= 0 && lo < T);
                    const int seg = g.s.pseg[lo] + (q - g.s.poff[lo]);
                    FCPP_ASSERT(seg >= 0 && seg + 1 < n_layer);
                    double ax, ay, bx, by;
                    uint8_t cls;
                    gen_point<OMEGA>(r, g.tt, tm, W, base_pt + seg, ax, ay, cls);
                    gen_point<OMEGA>(r, g.tt, tm, W, base_pt + seg + 1, bx, by, cls);
                    m = seg_measure<T>(o, rr, r2, ax, ay, bx, by, &g.s.ivl[0][tid]);
                }
                ordered_add<T>(g.s, m, head, acc);
            }
        }
    }
    if (tid == 0) a.out[cand] = acc;
}

__global__ void __launch_bounds__(TS_GEN) sweep_gen_kernel(const SweepArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    sweep_gen_body<false>(a, smem_raw, blockIdx.x);
}

__global__ void __launch_bounds__(TS_GEN) sweep_gen_omega_kernel(const SweepArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    sweep_gen_body<true>(a, smem_raw, blockIdx.x);
}

// ---------------------------------------------------------------------------------------------------------------------
// caller-supplied paths
// ---------------------------------------------------------------------------------------------------------------------
struct PathSweepArgs {
    const double *path;
    const int64_t *offsets;
    const int32_t *n_main;
    const int32_t *vert_start;
    const double *verts;
    int n_polys;
    double radius;
    fcpp_sweep *out;
};

__global__ void __launch_bounds__(TS_PATH) sweep_path_kernel(const PathSweepArgs a)
{
    constexpr int T = TS_PATH;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SweepShared<T> &sh = *reinterpret_cast<SweepShared<T> *>(smem_raw);
    size_t off = al16(sizeof(SweepShared<T>));
    double *s_xy = (double *)(smem_raw + off);
    off += al16(sizeof(double) * 2 * SW_MAX_VERTS);
    double *s_bb = (double *)(smem_raw + off);
    off += al16(sizeof(double) * 4 * SW_MAX_POLYS);
    int32_t *s_vs = (int32_t *)(smem_raw + off);
    FCPP_ASSERT(sweep_smem_bytes<T>(sizeof(SweepShared<T>), SW_MAX_VERTS, SW_MAX_POLYS) <= fcpp_dynamic_smem_bytes() + 0u);
    const int tid = threadIdx.x;
    const int64_t path = blockIdx.x;
    const int64_t o0 = a.offsets[path];
    const int N = (int)(a.offsets[path + 1] - o0);
    int nm = a.n_main ? a.n_main[path] : N;
    nm = nm < 0 ? 0 : (nm > N ? N : nm);
    if (a.n_polys <= 0 || N < 2) {
        if (tid == 0) a.out[path] = fcpp_sweep{0, 0, 0.0, 0.0};
        return;
    }
    const double rr = a.radius, r2 = rr * rr;
    const ObsView o = stage_obstacles(a.vert_start, a.verts, 0, a.n_polys, SW_MAX_VERTS, SW_MAX_POLYS, s_xy, s_bb, s_vs,
                                      rr, tid, T);
    const double2 *p = reinterpret_cast<const double2 *>(a.path) + o0;
    fcpp_sweep acc{0, 0, 0.0, 0.0};  // thread 0's
    for (int i0 = 0; i0 < N - 1; i0 += T) {
        const int i = i0 + tid;
        double m = 0.0;
        int layer = 2;
        if (i < N - 1) {
            layer = (i + 1 < nm) ? 0 : (i >= nm ? 1 : 2);  // the junction nm - 1 -> nm belongs to neither layer
            if (layer < 2) {
                const double2 pa = p[i], pb = p[i + 1];
                m = seg_measure<T>(o, rr, r2, pa.x, pa.y, pb.x, pb.y, &sh.ivl[0][tid]);
            }
        }
        ordered_add<T>(sh, m, layer, acc);
    }
    if (tid == 0) a.out[path] = acc;
}

}  // namespace

cudaError_t fcpp_launch_sweep(fcpp_handle *h, const fcpp_batch &b, fcpp_sweep *d_out, cudaStream_t st)
{
    if (b.n_cand == 0) return cudaSuccess;
    SweepArgs a{};
    a.b = b;
    a.recs = h->d_rec;
    a.trig = h->d_trig;
    a.out = d_out;
    a.cap_v = b.obs_poly_start ? min(b.max_obs_verts, SW_MAX_VERTS) : 0;
    a.cap_p = b.obs_poly_start ? min(b.max_obs_polys, SW_MAX_POLYS) : 0;
    const size_t bytes = sweep_smem_bytes<TS_GEN>(sizeof(GenShared), a.cap_v, a.cap_p);
    const bool omega = b.turn_model == FCPP_TURN_OMEGA;
    cudaError_t e = cudaFuncSetAttribute(omega ? sweep_gen_omega_kernel : sweep_gen_kernel,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return e;
    if (omega)
        sweep_gen_omega_kernel<<<(unsigned)b.n_cand, TS_GEN, bytes, st>>>(a);
    else
        sweep_gen_kernel<<<(unsigned)b.n_cand, TS_GEN, bytes, st>>>(a);
    h->launches++;
    return cudaGetLastError();
}

cudaError_t fcpp_launch_sweep_paths(fcpp_handle *h, const double *d_path, const int64_t *d_offsets, int64_t n_paths,
                                    const int32_t *d_n_main, const int32_t *d_vert_start, const double *d_verts,
                                    int32_t n_polys, double radius, fcpp_sweep *d_out, cudaStream_t st)
{
    if (n_paths == 0) return cudaSuccess;
    PathSweepArgs a{};
    a.path = d_path;
    a.offsets = d_offsets;
    a.n_main = d_n_main;
    a.vert_start = d_vert_start;
    a.verts = d_verts;
    a.n_polys = n_polys;
    a.radius = radius;
    a.out = d_out;
    const size_t bytes = sweep_smem_bytes<TS_PATH>(sizeof(SweepShared<TS_PATH>), SW_MAX_VERTS, SW_MAX_POLYS);
    cudaError_t e = cudaFuncSetAttribute(sweep_path_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return e;
    sweep_path_kernel<<<(unsigned)n_paths, TS_PATH, bytes, st>>>(a);
    h->launches++;
    return cudaGetLastError();
}
