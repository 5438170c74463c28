// fcpp_cover.cu — coverage rasterisation: the W/2 round buffer of a polyline is scatter-written
// (atomicOr) into a 1-bit occupancy grid held in SHARED MEMORY tiles and popcounted; the grid
// never touches HBM.  One CTA per candidate plan.
//
// Reference code replaced ("mlp3" = multi_layer_planner_v3.py):
//   A10 corner-grid verification   mlp3:1426-1510 (per corner) and :1512-1578 (four corners)
//   A11 headland coverage rate     mlp3:1357-1371, recast as integer cell counts (north_star)
//
// Decision D5 (DESIGN.md): all coordinates are snapped to the 1e-4 m lattice and a lattice point
// is covered iff dist²(point, segment) < r² EXACTLY (128-bit integers).
//
// Rasteriser (v5):
//  * polyline points are stored relative to their lattice origin (int32); per segment ("entry")
//    the offset vector r*n of the capsule's tangent lines and the slope dx/dy are computed once
//    per plan and kept in shared memory;
//  * work = all (entry, grid row) pairs of the resident rows, flattened through a prefix sum:
//    lane p of item i owns pair 32*i + p, so lanes never idle on short segments;
//  * the capsule's left and right boundaries are piecewise (arc of the lower end | tangent line |
//    arc of the upper end), selected branch-free; arcs use an FP32 sqrt of an exact integer;
//  * the boundary is CERTIFIED: only when it falls within 5e-6 m of a lattice point is that point
//    decided by the exact integer predicate, so the counts equal the per-cell brute force of
//    oracle/raster_oracle.c bit for bit;
//  * every grid row has up to two windows of band cells ([field_lo, main_lo) and (main_hi,
//    field_hi]); only their words are stored, zeroed, written and counted.
#include "fcpp_internal.cuh"
#ifdef FCPP_COVER_DEBUG
#include <cstdio>
#endif

namespace {

constexpr int T = FCPP_COVER_THREADS;
constexpr int NWARP = T / 32;
#ifndef FCPP_COVER_TW
#define FCPP_COVER_TW 8192
#define FCPP_COVER_ROWCAP 1024
#define FCPP_COVER_VPOLY 192
#define FCPP_COVER_MINBLOCKS 2
#endif
constexpr int TW = FCPP_COVER_TW;          // occupancy tile, 32-bit words (32 KB)
constexpr int ROWCAP = FCPP_COVER_ROWCAP;  // grid rows per tile (a multiple of T)
constexpr int VPOLY_CAP = FCPP_COVER_VPOLY;  // verification polyline (15-pt arc + reverse fill), per corner
static_assert(ROWCAP % T == 0, "row windows are computed ROWCAP / T rows per thread");
constexpr int ICAP = 1024;      // item -> active-entry table
constexpr int EPT = 2;          // entries per thread in a scheduling batch
constexpr int EBATCH = EPT * T; // entries per scheduling batch
constexpr int RECT_CAP = 64;    // vertical-chain rectangles per polyline (more: the chain stays one capsule)
// capsule boundaries: certification margin in lattice units (1e-4 m) = 0.03 + 3e-6 r.  The FP64
// tangent lines are good to 2e-7 units; the arcs use an approximate FP32 sqrt of an exact integer
// (relative error < 5e-7, i.e. < 5e-7 r units): at r = 1.6 m the margin is 0.078 units = 7.8e-6 m.
constexpr double AMBIG_BASE = 0.03, AMBIG_REL = 3e-6;
constexpr double AMBIG_Q = 1e-5;      // quad row intervals: margin in cells

struct Target {
    int j0, nrows;  // lattice rows [j0, j0 + nrows) are resident
    int koff;       // tile-row index of lattice row j0
};

struct CoverFixed {
    CandRec rec;
    TrigTables tt;
    uint32_t tile[TW];
    int4 rwin[ROWCAP];   // per tile row: window 1 cells [x, y], window 2 cells [z, w] (empty: lo > hi)
    int2 rbias[ROWCAP];  // per tile row: tile word index of cell i in window w = bias.w + (i >> 5)
    int scan[32];
    double qedge[2][4][3];  // field / main quad edges: ax, ay, k = ex/ey (relative coordinates)
    int4 qtype[2][4];       // per edge: x = +1 upper bound / -1 lower bound / 0 horizontal, y = ay, z = sign(ex)
    int2 fq[4], mq[4];      // snapped field quad and R-inset, relative to the band lattice origin
    Target tg[4];
    int nrows, total_words;
    int next_w0;
    double rconst[2];  // raster_entries: r^2 and the certification margin in cells
    int cnt[8];
    unsigned long long acc[2];
    uint64_t bar;
    int4 rects[RECT_CAP];  // axis-aligned chains: lattice columns [x, y] on lattice rows [z, w] (see setup_entries)
    int nrect;
    // zoned band evaluation (see band_zoned): boxes around the general entries, one per field quadrant
    int4 zbox[4];      // lattice columns [x, y], rows [z, w]; empty: x > y
    int ztarget[4];    // zone -> target index of the current pass, -1 = not resident
    int4 zt[4];        // per target of the current pass: zone, first tile word, words per row, unused
};

// Dynamic part, behind CoverFixed in the same dynamic shared-memory allocation: the scheduling
// tables (fixed size) and one 48-byte record per polyline segment ("entry"; capacity pc >= longest
// polyline staged).  Everything is addressed from the extern shared array itself, i.e. with
// compile-time offsets: no pointer lives in a register (a struct of eight pointers handed to the
// rasteriser by reference ended up in LOCAL memory and cost eight L1-missing loads per item).
struct Entry {
    int4 seg;     // pts[e] -> pts[e+1] with the lower end first: ax, ay, bx, by
    double2 og;   // (ox, oy) = r*(dy, dx)/len; oy = +inf if dy == 0
    double kk;    // dx/dy
    int2 erow;    // staging: the snapped point e relative to its lattice origin; per raster pass: first
                  // resident lattice row of the entry, its tile row (the points are dead by then)
};
static_assert(sizeof(Entry) == 48, "Entry layout");

extern __shared__ __align__(16) unsigned char cover_smem[];

__host__ __device__ constexpr size_t a16(size_t x) { return (x + 15) & ~size_t(15); }
constexpr size_t OFF_APRE = a16(sizeof(CoverFixed));                 // int [EBATCH + 16]: exclusive (entry,row)-pair
                                                                     // prefix over the ACTIVE entries
constexpr size_t OFF_ACT = OFF_APRE + sizeof(int) * (EBATCH + 16);   // uint16 [EBATCH]: active entries (batch-local)
constexpr size_t OFF_ITEM = OFF_ACT + sizeof(uint16_t) * EBATCH;     // uint16 [ICAP]: active index holding an item's first pair
constexpr size_t OFF_ENT = a16(OFF_ITEM + sizeof(uint16_t) * ICAP);  // Entry [pc]
struct CoverDyn {
    __device__ __forceinline__ Entry &ent(int e) const
    {
        FCPP_ASSERT(e >= 0 && OFF_ENT + (size_t)(e + 1) * sizeof(Entry) <= fcpp_dynamic_smem_bytes());
        return reinterpret_cast<Entry *>(cover_smem + OFF_ENT)[e];
    }
    __device__ __forceinline__ int *apre() const { return reinterpret_cast<int *>(cover_smem + OFF_APRE); }
    __device__ __forceinline__ uint16_t *act() const { return reinterpret_cast<uint16_t *>(cover_smem + OFF_ACT); }
    __device__ __forceinline__ uint16_t *item_first() const { return reinterpret_cast<uint16_t *>(cover_smem + OFF_ITEM); }
};
__host__ __device__ inline size_t cover_smem_bytes(int pc) { return OFF_ENT + (size_t)pc * sizeof(Entry); }

// exact floor(a / H) for |a| < 2^31, 0 < H < 2^20 through FP64 + integer correction
__device__ __forceinline__ int floor_div_i(int a, int H, double invH)
{
    int q = __double2int_rd((double)a * invH);
    const int rem = a - q * H;
    if (rem < 0) --q;
    if (rem >= H) ++q;
    return q;
}
__device__ __forceinline__ int64_t floor_div64(int64_t a, int64_t b)  // b > 0
{
    int64_t q = a / b;
    if ((a % b != 0) && (a < 0)) --q;
    return q;
}
__device__ __forceinline__ int64_t ceil_div64(int64_t a, int64_t b) { return -floor_div64(-a, b); }

// exact: dist²((px,py), segment a-b) < r2 (oracle/raster_oracle.c near_segment); coordinates may be
// relative to any common origin
__device__ __noinline__ bool near_seg(int64_t px, int64_t py, int64_t ax, int64_t ay, int64_t bx, int64_t by,
                                      int64_t r2)
{
    const int64_t dx = bx - ax, dy = by - ay;
    const int64_t wx = px - ax, wy = py - ay;
    const int64_t t = wx * dx + wy * dy;
    const int64_t dd = dx * dx + dy * dy;
    if (t <= 0) return wx * wx + wy * wy < r2;
    if (t >= dd) {
        const int64_t ux = px - bx, uy = py - by;
        return ux * ux + uy * uy < r2;
    }
    const int64_t cr = wx * dy - wy * dx;
    const uint64_t acr = cr < 0 ? (uint64_t)(-cr) : (uint64_t)cr;
    const uint64_t lhs_hi = __umul64hi(acr, acr), lhs_lo = acr * acr;
    const uint64_t rhs_hi = __umul64hi((uint64_t)r2, (uint64_t)dd), rhs_lo = (uint64_t)r2 * (uint64_t)dd;
    return lhs_hi < rhs_hi || (lhs_hi == rhs_hi && lhs_lo < rhs_lo);
}

// closed containment in a convex CCW quad with integer vertices
__device__ __noinline__ bool in_quad(const int2 *q, int px, int py)
{
    bool in = true;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int k1 = (k + 1) & 3;
        const int64_t cr = (int64_t)(q[k1].x - q[k].x) * (py - q[k].y) - (int64_t)(q[k1].y - q[k].y) * (px - q[k].x);
        in = in && (cr >= 0);
    }
    return in;
}

// per-edge constants of a convex quad for the row-interval evaluation
__device__ void quad_edges_setup(const int2 *q, double (*e)[3], int4 *ty, int k)
{
    const int k1 = (k + 1) & 3;
    const int exi = q[k1].x - q[k].x, eyi = q[k1].y - q[k].y;
    const double ex = (double)exi, ey = (double)eyi;
    e[k][0] = (double)q[k].x;
    e[k][1] = (double)q[k].y;
    e[k][2] = (ey != 0.0) ? ex / ey : 0.0;
    ty[k] = make_int4(eyi > 0 ? 1 : (eyi < 0 ? -1 : 0), q[k].y, exi > 0 ? 1 : (exi < 0 ? -1 : 0), 0);
}

// inclusive lattice-index interval [a, b] of row cy (relative) inside the CLOSED convex quad
// (empty: a > b).  Every edge is a half-plane bound for every row (convexity): edges going up
// bound x from above, edges going down from below, horizontal edges decide emptiness.  FP64
// boundary + exact test of a lattice point only when the boundary is within AMBIG_Q of it.
__device__ __forceinline__ void quad_row_interval(const int2 *q, const double (*e)[3], const int4 *ty, int cy, int H,
                                                  double invH, int nx, int &a, int &b)
{
    double lo = -1e300, hi = 1e300;
    bool empty = false;
    const double y = (double)cy;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int4 t = ty[k];
        const double x = e[k][0] + e[k][2] * (y - e[k][1]);
        if (t.x > 0)
            hi = (x < hi) ? x : hi;
        else if (t.x < 0)
            lo = (x > lo) ? x : lo;
        else if (t.z * (cy - t.y) < 0)
            empty = true;
    }
    a = 0;
    b = -1;
    if (empty || !(lo <= hi + 2.0)) return;
    // |lo|, |hi| < 2^31 here (they bound a non-empty row of a quad whose coordinates fit 2^30)
    const double tl = lo * invH, th = hi * invH;
    const int rl = __double2int_rn(tl), rh = __double2int_rn(th);
    const double dl = tl - (double)rl, dh = th - (double)rh;
    int ia = rl + (dl > 0.0 ? 1 : 0);  // closed: smallest i >= tl
    int ib = rh - (dh < 0.0 ? 1 : 0);  //         largest  i <= th
    if (fabs(dl) < AMBIG_Q) ia = in_quad(q, rl * H, cy) ? rl : rl + 1;
    if (fabs(dh) < AMBIG_Q) ib = in_quad(q, rh * H, cy) ? rh : rh - 1;
    ia = max(ia, 0);
    ib = min(ib, nx - 1);
    if (ia > ib) return;
    a = ia;
    b = ib;
}

__device__ __forceinline__ void or_span(uint32_t *base, int ia, int ib)
{
    const int w0 = ia >> 5, w1 = ib >> 5;
#ifdef FCPP_BOUNDS_DEBUG
    {
        const uint32_t *tile = reinterpret_cast<const CoverFixed *>(cover_smem)->tile;
        FCPP_ASSERT(ia >= 0 && ib >= ia && base + w0 >= tile && base + w1 < tile + TW);
    }
#endif
    const uint32_t m0 = 0xffffffffu << (ia & 31), m1 = 0xffffffffu >> (31 - (ib & 31));
    if (w0 == w1) {
        atomicOr(base + w0, m0 & m1);
    } else {
        atomicOr(base + w0, m0);
        // interior words: a plain store of all-ones is a benign race with the atomics of other
        // lanes (whatever they OR in is a subset)
        for (int w = w0 + 1; w < w1; ++w) base[w] = 0xffffffffu;
        atomicOr(base + w1, m1);
    }
}

// block-wide inclusive scan of N ints per thread (entries N*tid .. N*tid+N-1); returns the total
template <int N>
__device__ int block_scan(int (&v)[N], int *sh /*[T]*/)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int q = 1; q < N; ++q) v[q] += v[q - 1];
    int inc = v[N - 1];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += o;
    }
    __syncthreads();
    if (lane == 31) sh[warp] = inc;
    __syncthreads();
    // the NWARP warp totals: one per lane, prefix by shuffles
    int wt = (lane < NWARP) ? sh[lane] : 0, wi = wt;
#pragma unroll
    for (int d = 1; d < NWARP; d <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, wi, d);
        if (lane >= d) wi += o;
    }
    const int total = __shfl_sync(0xffffffffu, wi, NWARP - 1);
    const int woff = __shfl_sync(0xffffffffu, wi - wt, warp);
    const int off = woff + inc - v[N - 1];
#pragma unroll
    for (int q = 0; q < N; ++q) v[q] += off;
    return total;
}

__device__ __forceinline__ float sqrt_approx(float x)
{
    float y;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// direction class of an exactly axis-aligned, non-degenerate segment: 1 +x, 2 -x, 3 +y, 4 -y; 0 otherwise
__device__ __forceinline__ int axis_class(int2 p, int2 q)
{
    const int dx = q.x - p.x, dy = q.y - p.y;
    if (dy == 0 && dx != 0) return dx > 0 ? 1 : 2;
    if (dx == 0 && dy != 0) return dy > 0 ? 3 : 4;
    return 0;
}

// segment records of entries [e0, e0 + n): lower end first, tangent offsets and slope; once per polyline.
// MERGE: consecutive segments that run in the same direction along one axis-aligned line (the
// 20-point straights of an unrotated rectangular field) are collapsed into their first entry — the
// union of capsules along one straight line IS the capsule of the whole chain, exactly — and the
// other entries of the chain get an empty row range.
// RECT (band only): an axis-aligned chain of >= 2 entries is split, again exactly, into the two end
// discs (point segments in the chain's first two entries) and the rectangle between them, which
// needs no per-row geometry at all: for a vertical chain the covered columns on the lattice rows
// ay <= cy <= by are |i H - x| < r (a horizontal chain likewise with rows and columns swapped), four
// integers per chain.  The rectangles go to s.rects; they are filled by fill_rects, one row per
// thread, outside the (entry, row) pair scheduler, or counted without any bitmap (band_zoned).
__device__ __forceinline__ void write_entry(const CoverDyn &d, int e, int2 p, int2 q, double rd)
{
    if (q.y < p.y || (q.y == p.y && q.x < p.x)) {
        const int2 t = p;
        p = q;
        q = t;
    }
    d.ent(e).seg = make_int4(p.x, p.y, q.x, q.y);
    const double dx = (double)(q.x - p.x), dy = (double)(q.y - p.y);
    if (dy == 0.0) {  // horizontal segment or point: the general formula with oy = +inf
        d.ent(e).og = make_double2(0.0, INFINITY);
        d.ent(e).kk = 0.0;
    } else {
        const double len = sqrt(dx * dx + dy * dy);
        d.ent(e).og = make_double2(rd * dy / len, rd * dx / len);
        d.ent(e).kk = dx / dy;
    }
}
__device__ __forceinline__ void write_dead_entry(const CoverDyn &d, int e)
{
    d.ent(e).seg = make_int4(0, 1 << 30, 0, -(1 << 30));
    d.ent(e).og = make_double2(0.0, INFINITY);
    d.ent(e).kk = 0.0;
}

template <bool MERGE, bool RECT>
__device__ void setup_entries(CoverFixed &s, const CoverDyn &d, int e0, int n, double rd, int r, int H, double invH)
{
    for (int e = e0 + threadIdx.x; e < e0 + n; e += T) {
        const int2 p = d.ent(e).erow;
        int2 q = d.ent(e + 1).erow;
        if (MERGE) {
            const int c = axis_class(p, q);
            if (c) {
                if (e > e0 && axis_class(d.ent(e - 1).erow, p) == c) {  // inside a chain
                    // the chain's second entry is written by the thread of its first (RECT)
                    const bool second = !(e - 1 > e0 && axis_class(d.ent(e - 2).erow, d.ent(e - 1).erow) == c);
                    if (!(RECT && second)) write_dead_entry(d, e);
                    continue;
                }
                int j = e + 1;
                while (j < e0 + n && axis_class(d.ent(j).erow, d.ent(j + 1).erow) == c) ++j;
                q = d.ent(j).erow;
                if (RECT && j > e + 1) {
                    int slot = atomicAdd(&s.nrect, 1);
                    if (slot >= RECT_CAP) slot = -1;  // (the counter is clamped by the readers)
                    if (slot >= 0) {
                        if (c >= 3) {  // vertical: columns |i H - x| < r on the rows ylo <= j H <= yhi
                            const int ylo = min(p.y, q.y), yhi = max(p.y, q.y);
                            s.rects[slot] = make_int4(floor_div_i(p.x - r, H, invH) + 1, -floor_div_i(-(p.x + r), H, invH) - 1,
                                                      -floor_div_i(-ylo, H, invH), floor_div_i(yhi, H, invH));
                            write_entry(d, e, make_int2(p.x, ylo), make_int2(p.x, ylo), rd);
                            write_entry(d, e + 1, make_int2(p.x, yhi), make_int2(p.x, yhi), rd);
                        } else {  // horizontal: rows |j H - y| < r on the columns xlo <= i H <= xhi
                            const int xlo = min(p.x, q.x), xhi = max(p.x, q.x);
                            s.rects[slot] = make_int4(-floor_div_i(-xlo, H, invH), floor_div_i(xhi, H, invH),
                                                      floor_div_i(p.y - r, H, invH) + 1, -floor_div_i(-(p.y + r), H, invH) - 1);
                            write_entry(d, e, make_int2(xlo, p.y), make_int2(xlo, p.y), rd);
                            write_entry(d, e + 1, make_int2(xhi, p.y), make_int2(xhi, p.y), rd);
                        }
                        continue;
                    }
                    write_dead_entry(d, e + 1);
                }
            }
        }
        write_entry(d, e, p, q, rd);
    }
}

// the rectangles of the axis-aligned chains on the resident rows [j0, j0 + nrows), which start at
// tile row koff: one row per thread (columns are clipped by the row's windows)
__device__ void fill_rects(CoverFixed &s, int j0, int nrows, int koff)
{
    const int nr = min(s.nrect, RECT_CAP);
    for (int k = threadIdx.x; k < nrows; k += T) {
        const int j = j0 + k;
        const int4 w = s.rwin[k + koff];
        const int2 bias = s.rbias[k + koff];
        if (w.x > w.y && w.z > w.w) continue;
        for (int q = 0; q < nr; ++q) {
            const int4 rc = s.rects[q];
            if (j < rc.z || j > rc.w) continue;
            const int s1 = max(rc.x, w.x), e1 = min(rc.y, w.y);
            if (s1 <= e1) or_span(s.tile + bias.x, s1, e1);
            const int s2 = max(rc.x, w.z), e2 = min(rc.y, w.w);
            if (s2 <= e2) or_span(s.tile + bias.y, s2, e2);
        }
    }
}

// Rasterise the segments ("entries") e0 .. e0+n_ent-1 (entries that join two different polylines
// are masked by `tgt(e) < 0`) into the resident tile rows of their targets.  All targets of one
// call share the lattice pitch H.  Must be called after a __syncthreads() that follows
// setup_entries (the staging points are overwritten by the per-pass row records).
template <class TgFn>
__device__ void raster_entries(CoverFixed &s, const CoverDyn &d, int e0, int n_ent, TgFn tgt, int r, int H,
                               double invH)
{
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t r2 = (int64_t)r * r;
    // loop constants live in shared memory: under the 64-register cap the compiler would otherwise
    // re-derive them (an int->double conversion and five FP64 operations) for every item
    if (tid == 0) {
        s.rconst[0] = (double)r * (double)r;
        s.rconst[1] = (AMBIG_BASE + AMBIG_REL * (double)r) * invH;
    }
    for (int eb = 0; eb < n_ent; eb += EBATCH) {
        const int nb = min(EBATCH, n_ent - eb);
        // ---- resident rows each entry's capsule can touch; packed (active << 21 | rows) ----
        int rows[EPT], inc[EPT];
#pragma unroll
        for (int q = 0; q < EPT; ++q) {
            const int le = q * T + tid;  // interleaved: the entries of a short polyline spread over all warps
            rows[q] = 0;
            if (le < nb) {
                const int e = e0 + eb + le;
                const int ti = tgt(e);
                if (ti >= 0) {
                    const int4 sg = d.ent(e).seg;
                    const Target t = s.tg[ti];
                    int jlo = floor_div_i(sg.y - r, H, invH) + 1;      // cy > ymin - r
                    int jhi = -floor_div_i(-(sg.w + r), H, invH) - 1;  // cy < ymax + r
                    jlo = max(jlo, t.j0);
                    jhi = min(jhi, t.j0 + t.nrows - 1);
                    if (jhi >= jlo) rows[q] = jhi - jlo + 1;
                    d.ent(e).erow = make_int2(jlo, jlo - t.j0 + t.koff);
                }
            }
            inc[q] = rows[q] ? ((1 << 21) | rows[q]) : 0;
        }
        const unsigned tot = (unsigned)block_scan<EPT>(inc, s.scan);
        const int n_act = (int)(tot >> 21), n_pairs = (int)(tot & 0x1fffffu);
        const int n_items = (n_pairs + 31) >> 5;
        const bool table = n_items <= ICAP;
#pragma unroll
        for (int q = 0; q < EPT; ++q) {
            if (rows[q]) {
                const int ai = (int)((unsigned)inc[q] >> 21) - 1;
                const int first = (int)((unsigned)inc[q] & 0x1fffffu) - rows[q];
                FCPP_ASSERT(ai >= 0 && ai < EBATCH && first >= 0);
                d.act()[ai] = (uint16_t)(q * T + tid);
                d.apre()[ai] = first;
                if (table)
                    for (int i = (first + 31) >> 5; i <= (first + rows[q] - 1) >> 5; ++i) {
                        FCPP_ASSERT(i >= 0 && i < ICAP);
                        d.item_first()[i] = (uint16_t)ai;
                    }
            }
        }
        FCPP_ASSERT(n_act >= 0 && n_act <= EBATCH);
        if (tid == 0) d.apre()[n_act] = n_pairs;
        __syncthreads();
        // items go to the warps round-robin (handing them out through a shared counter was measured
        // twice and lost 2.5-4.5 %: the atomic sits on every item's critical path)
        for (int item = warp; item < n_items;) {
            const int pbase = 32 * item;
            const int next_item = item + NWARP;
            // ---- pair -> active entry: the entry boundaries inside this item as a bit mask ----
            int base_ai;
            if (table) {
                base_ai = d.item_first()[item];
            } else {  // upper_bound over the pair prefix (one lane), then broadcast
                int lo = 0;
                if (lane == 0) {
                    int hi = n_act - 1;
                    while (lo < hi) {
                        const int mid = (lo + hi + 1) >> 1;
                        if (d.apre()[mid] <= pbase)
                            lo = mid;
                        else
                            hi = mid - 1;
                    }
                }
                base_ai = __shfl_sync(0xffffffffu, lo, 0);
            }
            const int bidx = base_ai + 1 + lane;
            const int bnd = (bidx <= n_act) ? d.apre()[bidx] : 0x7fffffff;  // > pbase: entry base_ai holds pair pbase
            const unsigned mbit = (bnd < pbase + 32) ? (1u << ((bnd - pbase) & 31)) : 0u;
            const unsigned bmask = __reduce_or_sync(0xffffffffu, mbit);
            const int p = pbase + lane;
            item = next_item;
            if (p >= n_pairs) continue;
            const int ai = base_ai + __popc(bmask & ((2u << lane) - 1u));
            const int e = e0 + eb + d.act()[ai];
            const int qrow = p - d.apre()[ai];
            const int4 sg = d.ent(e).seg;
            const int2 er = d.ent(e).erow;
            const double2 og = d.ent(e).og;
            const double kk = d.ent(e).kk;
            const int k = er.y + qrow;
            const int cy = (er.x + qrow) * H;
            const double ax = (double)sg.x, bx = (double)sg.z;
            const double wa = (double)(cy - sg.y), wb = (double)(cy - sg.w);
            // half chords of the end discs: approximate FP32 sqrt of an exact integer
            const double r2d = s.rconst[0], amb = s.rconst[1];
            const double hA = (double)sqrt_approx(fmaxf((float)(r2d - wa * wa), 0.0f));
            const double hB = (double)sqrt_approx(fmaxf((float)(r2d - wb * wb), 0.0f));
            // left: arc A below yL0 = ay+oy | tangent line up to yL1 = by+oy | arc B;  right: -oy
            const double xl = (wa < og.y) ? ax - hA : ((wb <= og.y) ? (ax - og.x) + (wa - og.y) * kk : bx - hB);
            const double xr = (wa < -og.y) ? ax + hA : ((wb <= -og.y) ? (ax + og.x) + (wa + og.y) * kk : bx + hB);
            // lattice indices strictly inside (xl, xr); |xl|, |xr| < 2^31.  Certified: an end within
            // `amb` of a lattice point is decided by the exact integer predicate
            const double tl = xl * invH, th = xr * invH;
            const int rl = __double2int_rn(tl), rh = __double2int_rn(th);
            const double dl = tl - (double)rl, dh = th - (double)rh;
            int ia = rl + (dl >= 0.0 ? 1 : 0);  // smallest i > tl
            int ib = rh - (dh <= 0.0 ? 1 : 0);  // largest  i < th
            if (fabs(dl) < amb || fabs(dh) < amb) {
                if (fabs(dl) < amb) ia = near_seg((int64_t)rl * H, cy, sg.x, sg.y, sg.z, sg.w, r2) ? rl : rl + 1;
                if (fabs(dh) < amb) ib = near_seg((int64_t)rh * H, cy, sg.x, sg.y, sg.z, sg.w, r2) ? rh : rh - 1;
            }
            const int4 w = s.rwin[k];
            const int2 bias = s.rbias[k];
            const int s1 = max(ia, w.x), e1 = min(ib, w.y);
            if (s1 <= e1) or_span(s.tile + bias.x, s1, e1);
            const int s2 = max(ia, w.z), e2 = min(ib, w.w);
            if (s2 <= e2) or_span(s.tile + bias.y, s2, e2);
        }
        __syncthreads();
    }
}

// popcount of n words starting at a 16-byte aligned address (the words up to the next multiple
// of 4 are read too: callers keep them zero)
__device__ __forceinline__ int count_words(const uint32_t *w, int n)
{
    FCPP_ASSERT(n >= 0 && w >= reinterpret_cast<const CoverFixed *>(cover_smem)->tile &&
                w + ((n + 3) & ~3) <= reinterpret_cast<const CoverFixed *>(cover_smem)->tile + TW);
    int c = 0;
    const uint4 *v = reinterpret_cast<const uint4 *>(w);
    for (int i = threadIdx.x; i < (n + 3) >> 2; i += T) {
        const uint4 x = v[i];
        c += __popc(x.x) + __popc(x.y) + __popc(x.z) + __popc(x.w);
    }
    return c;
}
__device__ __forceinline__ void zero_words(uint32_t *w, int n)  // rounds n up to a multiple of 4
{
    FCPP_ASSERT(n >= 0 && w >= reinterpret_cast<const CoverFixed *>(cover_smem)->tile &&
                w + ((n + 3) & ~3) <= reinterpret_cast<const CoverFixed *>(cover_smem)->tile + TW);
    uint4 *v = reinterpret_cast<uint4 *>(w);
    for (int i = threadIdx.x; i < (n + 3) >> 2; i += T) v[i] = make_uint4(0u, 0u, 0u, 0u);
}

__device__ __forceinline__ int words_of(int lo, int hi) { return hi >= lo ? (hi >> 5) - (lo >> 5) + 1 : 0; }

// lattice-index intervals of row cy inside the closed field quad [x, y] and the closed R-inset
// [z, w] (empty: lo > hi, normalised to (0, -1))
__device__ __forceinline__ int4 band_row_raw(const CoverFixed &s, int cy, int H, double invH, int nx)
{
    int4 v;
    quad_row_interval(s.fq, s.qedge[0], s.qtype[0], cy, H, invH, nx, v.x, v.y);
    quad_row_interval(s.mq, s.qedge[1], s.qtype[1], cy, H, invH, nx, v.z, v.w);
    return v;
}
// band cells of a row: window 1 = [x, y], window 2 = [z, w] (empty: lo > hi) — the cells whose
// centre lies in the closed field quad and not in the closed R-inset
__device__ __forceinline__ int4 band_windows_of(int4 v)
{
    int4 win = make_int4(1, 0, 1, 0);
    if (v.x <= v.y) {
        if (v.z <= v.w) {  // the inset lies inside the field: clamp defensively
            const int ma = max(v.z, v.x), mb = min(v.w, v.y);
            win = make_int4(v.x, ma - 1, mb + 1, v.y);
        } else {
            win = make_int4(v.x, v.y, 1, 0);
        }
    }
    return win;
}
__device__ __forceinline__ int4 band_row_windows(const CoverFixed &s, int cy, int H, double invH, int nx)
{
    return band_windows_of(band_row_raw(s, cy, H, invH, nx));
}

// rows [ylo, yhi] (lattice coordinates) lie entirely below or entirely above the quad
__device__ __forceinline__ bool outside_rows(const int2 *q, int ylo, int yhi)
{
    const int ymin = min(min(q[0].y, q[1].y), min(q[2].y, q[3].y));
    const int ymax = max(max(q[0].y, q[1].y), max(q[2].y, q[3].y));
    return yhi < ymin || ylo > ymax;
}

// quadrant of a live entry: by the midpoint of its segment against the middle of the lattice
__device__ __forceinline__ int seg_quadrant(const int4 sg, int midx2, int midy2)
{
    return ((sg.y + sg.w) >= midy2 ? 2 : 0) | ((sg.x + sg.z) >= midx2 ? 1 : 0);
}

// number of lattice columns of [a, b] on row j covered by the chain rectangles (sorted by their
// first column): the classic sweep over sorted intervals
__device__ __forceinline__ int rect_cover(const CoverFixed &s, int nr, int j, int a, int b)
{
    int cur = a - 1, len = 0;
    for (int q = 0; q < nr; ++q) {
        const int4 rc = s.rects[q];
        if (rc.x > b) break;
        if (j < rc.z || j > rc.w) continue;
        const int lo = max(rc.x, cur + 1), hi = min(rc.y, b);
        if (lo <= hi) {
            len += hi - lo + 1;
            cur = hi;
        }
    }
    return len;
}

// Zoned evaluation of the headland band for fields whose straights are axis-aligned chains.
// Everything that is not a chain rectangle (turn arcs, reverse fills, the joins between loops, the
// end discs of the chains) sits near the field's corners: these "general" entries are boxed per
// field quadrant into at most four ZONES, and only the zones get a bitmap (rectangles + general
// entries, a few thousand words in total instead of the whole band).  Outside the zones a band
// cell can only be covered by a rectangle, so each row is counted in closed form:
//     covered(row) = |U ∩ W| - Σ_zones |U ∩ W ∩ Z|   (U = union of the rectangles' column intervals,
// W = the row's band windows, Z = the zones' column intervals; the zones are pairwise disjoint).
// Returns false (nothing counted) when the zones overlap or are too large; the caller then runs
// the row-tiled evaluation of the whole band.
__device__ __noinline__ bool band_zoned(CoverFixed &s, const CoverDyn &d, int n_ent, int rq, int H, double invH, int nx, int ny,
                           unsigned long long &my_total, unsigned long long &my_cov)
{
    const int tid = threadIdx.x;
    const int nr = min(s.nrect, RECT_CAP);
    const int midx2 = (nx - 1) * H, midy2 = (ny - 1) * H;
    // ---- sort the rectangles by first column (rank by counting), box the general entries ----
    int4 mine = make_int4(0, 0, 0, 0);
    int rank = 0;
    if (tid < nr) {
        mine = s.rects[tid];
        for (int q = 0; q < nr; ++q) {
            const int x = s.rects[q].x;
            rank += (x < mine.x || (x == mine.x && q < tid)) ? 1 : 0;
        }
    }
    if (tid < 4) s.zbox[tid] = make_int4(INT_MAX, INT_MIN, INT_MAX, INT_MIN);
    __syncthreads();
    if (tid < nr) s.rects[rank] = mine;
    for (int e = tid; e < n_ent; e += T) {
        const int4 sg = d.ent(e).seg;
        if (sg.y > sg.w) continue;  // dead entry of a chain
        const int jlo = max(floor_div_i(sg.y - rq, H, invH) + 1, 0);
        const int jhi = min(-floor_div_i(-(sg.w + rq), H, invH) - 1, ny - 1);
        const int cl = max(floor_div_i(min(sg.x, sg.z) - rq, H, invH), 0);
        const int ch = min(-floor_div_i(-(max(sg.x, sg.z) + rq), H, invH), nx - 1);
        if (jlo > jhi || cl > ch) continue;  // cannot touch the lattice
        int4 *zb = &s.zbox[seg_quadrant(sg, midx2, midy2)];
        atomicMin(&zb->x, cl);
        atomicMax(&zb->y, ch);
        atomicMin(&zb->z, jlo);
        atomicMax(&zb->w, jhi);
    }
    __syncthreads();
    // ---- the zones must be pairwise disjoint and small (uniform decision) ----
    {
        bool okz = true;
        long long words = 0;
        for (int z = 0; z < 4; ++z) {
            const int4 a = s.zbox[z];
            if (a.x > a.y) continue;
            const int rw = (a.y >> 5) - (a.x >> 5) + 1;
            words += (long long)rw * (a.w - a.z + 1);
            if (rw > TW - 16) okz = false;
            for (int y = z + 1; y < 4; ++y) {
                const int4 c = s.zbox[y];
                if (c.x <= c.y && a.x <= c.y && c.x <= a.y && a.z <= c.w && c.z <= a.w) okz = false;
            }
        }
        if (words > 12ll * TW) okz = false;
#ifdef FCPP_COVER_DEBUG
        if (tid == 0 && (blockIdx.x % 512) == 0) {  // (debug builds only)
            printf("cand %d nrect %d okz %d words %lld\n", (int)blockIdx.x, nr, (int)okz, words);
            for (int z = 0; z < 4; ++z) printf("  zone %d cols [%d,%d] rows [%d,%d]\n", z, s.zbox[z].x, s.zbox[z].y, s.zbox[z].z, s.zbox[z].w);
        }
#endif
        if (!okz) return false;
    }

    // ---- bitmap passes over the zones: whole zones are packed into one tile while they fit, a
    // zone larger than the tile is cut into row ranges (every thread derives the same packing) ----
    int z = 0, zrow = 0;
    while (true) {
        int nt = 0, used_w = 0, used_r = 0;
        __syncthreads();  // the previous pass is done with s.tg / s.zt / s.ztarget
        if (tid < 4) s.ztarget[tid] = -1;
        __syncthreads();
        while (z < 4 && nt < 4) {
            const int4 box = s.zbox[z];
            if (box.x > box.y) {
                ++z;
                zrow = 0;
                continue;
            }
            const int rw = (box.y >> 5) - (box.x >> 5) + 1;
            const int zrows = box.w - box.z + 1;
            const int n = min(zrows - zrow, min((TW - used_w) / rw, ROWCAP - used_r));
            if (n <= 0) break;
            if (tid == 0) {
                Target &t = s.tg[nt];
                t.j0 = box.z + zrow;
                t.nrows = n;
                t.koff = used_r;
                s.zt[nt] = make_int4(z, used_w, rw, 0);
                s.ztarget[z] = nt;
            }
            used_w += (n * rw + 3) & ~3;
            used_r += n;
            ++nt;
            zrow += n;
            if (zrow < zrows) break;  // a cut zone ends the pass
            ++z;
            zrow = 0;
        }
        if (nt == 0) break;
        __syncthreads();
        // row windows of the resident rows, clipped to their zone's columns
        for (int k = tid; k < used_r; k += T) {
            int t = 0;
            while (t + 1 < nt && k >= s.tg[t + 1].koff) ++t;
            const Target tg = s.tg[t];
            const int4 zt = s.zt[t];
            const int4 box = s.zbox[zt.x];
            int4 win = band_row_windows(s, (tg.j0 + (k - tg.koff)) * H, H, invH, nx);
            win.x = max(win.x, box.x);
            win.y = min(win.y, box.y);
            win.z = max(win.z, box.x);
            win.w = min(win.w, box.y);
            const int base = zt.y + (k - tg.koff) * zt.z - (box.x >> 5);
            s.rwin[k] = win;
            s.rbias[k] = make_int2(base, base);
        }
        zero_words(s.tile, used_w);
        __syncthreads();
        for (int t = 0; t < nt; ++t) fill_rects(s, s.tg[t].j0, s.tg[t].nrows, s.tg[t].koff);
        {
            auto tgt = [&](int e) {
                const int4 sg = d.ent(e).seg;
                return (sg.y > sg.w) ? -1 : s.ztarget[seg_quadrant(sg, midx2, midy2)];
            };
            raster_entries(s, d, 0, n_ent, tgt, rq, H, invH);
        }
        my_cov += (unsigned long long)count_words(s.tile, used_w);
    }
    // ---- every row in closed form: band cells, rectangle cover outside the zones.  Rows are
    // grouped into runs between BREAKPOINTS (rows where a rectangle or a zone starts or ends, and
    // the rows of the quads' vertices): inside a run the rectangles and zones are the same and each
    // of the four window boundaries follows ONE quad edge, i.e. is monotone in the row — if it has
    // the same lattice index on the first and the last row of the run it has it on every row, and
    // the run is counted once and multiplied.  Runs with slanted boundaries go row by row. ----
    __syncthreads();  // the last pass is done with the tile: reuse it for the breakpoints
    int *bp = reinterpret_cast<int *>(s.tile);  // [nb] sorted breakpoints, then [nb] slow runs (lo, hi)
    const int nb = 10 + 2 * nr + 8;
    static_assert(T >= 2 * (10 + 2 * RECT_CAP + 8), "one thread per (run, end)");
    static_assert(12 * (10 + 2 * RECT_CAP + 8) <= TW, "breakpoints, slow runs and row intervals live in the tile");
    {
        int v = -1;
        if (tid == 0) v = 0;
        else if (tid == 1) v = ny;
        else if (tid < 10) {
            const int y = (tid < 6) ? s.fq[tid - 2].y : s.mq[tid - 6].y;
            v = -floor_div_i(-y, H, invH);  // first row at or above the vertex
        } else if (tid < 10 + 2 * nr) {
            const int4 rc = s.rects[(tid - 10) >> 1];
            v = (tid & 1) ? rc.w + 1 : rc.z;
        } else if (tid < nb) {
            const int4 box = s.zbox[(tid - 10 - 2 * nr) >> 1];
            v = (box.x > box.y) ? 0 : ((tid & 1) ? box.w + 1 : box.z);
        }
        v = min(max(v, 0), ny);
        int *raw = bp + 2 * nb + 2;
        if (tid < nb) raw[tid] = v;
        __syncthreads();
        if (tid < nb) {
            int rk = 0;
            for (int q = 0; q < nb; ++q) {
                const int x = raw[q];
                rk += (x < v || (x == v && q < tid)) ? 1 : 0;
            }
            bp[rk] = v;
        }
        if (tid == 0) s.cnt[0] = 0;
        __syncthreads();
    }
    // one thread per (run, end): the raw row intervals of the run's first and last row
    int4 *rraw = reinterpret_cast<int4 *>(bp + 4 * nb);  // [2 nb], 16-byte aligned (nb is even)
    if (tid < 2 * (nb - 1)) {
        const int i = tid >> 1;
        const int lo = bp[i], hi = bp[i + 1] - 1;
        if (lo <= hi) rraw[tid] = band_row_raw(s, ((tid & 1) ? hi : lo) * H, H, invH, nx);
    }
    __syncthreads();
    // part p of a row's count: p = 0 the whole window pair, p = 1 + q what lies in zone q (subtracted)
    auto row_part = [&](int j, int4 win, int p, unsigned long long mult) {
        int4 box = make_int4(INT_MIN, INT_MAX, INT_MIN, INT_MAX);
        if (p > 0) {
            box = s.zbox[p - 1];
            if (box.x > box.y || j < box.z || j > box.w) return;
        }
        int cov = 0, cells = 0;
#pragma unroll
        for (int w = 0; w < 2; ++w) {
            const int a = max(w ? win.z : win.x, box.x), b = min(w ? win.w : win.y, box.y);
            if (a > b) continue;
            cells += b - a + 1;
            cov += rect_cover(s, nr, j, a, b);
        }
        if (p == 0) {
            my_total += mult * (unsigned long long)cells;
            my_cov += mult * (unsigned long long)cov;
        } else {
            my_cov -= mult * (unsigned long long)cov;
        }
    };
    int2 *slow = reinterpret_cast<int2 *>(bp + nb);
    for (int u = tid; u < 5 * (nb - 1); u += T) {
        const int i = u / 5, p = u - 5 * i;
        const int lo = bp[i], hi = bp[i + 1] - 1;
        if (lo > hi) continue;
        const int4 v0 = rraw[2 * i], v1 = rraw[2 * i + 1];
        bool same = v0.x == v1.x && v0.y == v1.y && v0.z == v1.z && v0.w == v1.w;
        // an EMPTY interval at both ends proves nothing about the rows between (a sliver thinner
        // than a cell) unless the whole run lies below or above the quad
        if (hi > lo && v0.x > v0.y) same = same && outside_rows(s.fq, lo * H, hi * H);
        if (hi > lo && v0.z > v0.w) same = same && outside_rows(s.mq, lo * H, hi * H);
        if (same)
            row_part(lo, band_windows_of(v0), p, (unsigned long long)(hi - lo + 1));
        else if (p == 0)
            slow[atomicAdd(&s.cnt[0], 1)] = make_int2(lo, hi);
    }
    __syncthreads();
    const int nslow = s.cnt[0];
    for (int q = 0; q < nslow; ++q) {
        const int2 run = slow[q];
        for (int j = run.x + tid; j <= run.y; j += T) {
            const int4 win = band_row_windows(s, j * H, H, invH, nx);
            for (int p = 0; p < 5; ++p) row_part(j, win, p, 1ull);
        }
    }
    __syncthreads();  // the caller may reuse the tile
    return true;
}

// One candidate's coverage by the T threads of a CTA (cover_kernel, or one listed item of cover_work_kernel).
__device__ __forceinline__ void cover_body(const fcpp_batch &b, const CandRec *__restrict__ recs,
                                           const TrigTables *__restrict__ trig, fcpp_summary *__restrict__ summary,
                                           int pc, int mode, const int32_t *__restrict__ rep /*[2][n_cand]*/,
                                           uint32_t *__restrict__ corner_bits, int64_t corner_bits_stride,
                                           const int64_t cand)
{
    // a part (A10 corner windows / A11 band) whose inputs equal those of an earlier candidate is
    // skipped: the candidate takes that one's counts afterwards (cover_copy_kernel).  A10 does not
    // depend on the start corner or the heading, A11 not on the heading.
    const bool do10 = !rep || rep[cand] == (int32_t)cand;
    const bool do11 = !rep || rep[b.n_cand + cand] == (int32_t)cand;
    if (!do10 && !do11) return;
    CoverFixed &s = *reinterpret_cast<CoverFixed *>(cover_smem);
    const CoverDyn d;
    const int tid = threadIdx.x;
    fcpp_summary *sum = summary + cand;

    if (tid == 0) mbar_init(&s.bar, 1);
    __syncthreads();
    if (tid == 0) {
        mbar_expect_tx(&s.bar, sizeof(CandRec));
        bulk_g2s(&s.rec, recs + cand, sizeof(CandRec), &s.bar);
        s.acc[0] = s.acc[1] = 0ull;
    }
    if (tid < 8) s.cnt[tid] = 0;
    for (int k = tid; k < (int)(sizeof(TrigTables) / sizeof(double)); k += T)
        ((double *)&s.tt)[k] = ((const double *)trig)[k];
    mbar_wait_block(&s.bar, 0);
    __syncthreads();
    const CandRec &r = s.rec;
    if (r.status != 0 || r.n_total == 0) {
        if (tid == 0) {
            if (do11) sum->cov_cells = sum->cov_total = 0;
            if (do10)
                for (int k = 0; k < 4; ++k) sum->corner_before[k] = sum->corner_after[k] = 0;
        }
        return;
    }
    const double W = b.vehicle.working_width;
    const int rq = (int)qfix(W / 2);
    const double rd = (double)rq;
    TurnModel tm;
    tm.model = b.turn_model;
    tm.lam = b.clothoid_share;
    int err10 = 0, err11 = 0;  // a grid that does not fit: per part (the parts may run in different CTAs)

    // =====================================================================================
    // A10: four verification corner windows (lattice POINTS, h = 0.1 m)
    // =====================================================================================
    if (do10) {
        const double fl = b.field_extent[2 * r.field], fw = b.field_extent[2 * r.field + 1];
        const int g = r.corner_g;
        const int rw = (g + 31) >> 5;
        const int Hc = (int)qfix(FCPP_CORNER_GRID_H);
        const double invHc = 1.0 / (double)Hc;
        const bool okc = (g >= 1) && (rw <= TW - 16) && (4 * VPOLY_CAP <= pc);
        if (!okc) err10 = 1;
        const int rpt = okc ? min(ROWCAP, (TW - 16) / rw) : 1;                          // rows per tile
        const int group = (okc && 4 * g <= rpt) ? 4 : ((okc && 2 * g <= rpt) ? 2 : 1);  // corners per pass
        // snapped polylines of the four corners: 15-pt arc + reverse fill (mlp3:1531-1554), relative
        // to the corner's lattice origin (mlp3:1461-1468); corner ci occupies pts[ci*VPOLY_CAP ...]
        int nv[4];
#pragma unroll
        for (int ci = 0; ci < 4; ++ci) {
            nv[ci] = min(r.vn_rev[ci], VPOLY_CAP - FCPP_CORNER_POINTS);
            if (r.vn_rev[ci] > VPOLY_CAP - FCPP_CORNER_POINTS) err10 = 1;
            if (!okc) continue;
            const double qx = (ci == 0 || ci == 3) ? r.R : fl - r.R;  // mlp3:1531-1536
            const double qy = (ci == 0 || ci == 1) ? r.R : fw - r.R;
            const int64_t X0 = qfix((ci == 0 || ci == 3) ? qx : qx - 2 * r.R);
            const int64_t Y0 = qfix((ci == 0 || ci == 1) ? qy : qy - 2 * r.R);
            for (int k = tid; k < FCPP_CORNER_POINTS + nv[ci]; k += T) {
                double x, y;
                if (k < FCPP_CORNER_POINTS) {
                    corner_arc_pt(s.tt, tm, qx, qy, r.R, ci, k, x, y);
                } else {
                    const int m = k - FCPP_CORNER_POINTS;
                    const double len = r.vrev[ci][4];
                    const double tt_ = (m == r.vn_rev[ci] - 1) ? len : m * (len / (r.vn_rev[ci] - 1));
                    x = r.vrev[ci][0] + tt_ * r.vrev[ci][2];
                    y = r.vrev[ci][1] + tt_ * r.vrev[ci][3];
                }
                d.ent(ci * VPOLY_CAP + k).erow = make_int2((int)(qfix(x) - X0), (int)(qfix(y) - Y0));
            }
        }
        __syncthreads();
        if (okc) {
#pragma unroll
            for (int ci = 0; ci < 4; ++ci) setup_entries<false, false>(s, d, ci * VPOLY_CAP, FCPP_CORNER_POINTS + nv[ci] - 1, rd, rq, Hc, invHc);
        }
        int before[4] = {0, 0, 0, 0}, after[4] = {0, 0, 0, 0};
        for (int c0 = 0; c0 < 4 && okc; c0 += group) {
            for (int j0 = 0; j0 < g; j0 += rpt) {
                const int nrows = (group > 1) ? g : min(rpt, g - j0);
                const int cstride = (nrows * rw + 3) & ~3;  // words per corner, 16-byte aligned
                if (tid < group) {
                    Target &t = s.tg[tid];
                    t.j0 = j0;
                    t.nrows = nrows;
                    t.koff = tid * nrows;
                }
                for (int k = tid; k < group * nrows; k += T) {
                    const int c = k / nrows;
                    s.rwin[k] = make_int4(0, g - 1, 1, 0);
                    s.rbias[k] = make_int2(c * cstride + (k - c * nrows) * rw, 0);
                }
                zero_words(s.tile, group * cstride);
                if (tid < 8) s.cnt[tid] = 0;
                __syncthreads();
                // pass 1: the turn arcs (entries 0..13 of every corner of the group)
                {
                    auto tgt = [&](int e) {
                        const int c = e / VPOLY_CAP, k = e - c * VPOLY_CAP;
                        return (k < FCPP_CORNER_POINTS - 1 && c >= c0 && c < c0 + group) ? c - c0 : -1;
                    };
                    raster_entries(s, d, c0 * VPOLY_CAP, (group - 1) * VPOLY_CAP + FCPP_CORNER_POINTS - 1, tgt, rq, Hc,
                                   invHc);
                }
                for (int c = 0; c < group; ++c) {
                    const int n = count_words(s.tile + c * cstride, nrows * rw);
                    if (n) atomicAdd(&s.cnt[c], n);
                }
                __syncthreads();
                // pass 2: the reverse fills (entries 15 .. 15+nv-2; entry 14 joins arc and fill and
                // is NOT part of either LineString, mlp3:1471 / :1487)
                {
                    auto tgt = [&](int e) {
                        const int c = e / VPOLY_CAP, k = e - c * VPOLY_CAP;
                        return (k >= FCPP_CORNER_POINTS && k < FCPP_CORNER_POINTS + nv[c] - 1 && c >= c0 && c < c0 + group)
                                   ? c - c0
                                   : -1;
                    };
                    raster_entries(s, d, c0 * VPOLY_CAP, group * VPOLY_CAP - 1, tgt, rq, Hc, invHc);
                }
                for (int c = 0; c < group; ++c) {
                    const int n = count_words(s.tile + c * cstride, nrows * rw);
                    if (n) atomicAdd(&s.cnt[4 + c], n);
                }
                if (corner_bits && (int64_t)4 * g * rw <= corner_bits_stride) {  // the 'grid' of mlp3:1503-1510
                    uint32_t *dst = corner_bits + cand * corner_bits_stride;
                    for (int k = tid; k < group * nrows * rw; k += T) {
                        const int c = k / (nrows * rw), w = k - c * nrows * rw;
                        dst[((int64_t)(c0 + c) * g + j0) * rw + w] = s.tile[c * cstride + w];
                    }
                }
                __syncthreads();
                for (int c = 0; c < group; ++c) {
                    before[c0 + c] += s.cnt[c];
                    after[c0 + c] += s.cnt[4 + c];
                }
                __syncthreads();
                if (group > 1) break;
            }
        }
        if (tid == 0)
            for (int k = 0; k < 4; ++k) {
                sum->corner_before[k] = okc ? before[k] : 0;
                sum->corner_after[k] = okc ? after[k] : 0;
            }
    }

    // =====================================================================================
    // A11: headland band (lattice of cell CENTRES anchored at the field bbox minimum)
    // =====================================================================================
    if (do11) {
        double bx0 = 1e300, by0 = 1e300, bx1 = -1e300, by1 = -1e300;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const double x = b.field_verts[(int64_t)r.field * 8 + 2 * k];
            const double y = b.field_verts[(int64_t)r.field * 8 + 2 * k + 1];
            bx0 = fmin(bx0, x);
            by0 = fmin(by0, y);
            bx1 = fmax(bx1, x);
            by1 = fmax(by1, y);
        }
        const int64_t H64 = qfix(b.grid_h);
        const int64_t X0 = qfix(bx0), Y0 = qfix(by0);
        const int64_t nx64 = ceil_div64(qfix(bx1) - X0, H64), ny64 = ceil_div64(qfix(by1) - Y0, H64);
        const int64_t Xc0 = X0 + H64 / 2, Yc0 = Y0 + H64 / 2;  // lattice origin: centre of cell (0, 0)
        const int H = (int)H64, nx = (int)nx64, ny = (int)ny64;
        const double invH = 1.0 / (double)H;
        const int nh = r.n_head;
        // relative coordinates must fit int32 with headroom (extent + r < 2^30 units = 107 km)
        const bool ok = (nh <= pc) && nx64 > 0 && ny64 > 0 && nx64 * H64 < (1ll << 30) && ny64 * H64 < (1ll << 30) &&
                        H64 < (1 << 20);
        if (!ok) err11 = 1;
        __syncthreads();
        if (ok) {
            if (tid == 0) s.nrect = 0;
            if (tid < 4) {
                s.fq[tid] = make_int2((int)(qfix(b.field_verts[(int64_t)r.field * 8 + 2 * tid]) - Xc0),
                                      (int)(qfix(b.field_verts[(int64_t)r.field * 8 + 2 * tid + 1]) - Yc0));
                s.mq[tid] = make_int2((int)(qfix(r.main_quad[tid][0]) - Xc0), (int)(qfix(r.main_quad[tid][1]) - Yc0));
            }
            for (int k = tid; k < nh; k += T) {
                double x, y;
                uint8_t c;
                gen_point(r, s.tt, tm, W, r.n_main + k, x, y, c);
                d.ent(k).erow = make_int2((int)(qfix(x) - Xc0), (int)(qfix(y) - Yc0));
            }
            __syncthreads();
            if (tid < 4) quad_edges_setup(s.fq, s.qedge[0], s.qtype[0], tid);
            if (tid >= 4 && tid < 8) quad_edges_setup(s.mq, s.qedge[1], s.qtype[1], tid - 4);
            setup_entries<true, FCPP_COVER_RECT != 0>(s, d, 0, nh - 1, rd, rq, H, invH);
            __syncthreads();
            // entries whose whole capsule (bounding box grown by r) lies in the closed R-inset cannot
            // cover a band cell — the inner ends of the inner loops' turn arcs, most of the joins
            for (int e = tid; e < nh - 1; e += T) {
                const int4 sg = d.ent(e).seg;
                if (sg.y > sg.w) continue;
                const int x0 = min(sg.x, sg.z) - rq, x1 = max(sg.x, sg.z) + rq, y0 = sg.y - rq, y1 = sg.w + rq;
                if (in_quad(s.mq, x0, y0) && in_quad(s.mq, x1, y0) && in_quad(s.mq, x1, y1) && in_quad(s.mq, x0, y1))
                    write_dead_entry(d, e);
            }
            __syncthreads();
            unsigned long long my_total = 0ull, my_cov = 0ull;
            int j0 = 0;
            if (tid == 0) s.next_w0 = 0;
            // axis-aligned straights: bitmap only around the corners, the rest in closed form
            if (FCPP_COVER_RECT && !(mode & 1) && s.nrect > 0 &&
                band_zoned(s, d, nh - 1, rq, H, invH, nx, ny, my_total, my_cov))
                j0 = ny;
            while (j0 < ny) {
                // --- how many rows to try: from the word count of the first row.  The previous pass
                // has usually computed it already (its first row that did not fit) ---
                if (tid == 0) {
                    int w0 = s.next_w0;
                    if (w0 <= 0) {
                        int a0, b0, a1, b1;
                        quad_row_interval(s.fq, s.qedge[0], s.qtype[0], j0 * H, H, invH, nx, a0, b0);
                        quad_row_interval(s.mq, s.qedge[1], s.qtype[1], j0 * H, H, invH, nx, a1, b1);
                        w0 = (a1 <= b1) ? words_of(a0, a1 - 1) + words_of(b1 + 1, b0) : words_of(a0, b0);
                    }
                    const int rt = (5 * TW) / (4 * (w0 > 0 ? w0 : 1)) + 8;
                    s.cnt[0] = min(max(rt, 8), min(ROWCAP, ny - j0));
                    s.next_w0 = 0;
                    s.nrows = 0;
                    s.total_words = 0;
                }
                __syncthreads();
                const int rows_try = s.cnt[0];
                // --- row windows + word counts: one row per thread and round (rows k = tid + round*T) ---
                constexpr int ROUNDS = ROWCAP / T;
                int wcnt[ROUNDS], cells[ROUNDS];
                int fit_rows = 0, fit_words = 0, carry = 0;
#pragma unroll
                for (int q = 0; q < ROUNDS; ++q) {
                    const int k = tid + q * T;
                    wcnt[q] = 0;
                    cells[q] = 0;
                    if (q * T >= rows_try) continue;  // uniform
                    int4 win = make_int4(1, 0, 1, 0);
                    int n1 = 0;
                    if (k < rows_try) {
                        win = band_row_windows(s, (j0 + k) * H, H, invH, nx);
                        n1 = words_of(win.x, win.y);
                        wcnt[q] = n1 + words_of(win.z, win.w);
                        cells[q] = max(win.y - win.x + 1, 0) + max(win.w - win.z + 1, 0);
                    }
                    int v[1] = {wcnt[q]};
                    const int round_total = block_scan<1>(v, s.scan);  // inclusive prefix (syncs inside)
                    const int wsum = carry + v[0];
                    carry += round_total;
                    if (k < rows_try) {
                        const int base = wsum - wcnt[q];
                        s.rwin[k] = win;
                        s.rbias[k] = make_int2(base - (win.x >> 5), base + n1 - (win.z >> 5));
                        if (wsum <= TW) {
                            fit_rows = k + 1;
                            fit_words = wsum;
                        }
                    }
                }
                if (fit_rows) {
                    atomicMax(&s.nrows, fit_rows);
                    atomicMax(&s.total_words, fit_words);
                }
                __syncthreads();
                const int nrows = s.nrows, nwords = s.total_words;
                if (nrows == 0) {  // a single row does not fit the tile
                    err11 = 1;
                    break;
                }
                zero_words(s.tile, nwords);
#pragma unroll
                for (int q = 0; q < ROUNDS; ++q) {
                    const int k = tid + q * T;
                    if (k < nrows) my_total += (unsigned long long)cells[q];
                    if (k == nrows && k < rows_try) s.next_w0 = wcnt[q];  // first row of the next pass
                }
                if (tid == 0) {
                    Target &t = s.tg[0];
                    t.j0 = j0;
                    t.nrows = nrows;
                    t.koff = 0;
                }
                __syncthreads();
                {
                    fill_rects(s, j0, nrows, 0);
                    auto tgt = [&](int) { return 0; };
                    raster_entries(s, d, 0, nh - 1, tgt, rq, H, invH);
                }
                my_cov += (unsigned long long)count_words(s.tile, nwords);
                __syncthreads();
                j0 += nrows;
            }
#pragma unroll
            for (int dd = 16; dd > 0; dd >>= 1) {
                my_total += __shfl_xor_sync(0xffffffffu, my_total, dd);
                my_cov += __shfl_xor_sync(0xffffffffu, my_cov, dd);
            }
            if ((tid & 31) == 0) {
                atomicAdd(&s.acc[0], my_total);
                atomicAdd(&s.acc[1], my_cov);
            }
            __syncthreads();
        }
        if (tid == 0) {
            sum->cov_total = (ok && !err11) ? (int64_t)s.acc[0] : 0;
            sum->cov_cells = (ok && !err11) ? (int64_t)s.acc[1] : 0;
        }
    }
    if (tid == 0 && (err10 | err11))
        sum->status |= FCPP_CAND_GRID_TOO_LARGE | (err10 ? FCPP_CAND_CORNER_GRID_TOO_LARGE : 0) |
                       (err11 ? FCPP_CAND_BAND_GRID_TOO_LARGE : 0);
}

__global__ void __launch_bounds__(T, FCPP_COVER_MINBLOCKS) cover_kernel(const fcpp_batch b, const CandRec *__restrict__ recs,
                                                                        const TrigTables *__restrict__ trig,
                                                                        fcpp_summary *__restrict__ summary, int pc, int mode,
                                                                        const int32_t *__restrict__ rep,
                                                                        uint32_t *__restrict__ corner_bits,
                                                                        int64_t corner_bits_stride)
{
    cover_body(b, recs, trig, summary, pc, mode, rep, corner_bits, corner_bits_stride, blockIdx.x);
}

// De-duplicated batches: the candidates that rasterise at least one part are listed (cover_list_kernel) and a
// PERSISTENT grid of two CTAs per SM takes them from the list with an atomic counter — a heading search of
// 737 280 candidates has ~4 096 of them, and launching 737 280 mostly empty 512-thread / 105 KB CTAs cost 4 ms.
__global__ void __launch_bounds__(T, FCPP_COVER_MINBLOCKS) cover_work_kernel(const fcpp_batch b, const CandRec *__restrict__ recs,
                                                                             const TrigTables *__restrict__ trig,
                                                                             fcpp_summary *__restrict__ summary, int pc, int mode,
                                                                             const int32_t *__restrict__ rep,
                                                                             uint32_t *__restrict__ corner_bits,
                                                                             int64_t corner_bits_stride,
                                                                             const int32_t *__restrict__ work,
                                                                             int32_t *__restrict__ counters /*[0] listed, [1] next*/)
{
    __shared__ int s_item;
    for (bool first = true;; first = false) {
        __syncthreads();  // the previous item's shared memory is no longer read
        if (threadIdx.x == 0) {
            CoverFixed &s = *reinterpret_cast<CoverFixed *>(cover_smem);
            s_item = atomicAdd(&counters[1], 1);
            // the next item initialises the mbarrier again (every listed item initialises and completes it)
            if (!first) asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(&s.bar)) : "memory");
        }
        __syncthreads();
        const int w = s_item;
        if (w >= counters[0]) return;
        cover_body(b, recs, trig, summary, pc, mode, rep, corner_bits, corner_bits_stride, work[w]);
    }
}

int cover_point_capacity(int max_head)
{
    const int pc = max_head > 4 * VPOLY_CAP ? max_head : 4 * VPOLY_CAP;
    return (pc + 63) / 64 * 64 + 16;  // a multiple of 16
}

}  // namespace


// ---------------------------------------------------------------------------------------------
// Coverage de-duplication.  A10 / A11 depend on the field, R, W, the start corner and the turn
// model only — not on the heading or the pass order — so in a heading search (BASELINE config 3:
// 180 headings per field) 179 of 180 candidates repeat the coverage of another one.  Candidates
// are grouped by a 64-bit hash of every CandRec field the coverage kernel reads (open-addressing
// table, lowest candidate index per key), the group's first candidate is VERIFIED field by field
// (a hash collision only costs the saving, never correctness), the kernel runs for one
// representative per group and the others copy its integers.
// ---------------------------------------------------------------------------------------------
namespace {

// table slot: key (0 = empty) and 0x7fffffff - (lowest candidate index) kept with atomicMax.  The
// table is zeroed when it is allocated and every batch clears the slots it used (cover_copy_kernel),
// so the steady state has no memset.  Both parts share the table (different hash seeds; a cross-part
// collision is caught by the verification like any other).
__global__ void __launch_bounds__(128) cover_key_kernel(const CandRec *__restrict__ recs, int64_t n,
                                                        unsigned long long *__restrict__ keys,
                                                        unsigned int *__restrict__ vals, uint32_t cap_mask,
                                                        unsigned long long *__restrict__ hash /*[2][n]*/)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
#pragma unroll
    for (int part = 0; part < 2; ++part) {
        const unsigned long long h = recs[c].cover_key[part];  // hashed by the layout kernel
        hash[part * n + c] = h;
        uint32_t slot = (uint32_t)(h >> 17) & cap_mask;
        while (true) {
            const unsigned long long prev = atomicCAS(&keys[slot], 0ull, h);
            if (prev == 0ull || prev == h) {
                atomicMax(&vals[slot], 0x7fffffffu - (unsigned int)c);
                break;
            }
            slot = (slot + 1) & cap_mask;
        }
    }
}

__global__ void __launch_bounds__(128) cover_rep_kernel(const CandRec *__restrict__ recs, int64_t n,
                                                        const unsigned long long *__restrict__ keys,
                                                        const unsigned int *__restrict__ vals, uint32_t cap_mask,
                                                        unsigned long long *__restrict__ hash /*[2][n]*/,
                                                        int32_t *__restrict__ rep /*[2][n]*/)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
#pragma unroll
    for (int part = 0; part < 2; ++part) {
        const unsigned long long h = hash[part * n + c];
        uint32_t slot = (uint32_t)(h >> 17) & cap_mask;
        while (keys[slot] != h) slot = (slot + 1) & cap_mask;
        hash[part * n + c] = slot;  // remembered for the clean-up
        const int64_t first = (int64_t)(0x7fffffffu - vals[slot]);
        rep[part * n + c] = (first < c && cover_same(recs[c], recs[first], part)) ? (int32_t)first : (int32_t)c;
    }
}

// the candidates that rasterise a part, in any order
__global__ void __launch_bounds__(128) cover_list_kernel(int64_t n, const int32_t *__restrict__ rep /*[2][n]*/,
                                                         int32_t *__restrict__ work, int32_t *__restrict__ counters)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool on = c < n && (rep[c] == (int32_t)c || rep[n + c] == (int32_t)c);
    const unsigned m = __ballot_sync(0xffffffffu, on);
    if (m == 0) return;
    const int lane = threadIdx.x & 31;
    int base = 0;
    if (lane == 0) base = atomicAdd(&counters[0], __popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (on) work[base + __popc(m & ((1u << lane) - 1))] = (int32_t)c;
}

__global__ void __launch_bounds__(128) cover_copy_kernel(fcpp_summary *__restrict__ summary, int64_t n,
                                                         const int32_t *__restrict__ rep /*[2][n]*/,
                                                         unsigned long long *__restrict__ keys,
                                                         unsigned int *__restrict__ vals,
                                                         const unsigned long long *__restrict__ slot_of /*[2][n]*/)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
#pragma unroll
    for (int part = 0; part < 2; ++part) {  // leave the table empty for the next batch
        const uint32_t slot = (uint32_t)slot_of[part * n + c];
        keys[slot] = 0ull;
        vals[slot] = 0u;
    }
    fcpp_summary &dst = summary[c];
    const int32_t q0 = rep[c], q1 = rep[n + c];
    if (q0 != (int32_t)c) {
        const fcpp_summary &src = summary[q0];
        for (int k = 0; k < 4; ++k) {
            dst.corner_before[k] = src.corner_before[k];
            dst.corner_after[k] = src.corner_after[k];
        }
        // only the part that was shared: the representative's detail bit of THIS part is final since the coverage
        // kernel (this kernel only ever adds the other part's bits to a candidate that represents a part)
        if (src.status & FCPP_CAND_CORNER_GRID_TOO_LARGE)
            dst.status |= FCPP_CAND_GRID_TOO_LARGE | FCPP_CAND_CORNER_GRID_TOO_LARGE;
    }
    if (q1 != (int32_t)c) {
        const fcpp_summary &src = summary[q1];
        dst.cov_cells = src.cov_cells;
        dst.cov_total = src.cov_total;
        if (src.status & FCPP_CAND_BAND_GRID_TOO_LARGE) dst.status |= FCPP_CAND_GRID_TOO_LARGE | FCPP_CAND_BAND_GRID_TOO_LARGE;
    }
}

}  // namespace

// few representatives expected (a heading search): persistent grid over the listed candidates.  (Measured: config 3
// coverage 4.0 -> 2.8 ms per 737 280 candidates; batches where most candidates rasterise a part — configs 2 and 5 —
// run 1.5-2.5 % slower that way, hence the hint.  Cover mode bits 6 / 7 force either.)
static bool cover_use_work_list(const fcpp_handle *h, const fcpp_batch &b)
{
    return (b.cover_dedupe >= 2 || (h->cover_mode & 128)) && !(h->cover_mode & 64);
}

static int dedupe_threads(const fcpp_handle *h, int64_t n) { return n <= 2 * 32 * (int64_t)h->sm_count ? 32 : 128; }

// Coverage of a batch: (when the batch asks for it) the de-duplication kernels, the coverage kernel, then the copy of
// the representatives' counts to the other members of their groups, which also empties the hash table.
cudaError_t fcpp_launch_cover(fcpp_handle *h, const fcpp_batch &b, const fcpp_outputs &o, cudaStream_t st)
{
    if (b.n_cand == 0) return cudaSuccess;
    int pc = cover_point_capacity(h->cover_pcap);
    while (cover_smem_bytes(pc) > (size_t)h->max_smem_optin && pc > 4 * VPOLY_CAP + 16) pc -= 64;
    const size_t bytes = cover_smem_bytes(pc);
    int32_t *d_rep = nullptr;
    unsigned long long *keys = nullptr, *hash = nullptr;
    unsigned int *vals = nullptr;
    int32_t *work = nullptr, *counters = nullptr;  // de-duplicated batches: the listed candidates (cover_work_kernel)
    cudaError_t e;
    // de-duplication (asked for by the batch, unless switched off by cover mode bit 1)
    const int64_t n = b.n_cand;
    // (one thread per candidate, latency bound: small batches use 32-thread CTAs to reach more SMs)
    const int th = dedupe_threads(h, n);
    if (b.cover_dedupe && n > 1 && !(h->cover_mode & 2) && n < (1ll << 28)) {
        uint32_t cap = 1024;
        while ((int64_t)cap < 4 * n) cap <<= 1;  // two keys per candidate, load factor <= 1/2
        const size_t need = (size_t)cap * 12 + (size_t)n * 28 + 64;
        if (need > h->dedupe_bytes) {
            if (h->d_dedupe) cudaFree(h->d_dedupe);
            h->d_dedupe = nullptr;
            h->dedupe_bytes = 0;
            e = cudaMalloc(&h->d_dedupe, need);
            if (e != cudaSuccess) return e;
            h->dedupe_bytes = need;
            h->dedupe_cap = 0;
        }
        // layout: keys [cap] | vals [cap] | hash / slot [2][n] | rep [2][n] | work [n] | counters [2]; a different
        // capacity moves the arrays, so the table is zeroed again
        keys = (unsigned long long *)h->d_dedupe;
        vals = (unsigned int *)(keys + cap);
        hash = (unsigned long long *)(vals + cap);
        d_rep = (int32_t *)(hash + 2 * n);
        if (h->dedupe_cap != cap) {
            e = cudaMemsetAsync(h->d_dedupe, 0, (size_t)cap * 12, st);
            if (e != cudaSuccess) return e;
            h->dedupe_cap = cap;
        }
        const unsigned g = (unsigned)((n + th - 1) / th);
        cover_key_kernel<<<g, th, 0, st>>>(h->d_rec, n, keys, vals, cap - 1, hash);
        cover_rep_kernel<<<g, th, 0, st>>>(h->d_rec, n, keys, vals, cap - 1, hash, d_rep);
        h->launches += 2;
        if (cover_use_work_list(h, b)) {
            work = d_rep + 2 * n;
            counters = work + n;
            e = cudaMemsetAsync(counters, 0, 2 * sizeof(int32_t), st);
            if (e != cudaSuccess) return e;
            cover_list_kernel<<<g, th, 0, st>>>(n, d_rep, work, counters);
            h->launches++;
        }
        e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    if (work) {
        e = cudaFuncSetAttribute(cover_work_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e != cudaSuccess) return e;
        int64_t grid = (int64_t)FCPP_COVER_MINBLOCKS * h->sm_count;
        if (grid > n) grid = n;
        cover_work_kernel<<<(unsigned)grid, T, bytes, st>>>(b, h->d_rec, h->d_trig, o.summary, pc, h->cover_mode, d_rep,
                                                            o.corner_bits, o.corner_bits_stride, work, counters);
    } else {
        e = cudaFuncSetAttribute(cover_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e != cudaSuccess) return e;
        cover_kernel<<<(unsigned)n, T, bytes, st>>>(b, h->d_rec, h->d_trig, o.summary, pc, h->cover_mode, d_rep,
                                                    o.corner_bits, o.corner_bits_stride);
    }
    h->launches++;
    e = cudaGetLastError();
    if (e != cudaSuccess || !d_rep) return e;
    cover_copy_kernel<<<(unsigned)((n + th - 1) / th), th, 0, st>>>(o.summary, n, d_rep, keys, vals, hash);
    h->launches++;
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// generic window raster for the drop-in verify_corner_coverage_grid_based (mlp3:1426-1510)
// ---------------------------------------------------------------------------------------------
namespace {

constexpr int WIN_PC = 1024 + 16;

__global__ void __launch_bounds__(T) window_kernel(const double *__restrict__ path, int n_pts, double radius,
                                                   double ox, double oy, double hc, int g,
                                                   uint32_t *__restrict__ bits, int64_t *__restrict__ count)
{
    // one CTA; rows are processed in tiles of the shared occupancy buffer, then merged into the
    // caller's row-major g x g bit grid (bit j*g+i)
    CoverFixed &s = *reinterpret_cast<CoverFixed *>(cover_smem);
    const CoverDyn d;
    const int tid = threadIdx.x;
    const int64_t X0 = qfix(ox), Y0 = qfix(oy);
    const int H = (int)qfix(hc);
    const double invH = 1.0 / (double)H;
    const int rq = (int)qfix(radius);
    const int rw = (g + 31) >> 5;
    const int rows_per_tile = min(ROWCAP, TW / rw);
    const int64_t lim = (1ll << 30);
    for (int j0 = 0; j0 < g; j0 += rows_per_tile) {
        const int nrows = min(rows_per_tile, g - j0);
        for (int k = tid; k < nrows; k += T) {
            s.rwin[k] = make_int4(0, g - 1, 1, 0);
            s.rbias[k] = make_int2(k * rw, 0);
        }
        zero_words(s.tile, nrows * rw);
        if (tid == 0) {
            Target &t = s.tg[0];
            t.j0 = j0;
            t.nrows = nrows;
            t.koff = 0;
        }
        __syncthreads();
        // polyline in chunks of 1024 points (chunks overlap by one point); points far outside
        // the window are clamped (they cannot reach it, the capsule radius is tiny against 2^30)
        for (int p0 = 0; p0 + 1 < n_pts; p0 += 1023) {
            const int np = min(1024, n_pts - p0);
            for (int k = tid; k < np; k += T) {
                int64_t x = qfix(path[2 * (p0 + k)]) - X0, y = qfix(path[2 * (p0 + k) + 1]) - Y0;
                x = x < -lim ? -lim : (x > lim ? lim : x);
                y = y < -lim ? -lim : (y > lim ? lim : y);
                d.ent(k).erow = make_int2((int)x, (int)y);
            }
            __syncthreads();
            setup_entries<true, false>(s, d, 0, np - 1, (double)rq, rq, H, invH);
            __syncthreads();
            auto tgt = [&](int) { return 0; };
            raster_entries(s, d, 0, np - 1, tgt, rq, H, invH);
        }
        // merge into the global bit grid
        for (int c = tid; c < nrows * g; c += T) {
            const int k = c / g, i = c - k * g;
            if ((s.tile[k * rw + (i >> 5)] >> (i & 31)) & 1u) {
                const int64_t bit = (int64_t)(j0 + k) * g + i;
                atomicOr(&bits[bit >> 5], 1u << (bit & 31));
            }
        }
        __syncthreads();
    }
    __threadfence();
    __syncthreads();
    // count all set bits of the (merged) grid
    if (tid == 0) s.acc[0] = 0ull;
    __syncthreads();
    const int64_t nw = ((int64_t)g * g + 31) >> 5;
    unsigned long long c = 0;
    for (int64_t w = tid; w < nw; w += T) c += __popc(bits[w]);
    atomicAdd(&s.acc[0], c);
    __syncthreads();
    if (tid == 0) *count = (int64_t)s.acc[0];
}

}  // namespace

cudaError_t fcpp_launch_raster_window(fcpp_handle *h, const double *d_path, int32_t n_pts, double radius,
                                      double ox, double oy, double hc, int32_t g, uint32_t *d_bits,
                                      int64_t *d_count, cudaStream_t st)
{
    const size_t bytes = cover_smem_bytes(WIN_PC);
    cudaError_t e = cudaFuncSetAttribute(window_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return e;
    window_kernel<<<1, T, bytes, st>>>(d_path, n_pts, radius, ox, oy, hc, g, d_bits, d_count);
    h->launches++;
    return cudaGetLastError();
}
