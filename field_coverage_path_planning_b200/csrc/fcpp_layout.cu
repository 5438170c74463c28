// fcpp_layout.cu — per-candidate FP64 geometry/layout pass (one thread per candidate) and the
// exclusive prefix sum of the point counts.
//
// Restates the scalar part of the reference planner (multi_layer_planner_v3.py, "mlp3"):
//   work-area inset + rotation + bounds + pass count      mlp3:591-611, :682-701, :731-739
//   headland loop rings and loop count                    mlp3:916, :924, :964-972
//   reverse-fill direction / length / sample count        mlp3:1066-1080, :1154-1288
//   verification-corner reverse fills                     mlp3:1531-1554
// in the same FP64 operation order as oracle/ref_planner.py (compiled with -fmad=false).
#include "fcpp_internal.cuh"

namespace {


__device__ int layout_one(const fcpp_batch &b, const TrigTables *__restrict__ trig, CandRec *__restrict__ recs,
                          int32_t *__restrict__ n_pts, int64_t c)
{
    const TrigTables &tt = *trig;
    TurnModel tm;
    tm.model = b.turn_model;
    tm.lam = b.clothoid_share;
    CandRec &r = recs[c];
    const double W = b.vehicle.working_width;
    // the candidate's parameters: explicit arrays, or decoded from its index in the Cartesian product of the axes
    int f, flags;
    double R;
    const double *rot;
    if (b.cand_field) {
        f = b.cand_field[c];
        R = b.cand_R[c];
        flags = b.cand_flags[c];
        rot = b.cand_rot + 4 * c;
    } else {
        const int nh = max(b.n_ax_headings, 1), nr = max(b.n_ax_radii, 1), nc = max(b.n_ax_corners, 1);
        const int64_t per = (int64_t)nh * nr * nc;
        const int64_t g = b.cand_first + c;
        f = (int)(g / per);
        const int rem = (int)(g - (int64_t)f * per);
        const int ih = rem / (nr * nc), ir = (rem / nc) % nr, ic = rem % nc;
        flags = 0;
        if (b.n_ax_corners > 0) {
            // corner k in {0: LB, 1: RB, 2: RT, 3: LT}: reverse order iff k in {2, 3}, start from the right iff k in
            // {1, 2} (mlp3:650-658)
            const int k = b.ax_corners[ic] & 3, hi = k >> 1;
            flags = k | (hi ? FCPP_FLAG_REVERSE_ORDER : 0) | (((k ^ hi) & 1) ? FCPP_FLAG_START_FROM_RIGHT : 0);
        }
        if (b.n_ax_radii > 0) {
            R = b.ax_radii[ir];
            flags |= b.ax_radius_flags[ir];
        } else {
            R = b.ax_default_radius;
            flags |= b.ax_default_radius_flags;
        }
        if (b.n_ax_headings > 0) {
            rot = b.ax_heading_rot + 4 * ih;
            flags |= b.ax_heading_flags[ih];
        } else {
            rot = b.field_rot + 4 * (int64_t)f;
            flags |= b.field_rot_flags[f];
        }
    }
    double v[4][2];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        v[k][0] = b.field_verts[(int64_t)f * 8 + 2 * k];
        v[k][1] = b.field_verts[(int64_t)f * 8 + 2 * k + 1];
    }
    const double fl = b.field_extent[2 * f], fw = b.field_extent[2 * f + 1];
    const int fflags = b.field_flags[f];
    int status = 0;

    // ---- layer 1: work area (mlp3:594-598) ----
    double mq[4][2];
    bool ok = inset4(v, R, mq);
    const double area = fabs(signed_area4(mq));
    if (!ok || area < 1.0) status |= FCPP_CAND_INSET_EMPTY;
    double cx = 0.0, cy = 0.0;
    double rv[4][2];
    if (flags & FCPP_FLAG_ROTATED) {
        // centroid of work area minus buffered obstacles (mlp3:601-609, :690) — oracle
        // work_area_centroid order: a, a*c, then sequential subtraction per obstacle
        double gx, gy;
        centroid4(mq, gx, gy);
        const int p0 = b.obs_poly_start ? b.obs_poly_start[f] : 0;
        const int p1 = b.obs_poly_start ? b.obs_poly_start[f + 1] : 0;
        if (p1 > p0) {
            double a = area, mx = area * gx, my = area * gy;
            for (int p = p0; p < p1; ++p) {
                a -= b.obs_moments[3 * p];
                mx -= b.obs_moments[3 * p + 1];
                my -= b.obs_moments[3 * p + 2];
            }
            cx = mx / a;
            cy = my / a;
        } else {
            cx = gx;
            cy = gy;
        }
        const double cn = rot[0], sn = rot[1];
#pragma unroll
        for (int k = 0; k < 4; ++k) rotate_pt(mq[k][0], mq[k][1], cn, sn, cx, cy, rv[k][0], rv[k][1]);
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            rv[k][0] = mq[k][0];
            rv[k][1] = mq[k][1];
        }
    }
    double min_x = rv[0][0], max_x = rv[0][0], min_y = rv[0][1], max_y = rv[0][1];
#pragma unroll
    for (int k = 1; k < 4; ++k) {
        min_x = fmin(min_x, rv[k][0]);
        max_x = fmax(max_x, rv[k][0]);
        min_y = fmin(min_y, rv[k][1]);
        max_y = fmax(max_y, rv[k][1]);
    }
    if ((flags & FCPP_FLAG_START_POINT) && b.cand_start) {
        // mlp3:689-696 + :649-658: pass order from the (rotated) start point
        double sx = b.cand_start[2 * c], sy = b.cand_start[2 * c + 1];
        if (flags & FCPP_FLAG_ROTATED) rotate_pt(sx, sy, rot[0], rot[1], cx, cy, sx, sy);
        flags &= ~(FCPP_FLAG_REVERSE_ORDER | FCPP_FLAG_START_FROM_RIGHT);
        if (sy > (min_y + max_y) / 2) flags |= FCPP_FLAG_REVERSE_ORDER;
        if (sx > (min_x + max_x) / 2) flags |= FCPP_FLAG_START_FROM_RIGHT;
    }
    int P = 1;
    if (!(status & FCPP_CAND_INSET_EMPTY)) P = (int)((max_y - min_y) / W) + 1;  // mlp3:739
    if (P < 1) P = 1;
    const int n_main = 2 * P + FCPP_UTURN_POINTS * (P - 1);

    // ---- layer 2: K loops (mlp3:916-933, :964-972) ----
    int K = (int)ceil(R / W);
    if (K > FCPP_MAX_LOOPS) {
        status |= FCPP_CAND_TOO_MANY_LOOPS;
        K = FCPP_MAX_LOOPS;
    }
    if (K < 0) K = 0;
    for (int k = 0; k < K; ++k) {
        const double off = W / 2 + k * W;
        double ring[4][2];
        const bool okk = inset4(v, off, ring);
        if (!okk || fabs(signed_area4(ring)) < 1.0) status |= FCPP_CAND_LOOP_SKIPPED;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            r.corners[k][q][0] = ring[q][0];
            r.corners[k][q][1] = ring[q][1];
        }
    }
    const int sc = flags & FCPP_FLAG_CORNER_MASK;
    const bool gate = (flags & FCPP_FLAG_GAP_GATE) != 0;
    int n_head = (FCPP_POINTS_PER_LOOP)*K;
    for (int t = 0; t < 3; ++t) {
        const int ni = (sc + t + 1) & 3;
        int n = 0;
        if (K > 0 && gate && ((fflags >> ni) & 1))  // mlp3:1043, :1070
            n = reverse_fill(tt, tm, r.corners[0][ni][0], r.corners[0][ni][1], ni, R, fl, fw, r.rev[t]);
        else {
#pragma unroll
            for (int q = 0; q < 5; ++q) r.rev[t][q] = 0.0;
        }
        r.n_rev[t] = n;
        n_head += n;
    }
    // every straight of every loop axis-aligned on the lattice: the band's corner zones do not depend on the
    // start corner (fcpp_cover.cu: band_grouped); only de-duplicated batches group bands
    const bool dd = b.cover_dedupe && b.do_coverage;
    bool axis = dd && K > 0;
    for (int k = 0; axis && k < K; ++k)
        for (int q = 0; q < 4; ++q) {
            const int q1 = (q + 1) & 3;
            const bool vx = qfix(r.corners[k][q][0]) == qfix(r.corners[k][q1][0]);
            const bool vy = qfix(r.corners[k][q][1]) == qfix(r.corners[k][q1][1]);
            axis = axis && (vx != vy);
        }
    // ---- verification corners (mlp3:1531-1554): main-area corners (hw,hw)… with hw = R ----
    for (int ci = 0; ci < 4; ++ci) {
        const double qx = (ci == 0 || ci == 3) ? R : fl - R;
        const double qy = (ci == 0 || ci == 1) ? R : fw - R;
        int n = 0;
        if (gate)
            n = reverse_fill(tt, tm, qx, qy, ci, R, fl, fw, r.vrev[ci]);
        else {
#pragma unroll
            for (int q = 0; q < 5; ++q) r.vrev[ci][q] = 0.0;
        }
        r.vn_rev[ci] = n;
    }
    r.corner_g = (int)(2 * R / FCPP_CORNER_GRID_H);  // mlp3:1457
    // the reference raises at the first failure: layer 1 (mlp3:597) comes before layer 2 (mlp3:967)
    if (status & FCPP_CAND_INSET_EMPTY) status = FCPP_CAND_INSET_EMPTY;
    if (status & (FCPP_CAND_INSET_EMPTY | FCPP_CAND_LOOP_SKIPPED | FCPP_CAND_TOO_MANY_LOOPS)) {
        // the reference raises here; no points are produced
        r.n_main = 0;
        r.n_head = 0;
        r.n_total = 0;
    } else {
        r.n_main = n_main;
        r.n_head = n_head;
        r.n_total = n_main + n_head;
    }
    r.status = status;
    r.band_group = (axis && status == 0) ? 1 : 0;
    r.P = P;
    r.K = K;
    r.flags = flags;
    r.field = f;
    r.R = R;
    r.min_x = min_x;
    r.min_y = min_y;
    r.max_x = max_x;
    r.max_y = max_y;
    r.cx = cx;
    r.cy = cy;
    r.cos_a = rot[2];
    r.sin_a = rot[3];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        r.main_quad[k][0] = mq[k][0];
        r.main_quad[k][1] = mq[k][1];
    }
    r.cover_key[0] = dd ? cover_key(r, 0) : 0ull;
    r.cover_key[1] = dd ? cover_key(r, 1) : 0ull;
    r.pad1 = 0;
    if (n_pts) n_pts[c] = r.n_total;
    return r.n_total;
}

__global__ void __launch_bounds__(128) layout_kernel(fcpp_batch b, const TrigTables *__restrict__ trig,
                                                     CandRec *__restrict__ recs, int32_t *__restrict__ n_pts,
                                                     int *__restrict__ maxn)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int nt = 0, nh = 0;
    if (c < b.n_cand) {
        nt = layout_one(b, trig, recs, n_pts, c);
        nh = recs[c].n_head;
    }
    const int wmax = __reduce_max_sync(0xffffffffu, nt);
    const int hmax = __reduce_max_sync(0xffffffffu, nh);
    if ((threadIdx.x & 31) == 0) {
        atomicMax(maxn, wmax);
        atomicMax(maxn + 1, hmax);
    }
}

// ---- exclusive prefix sum int32 -> int64 (three small kernels; B is at most a few million) ----
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 16;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__device__ __forceinline__ int64_t block_exclusive_scan(int64_t v, int64_t *sh, int64_t &total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int64_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int64_t o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += o;
    }
    if (lane == 31) sh[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int64_t w = (lane < SCAN_THREADS / 32) ? sh[lane] : 0;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int64_t o = __shfl_up_sync(0xffffffffu, w, d);
            if (lane >= d) w += o;
        }
        sh[32 + lane] = w;
    }
    __syncthreads();
    const int64_t warp_off = warp ? sh[32 + warp - 1] : 0;
    total = sh[32 + SCAN_THREADS / 32 - 1];
    __syncthreads();
    return warp_off + inc - v;
}

__global__ void __launch_bounds__(SCAN_THREADS) scan_tiles_kernel(const CandRec *__restrict__ recs, int64_t n,
                                                                   int64_t *__restrict__ offsets,
                                                                   int64_t *__restrict__ tile_sums,
                                                                   int64_t *__restrict__ single_total)
{
    __shared__ int64_t sh[64];
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    int64_t loc[SCAN_ITEMS];
    int64_t s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
        const int64_t i = base + k;
        const int64_t x = (i < n) ? recs[i].n_total : 0;
        loc[k] = s;
        s += x;
    }
    int64_t total;
    const int64_t off = block_exclusive_scan(s, sh, total);
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
        const int64_t i = base + k;
        if (i < n) offsets[i] = off + loc[k];
    }
    if (threadIdx.x == 0) {
        tile_sums[blockIdx.x] = total;
        if (single_total) *single_total = total;  // one tile: the scan is complete, offsets[n] = total
    }
}

__global__ void __launch_bounds__(SCAN_THREADS) scan_sums_kernel(int64_t *tile_sums, int64_t n_tiles,
                                                                  int64_t *offsets_total)
{
    __shared__ int64_t sh[64];
    int64_t carry = 0;
    for (int64_t base = 0; base < n_tiles; base += SCAN_THREADS) {
        const int64_t i = base + threadIdx.x;
        const int64_t x = (i < n_tiles) ? tile_sums[i] : 0;
        int64_t total;
        const int64_t off = block_exclusive_scan(x, sh, total);
        if (i < n_tiles) tile_sums[i] = carry + off;
        carry += total;
    }
    if (threadIdx.x == 0) *offsets_total = carry;
}

__global__ void __launch_bounds__(SCAN_THREADS) scan_add_kernel(int64_t *__restrict__ offsets, int64_t n,
                                                                 const int64_t *__restrict__ tile_sums)
{
    const int64_t add = tile_sums[blockIdx.x];
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE;
    for (int k = threadIdx.x; k < SCAN_TILE; k += SCAN_THREADS) {
        const int64_t i = base + k;
        if (i < n) offsets[i] += add;
    }
}

}  // namespace

cudaError_t fcpp_launch_layout(fcpp_handle *h, const fcpp_batch &b, int32_t *d_n_pts, int64_t *d_offsets,
                               cudaStream_t st)
{
    const int64_t B = b.n_cand;
    if (B == 0) {
        if (d_offsets) return cudaMemsetAsync(d_offsets, 0, sizeof(int64_t), st);
        return cudaSuccess;
    }
    // one thread per candidate and a long dependent FP64 chain ending in a 1.5 KB record: a small batch is spread
    // over as many SMs as possible (32-thread CTAs up to ~2 CTAs per SM, then 64, then 128; measured at 4096
    // candidates: 34 / 28 / 26 us with 128 / 64 / 32 threads per CTA)
    int threads = 128;
    if (B <= 2 * 32 * (int64_t)h->sm_count)
        threads = 32;
    else if (B <= 2 * 64 * (int64_t)h->sm_count)
        threads = 64;
    const unsigned blocks = (unsigned)((B + threads - 1) / threads);
    cudaError_t e = cudaMemsetAsync(h->d_maxn, 0, 2 * sizeof(int), st);
    if (e != cudaSuccess) return e;
    layout_kernel<<<blocks, threads, 0, st>>>(b, h->d_trig, h->d_rec, d_n_pts, h->d_maxn);
    h->launches++;
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    if (d_offsets) {
        const int64_t n_tiles = (B + SCAN_TILE - 1) / SCAN_TILE;
        int64_t *tile_sums = (int64_t *)h->d_scan_tmp;
        scan_tiles_kernel<<<(unsigned)n_tiles, SCAN_THREADS, 0, st>>>(h->d_rec, B, d_offsets, tile_sums,
                                                                        n_tiles == 1 ? d_offsets + B : nullptr);
        h->launches++;
        if (n_tiles > 1) {  // batches of more than 4096 candidates: prefix of the tile sums, then add
            scan_sums_kernel<<<1, SCAN_THREADS, 0, st>>>(tile_sums, n_tiles, d_offsets + B);
            scan_add_kernel<<<(unsigned)n_tiles, SCAN_THREADS, 0, st>>>(d_offsets, B, tile_sums);
            h->launches += 2;
        }
        e = cudaGetLastError();
    }
    return e;
}
