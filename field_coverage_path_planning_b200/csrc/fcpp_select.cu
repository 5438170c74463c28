// fcpp_select.cu — per-field top-k of the candidates under a constraint-aware cost (fcpp_field_select) and the
// multi-GPU merge of the ranks' rankings (fcpp_field_select_merge).  No reference counterpart: build-defined
// selection on top of the per-candidate summaries (DESIGN.md §3.8; SURVEY.md §8(b): ties to the lowest index).
//
// A PLAIN selection (top_k 1, no limit, the weights of length alone or time alone) is the per-field argmin and runs
// the argmin kernels: one CTA up to 16 384 candidates and fields, else four kernels — one launch where the pipeline
// below takes five.  Every other selection runs the pipeline.
//
// Pipeline (every stage exact, the order of the results independent of the order of the candidates):
//   1. select_keys      1 thread / candidate: eligibility, FP64 cost, key = order_bits(cost); the candidate's rank
//                       among the eligible ones of its field from a warp-aggregated atomic on the field's count
//   2. select_scan_*    exclusive prefix of the F + 1 counts: segment [seg[f], seg[f+1]) of field f
//   3. select_scatter   counting sort by field: entry (key, global index, field) to seg[f] + rank.  The rank order
//                       inside a field is arbitrary — the index is part of the key
//   4. select_level     a segmented tree reduction over the sorted entries.  A level-0 unit is a tile of
//                       SEL_TILE entries, a level-l unit the SEL_FANIN units below it.  A unit groups its items
//                       by field; one warp per group selects the group's k lowest (key, index).  A field whose
//                       whole segment lies inside the unit is final and written out; the field of the unit's
//                       first and of its last item may continue in the neighbours: their lists go up one level.
//                       No CTA ever holds more than SEL_TILE items, whatever the length of a field.
#include "fcpp_internal.cuh"

namespace {

constexpr int SEL_THREADS = 256;
constexpr int SEL_TILE = 1024;     // items of a unit (level 0: sorted entries; above: 2 lists x k of each child)
constexpr int SEL_FANIN = 8;       // 8 children x 2 lists x FCPP_SELECT_MAX_K = SEL_TILE
constexpr int SEL_PER_THREAD = SEL_TILE / SEL_THREADS;
constexpr int SCAN_THREADS = 1024;
constexpr int SCAN_PER = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_PER;
constexpr unsigned long long SENT = ~0ull;  // (SENT, SENT) sorts after every real (key, index)
static_assert(SEL_FANIN * 2 * FCPP_SELECT_MAX_K <= SEL_TILE, "a unit's children must fit its item tile");

__device__ __forceinline__ bool key_less(unsigned long long ah, unsigned long long ai, unsigned long long bh,
                                         unsigned long long bi)
{
    return ah < bh || (ah == bh && ai < bi);
}

// include/fcpp.h, fcpp_selection: eligibility and the FP64 cost, left to right (-fmad=false)
__device__ __forceinline__ bool sel_eval(const fcpp_summary &s, const fcpp_selection &p, double &cost)
{
    if (s.status != 0) return false;
    if (p.max_boundary_viol >= 0 && s.n_boundary_viol > p.max_boundary_viol) return false;
    if (p.max_obstacle_viol >= 0 && s.n_obstacle_viol > p.max_obstacle_viol) return false;
    if (p.max_accel_viol >= 0 && s.n_accel_viol > p.max_accel_viol) return false;
    if (p.min_coverage >= 0.0 &&
        !(s.cov_total > 0 && (double)s.cov_cells >= p.min_coverage * (double)s.cov_total))
        return false;
    const double L = s.len_main + s.len_head;
    const double T = s.time_main + s.time_head;
    const double U = (double)(s.cov_total - s.cov_cells) * p.cell_area;
    cost = p.w_length * L + p.w_time * T + p.w_boundary * (double)s.n_boundary_viol +
           p.w_obstacle * (double)s.n_obstacle_viol + p.w_accel * (double)s.n_accel_viol + p.w_uncovered * U;
    return true;
}

// 1. keys and per-field ranks; also pads the outputs (+inf / -1: fields without an eligible candidate keep them)
__global__ void __launch_bounds__(256) select_keys(const fcpp_summary *__restrict__ sm, const int32_t *__restrict__ cf,
                                                   const CandRec *__restrict__ recs, int64_t n, int n_fields,
                                                   fcpp_selection p, unsigned long long *__restrict__ cnt,
                                                   unsigned long long *__restrict__ ckey, int2 *__restrict__ frk,
                                                   double *__restrict__ out_cost, long long *__restrict__ out_cand,
                                                   int64_t n_out)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n_out) {
        out_cost[t] = INFINITY;
        out_cand[t] = -1;
    }
    bool on = false;
    int f = -1;
    double cost = 0.0;
    if (t < n) {
        f = cf ? cf[t] : recs[t].field;
        on = f >= 0 && f < n_fields && sel_eval(sm[t], p, cost);
    }
    // warp-aggregated rank: the lanes of one field take consecutive ranks from ONE atomic
    const unsigned act = __ballot_sync(0xffffffffu, on);
    int rank = 0;
    if (on) {
        const unsigned peers = __match_any_sync(act, f);
        const int lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
        unsigned long long base = 0;
        if (lane == leader) base = atomicAdd(&cnt[f], (unsigned long long)__popc(peers));
        base = __shfl_sync(peers, base, leader);
        rank = (int)base + __popc(peers & ((1u << lane) - 1u));
        ckey[t] = order_bits(cost);
    }
    if (t < n) frk[t] = make_int2(on ? f : -1, rank);
}

__device__ __forceinline__ long long block_exclusive_scan(long long v, long long *sh, long long &total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    long long x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const long long y = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= d) x += y;
    }
    if (lane == 31) sh[warp] = x;
    __syncthreads();
    if (warp == 0) {
        long long w = lane < nw ? sh[lane] : 0;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const long long y = __shfl_up_sync(0xffffffffu, w, d);
            if (lane >= d) w += y;
        }
        if (lane < nw) sh[lane] = w;
    }
    __syncthreads();
    const long long before = warp ? sh[warp - 1] : 0;
    total = sh[nw - 1];
    __syncthreads();  // sh is reused by the caller's next scan
    return before + x - v;
}

// 2. exclusive scan of m counts in place: tiles of SCAN_TILE, their totals, the totals added back
__global__ void __launch_bounds__(SCAN_THREADS) select_scan_tiles(unsigned long long *__restrict__ a, int64_t m,
                                                                  long long *__restrict__ tile_sums)
{
    __shared__ long long sh[32];
    const int64_t i0 = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_PER;
    long long v[SCAN_PER], s = 0;
#pragma unroll
    for (int j = 0; j < SCAN_PER; ++j) {
        v[j] = i0 + j < m ? (long long)a[i0 + j] : 0;
        s += v[j];
    }
    long long total;
    long long run = block_exclusive_scan(s, sh, total);
#pragma unroll
    for (int j = 0; j < SCAN_PER; ++j) {
        if (i0 + j < m) a[i0 + j] = (unsigned long long)run;
        run += v[j];
    }
    if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}
__global__ void __launch_bounds__(SCAN_THREADS) select_scan_sums(long long *tile_sums, int64_t n_tiles)
{
    __shared__ long long sh[32];
    long long carry = 0;
    for (int64_t i0 = 0; i0 < n_tiles; i0 += SCAN_THREADS) {
        const int64_t i = i0 + threadIdx.x;
        const long long v = i < n_tiles ? tile_sums[i] : 0;
        long long total;
        const long long ex = block_exclusive_scan(v, sh, total);
        if (i < n_tiles) tile_sums[i] = carry + ex;
        carry += total;
    }
}
__global__ void __launch_bounds__(SCAN_THREADS) select_scan_add(unsigned long long *__restrict__ a, int64_t m,
                                                                const long long *__restrict__ tile_sums)
{
    const long long add = tile_sums[blockIdx.x];
    const int64_t i0 = (int64_t)blockIdx.x * SCAN_TILE;
    for (int j = threadIdx.x; j < SCAN_TILE; j += SCAN_THREADS)
        if (i0 + j < m) a[i0 + j] += (unsigned long long)add;
}

// 3. counting sort by field
__global__ void __launch_bounds__(256) select_scatter(const unsigned long long *__restrict__ seg,
                                                      const unsigned long long *__restrict__ ckey,
                                                      const int2 *__restrict__ frk, int64_t n, int64_t base,
                                                      ulonglong2 *__restrict__ ent, int32_t *__restrict__ efld)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    const int2 fr = frk[c];
    if (fr.x < 0) return;
    const int64_t pos = (int64_t)seg[fr.x] + fr.y;
    ent[pos] = make_ulonglong2(ckey[c], (unsigned long long)(base + c));
    efld[pos] = fr.x;
}

// the k lowest (key, index) of items [p, q) of the unit's shared tile, one warp; lane j < k returns the j-th
// (SENT, SENT past the last).  Each lane keeps the minimum of its own items (p + lane, p + lane + 32, ...); the
// lane whose minimum wins retires that item and rescans its own items only.
__device__ __forceinline__ void warp_select(unsigned long long *s_hi, unsigned long long *s_idx, int p, int q, int k,
                                            unsigned long long &my_h, unsigned long long &my_i)
{
    const int lane = threadIdx.x & 31;
    unsigned long long bh = SENT, bi = SENT;
    int bp = -1;
    auto rescan = [&]() {
        bh = bi = SENT;
        bp = -1;
        for (int i = p + lane; i < q; i += 32) {
            FCPP_ASSERT(i >= 0 && i < SEL_TILE);
            if (key_less(s_hi[i], s_idx[i], bh, bi)) {
                bh = s_hi[i];
                bi = s_idx[i];
                bp = i;
            }
        }
    };
    rescan();
    my_h = my_i = SENT;
    for (int it = 0; it < k; ++it) {
        unsigned long long wh = bh, wi = bi;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const unsigned long long oh = __shfl_xor_sync(0xffffffffu, wh, d);
            const unsigned long long oi = __shfl_xor_sync(0xffffffffu, wi, d);
            if (key_less(oh, oi, wh, wi)) {
                wh = oh;
                wi = oi;
            }
        }
        if (wh == SENT && wi == SENT) break;  // warp-uniform: every lane holds the same minimum
        if (lane == it) {
            my_h = wh;
            my_i = wi;
        }
        if (bp >= 0 && bh == wh && bi == wi) {  // indices are unique: exactly one lane owns the winner
            FCPP_ASSERT(bp < SEL_TILE);
            s_hi[bp] = SENT;
            s_idx[bp] = SENT;
            rescan();
        }
    }
}

// 4. one unit per CTA.  LEAF: items = sorted entries [lo, hi); else the lists of the unit's present children
// (child c: list 0 of field in_f[2c], list 1 of field in_f[2c + 1], k entries each).  Writes the final rankings of
// the fields complete in [lo, hi) and the unit's own two lists (first / last field) for the level above.
template <bool LEAF>
__global__ void __launch_bounds__(SEL_THREADS) select_level(const unsigned long long *__restrict__ seg, int n_fields,
                                                            int k, int64_t span, int64_t child_span,
                                                            const ulonglong2 *__restrict__ ent,
                                                            const int32_t *__restrict__ efld,
                                                            const int32_t *__restrict__ in_f,
                                                            const ulonglong2 *__restrict__ in_e,
                                                            int32_t *__restrict__ out_f, ulonglong2 *__restrict__ out_e,
                                                            double *__restrict__ out_cost,
                                                            long long *__restrict__ out_cand)
{
    __shared__ unsigned long long s_hi[SEL_TILE], s_idx[SEL_TILE];
    __shared__ int32_t s_fld[SEL_TILE];
    __shared__ int32_t s_gs[SEL_TILE + 1];  // group starts, then n_items
    __shared__ int32_t s_wcount[SEL_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t N = (int64_t)seg[n_fields];
    const int64_t lo = (int64_t)blockIdx.x * span;
    if (lo >= N) return;  // block-uniform
    const int64_t hi = min(lo + span, N);
    const int per_child = 2 * k;
    const int n_it = LEAF ? (int)(hi - lo) : (int)((hi - lo + child_span - 1) / child_span) * per_child;
    FCPP_ASSERT(n_it > 0 && n_it <= SEL_TILE);
    for (int i = tid; i < n_it; i += SEL_THREADS) {
        FCPP_ASSERT(i < SEL_TILE);
        if (LEAF) {
            const ulonglong2 e = ent[lo + i];
            s_hi[i] = e.x;
            s_idx[i] = e.y;
            s_fld[i] = efld[lo + i];
        } else {
            const int64_t child = (int64_t)blockIdx.x * SEL_FANIN + i / per_child;
            const int r = i % per_child;
            const ulonglong2 e = in_e[child * per_child + r];
            s_hi[i] = e.x;
            s_idx[i] = e.y;
            s_fld[i] = in_f[2 * child + (r >= k)];
        }
    }
    // the unit's lists start empty: only a field that continues past the unit's first / last item fills them
    if (tid < per_child) out_e[(int64_t)blockIdx.x * per_child + tid] = make_ulonglong2(SENT, SENT);
    __syncthreads();
    if (tid == 0) {
        out_f[2 * blockIdx.x] = s_fld[0];
        out_f[2 * blockIdx.x + 1] = s_fld[n_it - 1];
    }
    // group starts (items are sorted by field): block compaction of the start flags
    int flag[SEL_PER_THREAD], nf = 0;
#pragma unroll
    for (int j = 0; j < SEL_PER_THREAD; ++j) {
        const int i = tid * SEL_PER_THREAD + j;
        flag[j] = i < n_it && (i == 0 || s_fld[i] != s_fld[i - 1]);
        nf += flag[j];
    }
    int x = nf;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= d) x += y;
    }
    if (lane == 31) s_wcount[warp] = x;
    __syncthreads();
    int before = 0, n_groups = 0;
#pragma unroll
    for (int w = 0; w < SEL_THREADS / 32; ++w) {
        const int c = s_wcount[w];
        before += w < warp ? c : 0;
        n_groups += c;
    }
    int at = before + x - nf;
#pragma unroll
    for (int j = 0; j < SEL_PER_THREAD; ++j)
        if (flag[j]) {
            FCPP_ASSERT(at < SEL_TILE);
            s_gs[at++] = tid * SEL_PER_THREAD + j;
        }
    if (tid == 0) s_gs[n_groups] = n_it;
    __syncthreads();
    for (int g = warp; g < n_groups; g += SEL_THREADS / 32) {
        FCPP_ASSERT(g + 1 <= SEL_TILE);
        const int p = s_gs[g], q = s_gs[g + 1];
        const int f = s_fld[p];
        unsigned long long my_h, my_i;
        warp_select(s_hi, s_idx, p, q, k, my_h, my_i);
        // a group without a real item: lists of a field completed below (or an empty list) — nothing to write
        const bool any = __shfl_sync(0xffffffffu, my_i, 0) != SENT;
        if (!any) continue;
        const bool complete = (int64_t)seg[f] >= lo && (int64_t)seg[f + 1] <= hi;
        if (complete) {
            if (lane < k) {
                const bool real = my_i != SENT;
                out_cost[(int64_t)f * k + lane] = real ? unorder_bits(my_h) : INFINITY;
                out_cand[(int64_t)f * k + lane] = real ? (long long)my_i : -1;
            }
        } else if (lane < k) {
            // only the first and the last group can run past the unit's ends
            FCPP_ASSERT(g == 0 || g == n_groups - 1);
            const int which = g == 0 ? 0 : 1;
            out_e[(int64_t)blockIdx.x * per_child + which * k + lane] = make_ulonglong2(my_h, my_i);
        }
    }
}

// multi-GPU merge: one warp per field over the world x k entries of the ranks' sorted lists; each round takes the
// lowest (key, index) strictly above the previous round's
__global__ void __launch_bounds__(256) select_merge_kernel(const long long *__restrict__ g, int world, int n_fields,
                                                           int k, double *__restrict__ cost, long long *__restrict__ cand)
{
    const int64_t f = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (f >= n_fields) return;  // warp-uniform
    const int lane = threadIdx.x & 31;
    const int64_t fk = (int64_t)n_fields * k, row = 2 * fk;
    const long long *cost_row = g + f * k, *cand_row = g + fk + f * k;
    unsigned long long lh = 0, li = 0, my_h = SENT, my_i = SENT;
    const int n_items = world * k;
    for (int it = 0; it < k; ++it) {
        unsigned long long bh = SENT, bi = SENT;
        for (int i = lane; i < n_items; i += 32) {
            const int r = i / k, j = i - r * k;
            const long long idx = cand_row[r * row + j];
            const unsigned long long h = order_bits(__longlong_as_double(cost_row[r * row + j]));
            const unsigned long long u = (unsigned long long)idx;
            const bool fresh = idx >= 0 && (it == 0 || key_less(lh, li, h, u));
            if (fresh && key_less(h, u, bh, bi)) {
                bh = h;
                bi = u;
            }
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const unsigned long long oh = __shfl_xor_sync(0xffffffffu, bh, d);
            const unsigned long long oi = __shfl_xor_sync(0xffffffffu, bi, d);
            if (key_less(oh, oi, bh, bi)) {
                bh = oh;
                bi = oi;
            }
        }
        if (lane == it) {
            my_h = bh;
            my_i = bi;
        }
        lh = bh;  // once exhausted, (SENT, SENT): nothing is fresh any more
        li = bi;
    }
    if (lane < k) {
        const bool real = my_i != SENT;
        cost[f * k + lane] = real ? unorder_bits(my_h) : INFINITY;
        cand[f * k + lane] = real ? (long long)my_i : -1;
    }
}

// ---- per-field argmin: the plain selections (cost kind 0: len_main + len_head, 1: time_main + time_head).  As in
// select_keys, a candidate whose field lies outside [0, n_fields) is skipped ----
__device__ __forceinline__ double cand_cost(const fcpp_summary &s, int kind)
{
    return kind == 0 ? s.len_main + s.len_head : s.time_main + s.time_head;
}

__global__ void argmin_init(unsigned long long *key, int64_t *cand, int n_fields)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f < n_fields) {
        key[f] = ~0ull;
        cand[f] = 0x7fffffffffffffffll;
    }
}
// field of candidate c: the caller's array, or (factored candidate sets) the library's candidate record
__device__ __forceinline__ int cand_field_of(const int32_t *__restrict__ cf, const CandRec *__restrict__ recs, int64_t c)
{
    return cf ? cf[c] : recs[c].field;
}

__global__ void argmin_cost(const fcpp_summary *__restrict__ sm, const int32_t *__restrict__ cf,
                            const CandRec *__restrict__ recs, int64_t n, int n_fields, int kind, unsigned long long *key)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n || sm[c].status != 0) return;
    const int f = cand_field_of(cf, recs, c);
    if (f >= 0 && f < n_fields) atomicMin(&key[f], order_bits(cand_cost(sm[c], kind)));
}
__global__ void argmin_index(const fcpp_summary *__restrict__ sm, const int32_t *__restrict__ cf,
                             const CandRec *__restrict__ recs, int64_t n, int n_fields, int kind, int64_t base,
                             const unsigned long long *__restrict__ key, int64_t *cand)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n || sm[c].status != 0) return;
    const int f = cand_field_of(cf, recs, c);
    if (f >= 0 && f < n_fields && order_bits(cand_cost(sm[c], kind)) == key[f])
        atomicMin((long long *)&cand[f], (long long)(base + c));
}
__global__ void argmin_final(unsigned long long *key, int64_t *cand, int n_fields)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f < n_fields) {
        const unsigned long long k = key[f];
        double *out = reinterpret_cast<double *>(key);
        if (k == ~0ull) {
            out[f] = INFINITY;
            cand[f] = -1;
        } else {
            out[f] = unorder_bits(k);
        }
    }
}

// atomicMin(&table[f], v) for the active lanes of a warp (all 32 lanes call it): one atomic per warp when its active
// lanes share the field, else one per lane.  Values are unsigned-ordered (candidate indices are >= 0).
__device__ __forceinline__ void warp_field_min(unsigned long long *table, int f, unsigned long long v, bool active)
{
    const unsigned m = __ballot_sync(0xffffffffu, active);
    if (m == 0) return;
    const int f0 = __shfl_sync(0xffffffffu, f, __ffs(m) - 1);
    if (__all_sync(0xffffffffu, !active || f == f0)) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const unsigned long long o = __shfl_xor_sync(0xffffffffu, v, d);
            v = o < v ? o : v;
        }
        if ((threadIdx.x & 31) == 0) atomicMin(&table[f0], v);
    } else if (active) {
        atomicMin(&table[f], v);
    }
}

// the four phases in ONE CTA (small batches: four dependent launches cost more than the work)
constexpr int ARGMIN_SMALL_THREADS = 1024;
constexpr int ARGMIN_SMALL_MAX = 16384;  // candidates and fields
__global__ void __launch_bounds__(ARGMIN_SMALL_THREADS) argmin_small(const fcpp_summary *__restrict__ sm,
                                                                      const int32_t *__restrict__ cf,
                                                                      const CandRec *__restrict__ recs, int64_t n, int kind,
                                                                      int64_t base, unsigned long long *key, int64_t *cand,
                                                                      int n_fields)
{
    for (int f = threadIdx.x; f < n_fields; f += ARGMIN_SMALL_THREADS) {
        key[f] = ~0ull;
        cand[f] = 0x7fffffffffffffffll;
    }
    __threadfence();
    __syncthreads();
    // candidates of one field are contiguous (field-major order), so a warp usually holds ONE field: its minimum is
    // reduced by shuffles and costs one atomic instead of 32 on the same address (config 2: 4096 candidates, 1 field)
    for (int64_t c0 = 0; c0 < n; c0 += ARGMIN_SMALL_THREADS) {
        const int64_t c = c0 + threadIdx.x;
        bool on = c < n && sm[c].status == 0;
        const int f = on ? cand_field_of(cf, recs, c) : -1;
        on = on && f >= 0 && f < n_fields;
        warp_field_min(key, f, on ? order_bits(cand_cost(sm[c], kind)) : ~0ull, on);
    }
    __threadfence();
    __syncthreads();
    for (int64_t c0 = 0; c0 < n; c0 += ARGMIN_SMALL_THREADS) {
        const int64_t c = c0 + threadIdx.x;
        bool on = c < n && sm[c].status == 0;
        const int f = on ? cand_field_of(cf, recs, c) : -1;
        on = on && f >= 0 && f < n_fields && order_bits(cand_cost(sm[c], kind)) == __ldcg(&key[f]);
        warp_field_min(reinterpret_cast<unsigned long long *>(cand), on ? f : -1,
                       on ? (unsigned long long)(base + c) : ~0ull, on);
    }
    __threadfence();
    __syncthreads();
    for (int f = threadIdx.x; f < n_fields; f += ARGMIN_SMALL_THREADS) {
        const unsigned long long k = __ldcg(&key[f]);
        double *out = reinterpret_cast<double *>(key);
        if (k == ~0ull) {
            out[f] = INFINITY;
            cand[f] = -1;
        } else {
            out[f] = unorder_bits(k);
        }
    }
}

// multi-GPU merge at k = 1: one thread per field over the ranks' (cost, candidate) words (layout of
// select_merge_kernel); lowest cost wins, ties go to the lowest global candidate index, -1 = no candidate.  Kept next
// to select_merge_kernel because it is faster for few fields (DESIGN.md §3.8)
__global__ void argmin_merge_kernel(const long long *__restrict__ g, int world, int n_fields,
                                    double *__restrict__ best_cost, long long *__restrict__ best_cand)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_fields) return;
    double bc = INFINITY;
    long long bi = -1;
    for (int r = 0; r < world; ++r) {
        const long long *row = g + (int64_t)r * 2 * n_fields;
        const double c = __longlong_as_double(row[f]);
        const long long i = row[n_fields + f];
        if (i >= 0 && (bi < 0 || c < bc || (c == bc && i < bi))) {
            bc = c;
            bi = i;
        }
    }
    best_cost[f] = bc;
    best_cand[f] = bi;
}

// the cost kind of a plain selection (include/fcpp.h: its cost is L or T, bit for bit), -1 for any other
int plain_cost_kind(const fcpp_selection &s)
{
    if (s.top_k != 1 || s.max_boundary_viol >= 0 || s.max_obstacle_viol >= 0 || s.max_accel_viol >= 0 ||
        s.min_coverage >= 0.0 || s.w_boundary != 0.0 || s.w_obstacle != 0.0 || s.w_accel != 0.0 ||
        s.w_uncovered != 0.0)
        return -1;
    if (s.w_length == 1.0 && s.w_time == 0.0) return 0;
    if (s.w_length == 0.0 && s.w_time == 1.0) return 1;
    return -1;
}

cudaError_t launch_argmin(fcpp_handle *h, const fcpp_summary *d_summary, const int32_t *d_cand_field, int64_t n_cand,
                          int32_t n_fields, int cost_kind, int64_t cand_base, double *d_best_cost,
                          int64_t *d_best_cand, cudaStream_t st)
{
    unsigned long long *key = reinterpret_cast<unsigned long long *>(d_best_cost);
    if (n_cand <= ARGMIN_SMALL_MAX && n_fields <= ARGMIN_SMALL_MAX) {
        argmin_small<<<1, ARGMIN_SMALL_THREADS, 0, st>>>(d_summary, d_cand_field, h->d_rec, n_cand, cost_kind, cand_base,
                                                           key, d_best_cand, n_fields);
        h->launches++;
        return cudaGetLastError();
    }
    const int th = 256;
    const unsigned fb = (unsigned)((n_fields + th - 1) / th);
    argmin_init<<<fb, th, 0, st>>>(key, d_best_cand, n_fields);
    h->launches++;
    if (n_cand > 0) {
        const unsigned cb = (unsigned)((n_cand + th - 1) / th);
        argmin_cost<<<cb, th, 0, st>>>(d_summary, d_cand_field, h->d_rec, n_cand, n_fields, cost_kind, key);
        argmin_index<<<cb, th, 0, st>>>(d_summary, d_cand_field, h->d_rec, n_cand, n_fields, cost_kind, cand_base, key,
                                        d_best_cand);
        h->launches += 2;
    }
    argmin_final<<<fb, th, 0, st>>>(key, d_best_cand, n_fields);
    h->launches++;
    return cudaGetLastError();
}

size_t al256(size_t x) { return (x + 255) & ~size_t(255); }

}  // namespace

cudaError_t fcpp_launch_select(fcpp_handle *h, const fcpp_summary *d_summary, const int32_t *d_cand_field,
                               int64_t n_cand, int32_t n_fields, const fcpp_selection &sel, int64_t cand_base,
                               double *d_cost, int64_t *d_cand, cudaStream_t st)
{
    if (n_fields == 0) return cudaSuccess;
    const int kind = plain_cost_kind(sel);
    if (kind >= 0) return launch_argmin(h, d_summary, d_cand_field, n_cand, n_fields, kind, cand_base, d_cost, d_cand, st);
    const int k = sel.top_k;
    const int64_t n = n_cand, m = (int64_t)n_fields + 1;
    const int64_t scan_tiles = (m + SCAN_TILE - 1) / SCAN_TILE;
    const int64_t units0 = (n + SEL_TILE - 1) / SEL_TILE;
    // workspace: counts / segments [F+1], scan tile sums, keys [n], (field, rank) [n], sorted entries [n] + fields
    // [n], two generations of unit lists [units0][2][k] + their fields
    const size_t b_seg = al256(m * 8), b_tmp = al256(scan_tiles * 8), b_key = al256(n * 8), b_frk = al256(n * 8);
    const size_t b_ent = al256(n * 16), b_efld = al256(n * 4), b_uf = al256(units0 * 8),
                 b_ue = al256(units0 * 2 * k * 16);
    const size_t total = b_seg + b_tmp + b_key + b_frk + b_ent + b_efld + 2 * (b_uf + b_ue);
    if (total > h->sel_bytes) {
        if (h->d_sel) cudaFree(h->d_sel);
        h->d_sel = nullptr;
        h->sel_bytes = 0;
        const size_t cap = total + total / 8 + (1 << 20);
        cudaError_t e = cudaMalloc(&h->d_sel, cap);
        if (e != cudaSuccess) return e;
        h->sel_bytes = cap;
    }
    unsigned char *p = (unsigned char *)h->d_sel;
    unsigned long long *seg = (unsigned long long *)p;
    p += b_seg;
    long long *tmp = (long long *)p;
    p += b_tmp;
    unsigned long long *ckey = (unsigned long long *)p;
    p += b_key;
    int2 *frk = (int2 *)p;
    p += b_frk;
    ulonglong2 *ent = (ulonglong2 *)p;
    p += b_ent;
    int32_t *efld = (int32_t *)p;
    p += b_efld;
    int32_t *uf[2];
    ulonglong2 *ue[2];
    for (int b = 0; b < 2; ++b) {
        uf[b] = (int32_t *)p;
        p += b_uf;
        ue[b] = (ulonglong2 *)p;
        p += b_ue;
    }
    cudaError_t e = cudaMemsetAsync(seg, 0, m * 8, st);
    if (e != cudaSuccess) return e;
    const int64_t n_out = (int64_t)n_fields * k;
    const int64_t t1 = n > n_out ? n : n_out;
    select_keys<<<(unsigned)((t1 + 255) / 256), 256, 0, st>>>(d_summary, d_cand_field, h->d_rec, n, n_fields, sel, seg,
                                                             ckey, frk, d_cost, (long long *)d_cand, n_out);
    h->launches++;
    if (n == 0) return cudaGetLastError();
    select_scan_tiles<<<(unsigned)scan_tiles, SCAN_THREADS, 0, st>>>(seg, m, tmp);
    h->launches++;
    if (scan_tiles > 1) {
        select_scan_sums<<<1, SCAN_THREADS, 0, st>>>(tmp, scan_tiles);
        select_scan_add<<<(unsigned)scan_tiles, SCAN_THREADS, 0, st>>>(seg, m, tmp);
        h->launches += 2;
    }
    select_scatter<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(seg, ckey, frk, n, cand_base, ent, efld);
    h->launches++;
    int64_t units = units0, span = SEL_TILE;
    select_level<true><<<(unsigned)units, SEL_THREADS, 0, st>>>(seg, n_fields, k, span, 0, ent, efld, nullptr, nullptr,
                                                                uf[0], ue[0], d_cost, (long long *)d_cand);
    h->launches++;
    int cur = 0;
    while (units > 1) {
        units = (units + SEL_FANIN - 1) / SEL_FANIN;
        const int64_t child_span = span;
        span *= SEL_FANIN;
        select_level<false><<<(unsigned)units, SEL_THREADS, 0, st>>>(seg, n_fields, k, span, child_span, nullptr,
                                                                     nullptr, uf[cur], ue[cur], uf[cur ^ 1],
                                                                     ue[cur ^ 1], d_cost, (long long *)d_cand);
        h->launches++;
        cur ^= 1;
    }
    return cudaGetLastError();
}

cudaError_t fcpp_launch_select_merge(fcpp_handle *h, const int64_t *d_gathered, int world, int32_t n_fields, int k,
                                     double *d_cost, int64_t *d_cand, cudaStream_t st)
{
    if (n_fields == 0) return cudaSuccess;
    if (k == 1) {
        argmin_merge_kernel<<<(n_fields + 255) / 256, 256, 0, st>>>((const long long *)d_gathered, world, n_fields,
                                                                    d_cost, (long long *)d_cand);
        h->launches++;
        return cudaGetLastError();
    }
    const int64_t threads = (int64_t)n_fields * 32;
    select_merge_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>((const long long *)d_gathered, world,
                                                                          n_fields, k, d_cost, (long long *)d_cand);
    h->launches++;
    return cudaGetLastError();
}
