/* fcpp.h — C-ABI of libfcpp.so: the B200-native batched plan-generation-and-validation path
 * of the two-layer field coverage planner.
 *
 * The reference (qwagrox/field-coverage-path-planning) is pure Python and has NO FFI boundary
 * (SURVEY.md §8(b)); its boundary for this path is the Python class API.  This header is the
 * boundary a maintainer would bind from Python with ctypes (INTEGRATION.md shows the stub).
 * Each entry point cites the reference code it replaces; "mlp3" = multi_layer_planner_v3.py,
 * "ga" = genetic_algorithm_solver.py.
 *
 * Conventions
 *  - Plain C, no torch types.  Every buffer is CALLER-OWNED.  Pointers in fcpp_batch /
 *    fcpp_outputs and all `d_*` arguments are DEVICE pointers on the handle's device,
 *    contiguous, naturally aligned (16 B for double pairs).  The library owns only its
 *    handle workspace.
 *  - Every function returns 0 on success or a negative fcpp_status; it never throws, never
 *    exits.  fcpp_last_error(handle) gives the message.  Per-candidate geometric failures
 *    (mlp3:597 "headland too wide", mlp3:967-969 skipped loop) go to summary.status, not to
 *    the return code.
 *  - Work is enqueued on the cudaStream_t given (void* here so that the header needs no CUDA
 *    include) and is asynchronous; one handle per (device, stream), not re-entrant.
 *  - Units follow the reference: metres, km/h for speeds, m/s² for accelerations.
 *  - There is no CPU fallback: without a CUDA device fcpp_create fails.
 */
#ifndef FCPP_H
#define FCPP_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FCPP_ABI_VERSION 5

/* hard-coded sample counts of the reference (SURVEY.md §5) */
#define FCPP_UTURN_POINTS 20      /* mlp3:807  */
#define FCPP_CORNER_POINTS 15     /* mlp3:1046, :1589 */
#define FCPP_STRAIGHT_POINTS 20   /* mlp3:990  */
#define FCPP_MAX_LOOPS 16         /* K = ceil(R/W) (mlp3:916) supported up to this */
#define FCPP_POINTS_PER_LOOP 126   /* 1 + 4*20 + 3*15, mlp3:979-1007 */
#define FCPP_FIXED_UNIT 1e4       /* coverage lattice: 1e-4 m fixed point (DESIGN.md D5) */

typedef enum {
    FCPP_OK = 0,
    FCPP_ERR_INVALID = -1,   /* bad argument */
    FCPP_ERR_CUDA = -2,      /* CUDA runtime error (message in fcpp_last_error) */
    FCPP_ERR_NO_DEVICE = -3, /* no usable CUDA device: there is no CPU path */
    FCPP_ERR_TOO_LARGE = -4  /* a plan does not fit the on-chip staging (see DESIGN.md) */
} fcpp_status;

/* per-candidate status bits in fcpp_summary.status */
#define FCPP_CAND_OK 0
#define FCPP_CAND_INSET_EMPTY 1   /* mlp3:597-598 ValueError */
#define FCPP_CAND_LOOP_SKIPPED 2  /* mlp3:967-969 + :939 (vstack shape error) */
#define FCPP_CAND_TOO_MANY_LOOPS 4
#define FCPP_CAND_TOO_LARGE 8     /* the staged part exceeds the shared-memory capacity, or the plan's points the
                                     caller's path buffers (fcpp_outputs.path_capacity) */
#define FCPP_CAND_GRID_TOO_LARGE 16 /* a coverage grid does not fit the kernel's tiles; detail in the next two bits */
#define FCPP_CAND_CORNER_GRID_TOO_LARGE 32 /* ... the corner windows (A10); set together with 16 */
#define FCPP_CAND_BAND_GRID_TOO_LARGE 64   /* ... the headland band (A11); set together with 16 */

typedef struct fcpp_handle fcpp_handle;

/* A1 VehicleParams, mlp3:29-39 (min_turn_radius is per candidate: fcpp_batch.cand_R) */
typedef struct {
    double working_width;
    double max_work_speed_kmh;
    double max_headland_speed_kmh;
    double headland_turn_speed_kmh;
    double max_lateral_accel;
    double max_longitudinal_accel;
    double safety_factor;
    double reverse_speed_kmh; /* literal 2.5 at mlp3:1080 */
} fcpp_vehicle;

/* Inputs of one batch.  F fields, B candidates (field x heading x turn radius x start corner). */
typedef struct {
    fcpp_vehicle vehicle;
    /* ---- fields (A2 results are computed by the Python host in FP64, mlp3:109-343) ---- */
    int32_t n_fields;
    const double *field_verts;     /* [F][4][2] convex, CCW, vertex 0 = "lower-left" (mlp3:127-132) */
    const double *field_extent;    /* [F][2] field_length, field_width = bbox extents (mlp3:120-122) */
    const int32_t *field_flags;    /* [F] bit i: reverse fill allowed at corner i (angle>=60, mlp3:224-242) */
    /* obstacles (mlp3:600-609): polygons of field f are obs_poly_start[f] .. obs_poly_start[f+1] */
    const int32_t *obs_poly_start; /* [F+1]  (may be NULL when there are no obstacles at all) */
    const int32_t *obs_vert_start; /* [NP+1] vertices of polygon p are obs_vert_start[p] .. [p+1] */
    const double *obs_verts;       /* [NV][2] */
    const double *obs_moments;     /* [NP][3] area, area*cx, area*cy of the W/2 round buffer (D2) */
    int32_t max_obs_verts;         /* max over fields of the obstacle vertices of one field */
    int32_t max_obs_polys;         /* max over fields of the obstacle polygons of one field */
    /* ---- candidates ---- */
    int64_t n_cand;
    const int32_t *cand_field;     /* [B] field index */
    const double *cand_R;          /* [B] min_turn_radius = headland width (mlp3:295-310) */
    const double *cand_rot;        /* [B][4] cos(-a), sin(-a), cos(a), sin(a) of the swath heading a
                                      (host libm/numpy values; replaces mlp3:244-263, used :682-716) */
    const int32_t *cand_flags;     /* [B] bits 0-1 start corner (mlp3:397-399), bit 2 reverse_order,
                                      bit 3 start_from_right (mlp3:631-668), bit 4 rotated
                                      (|a| > 0.01, mlp3:686), bit 5 corner gap gate (mlp3:1070),
                                      bit 6: derive bits 2-3 from cand_start (mlp3:649-658) */
    const double *cand_start;      /* [B][2] start_point (mlp3:689-696) or NULL; read when bit 6 is set */
    /* ---- coverage raster ---- */
    double grid_h;                 /* headland-band cell size in m (0.1 default, 0.05 in config 5) */
    int32_t do_coverage;           /* 0: skip A10/A11 */
    int32_t max_points_hint;       /* >0: upper bound of points per plan known to the caller (e.g. from a
                                      previous fcpp_layout of the same batch): fcpp_layout then skips its
                                      8-byte readback + stream synchronisation and stays fully asynchronous */
    int32_t max_head_points_hint;  /* same for the headland part alone (n_head); used with max_points_hint */
    /* ---- turn model (SURVEY.md row A16; README.md:105-113 describes it, the reference has no code) ---- */
    int32_t turn_model;            /* 0: the reference's sampled circular arcs (mlp3:807-830, :1046-1062);
                                      1: clothoid -> arc -> clothoid turns with Fresnel integrals evaluated
                                      per sample point on the device (same sample counts, same layout) */
    int32_t cover_dedupe;     /* 1: coverage work with identical inputs is done once and shared — the corner windows
                               * (A10) of candidates with the same field and R (any start corner, any heading), the
                               * headland band (A11) of candidates with the same field, R and start corner (any
                               * heading); 0: every candidate is rasterised.  2: as 1, and the caller expects FEW
                               * representatives (a heading search: many headings per field): the coverage kernel then
                               * runs as a persistent grid over the list of coverage tasks instead of one (mostly
                               * empty) CTA per possible task.  Same integers either way. */
    double clothoid_share;         /* share of a turn's deflection spent on the two clothoids, (0, 1] */
    /* ---- factored candidate set (optional): cand_field == NULL selects it.  The candidates are the Cartesian
     * product field x heading x radius x start corner, field-major (the order of make_candidates): candidate c of
     * this batch is product index g = cand_first + c, field g / per, heading (g % per) / (NR' NC'), radius
     * (g / NC') % NR', corner g % NC' with per = NH' NR' NC' and N' = max(N, 1).  The host supplies only the AXES
     * (a few hundred values) — nothing per candidate is computed or copied by the host. ---- */
    int32_t n_ax_headings;           /* 0: the axis is absent — every candidate takes its field's own heading */
    int32_t n_ax_radii;              /* 0: absent — ax_default_radius */
    int32_t n_ax_corners;            /* 0: absent — start corner 0, no pass-order bits */
    int32_t ax_default_radius_flags; /* FCPP_FLAG_GAP_GATE or 0 for ax_default_radius */
    const double *ax_heading_rot;    /* [NH][4] cos(-a), sin(-a), cos(a), sin(a) (host libm / numpy values) */
    const int32_t *ax_heading_flags; /* [NH] FCPP_FLAG_ROTATED when |a| > 0.01 (mlp3:686), else 0 */
    const double *ax_radii;          /* [NR] */
    const int32_t *ax_radius_flags;  /* [NR] FCPP_FLAG_GAP_GATE when the corner gap gate holds for the radius (mlp3:1070) */
    const int32_t *ax_corners;       /* [NC] start corners 0..3; the pass-order bits follow mlp3:650-658 */
    const double *field_rot;         /* [F][4] the rotation of the field's own heading (edge 0, mlp3:244-263) */
    const int32_t *field_rot_flags;  /* [F] FCPP_FLAG_ROTATED or 0 for it */
    double ax_default_radius;
    int64_t cand_first;              /* product index of this batch's first candidate (contiguous multi-GPU shards) */
} fcpp_batch;

#define FCPP_TURN_ARC 0
#define FCPP_TURN_CLOTHOID 1
#define FCPP_TURN_OMEGA 2 /* BUILD-DEFINED main-work pattern (the reference only returns the label "Ω型跨行",
                             mlp3:312-320): same rows, swath ends and sample counts as the U pattern, but the rows are
                             visited in skip order (blocks of 2 s rows, s = ceil(2 R / W); lower and upper half of a
                             block alternate) and every 20-sample turn really connects the two swath ends — a half
                             circle of radius gap / 2 when the gap is >= 2 R, else the Ω (bulb) turn of three radius-R
                             arcs.  Headland turns stay the reference's arcs.  Parity unpinned (oracle restatement
                             only). */

#define FCPP_FLAG_CORNER_MASK 3
#define FCPP_FLAG_REVERSE_ORDER 4
#define FCPP_FLAG_START_FROM_RIGHT 8
#define FCPP_FLAG_ROTATED 16
#define FCPP_FLAG_GAP_GATE 32
#define FCPP_FLAG_START_POINT 64

/* One record per candidate (A8-A11, A13 + layout). 176 bytes. */
typedef struct {
    int32_t status;           /* FCPP_CAND_* bits */
    int32_t n_passes;         /* P, mlp3:739 */
    int32_t n_loops;          /* K, mlp3:916 */
    int32_t n_main;           /* points of main_work.path */
    int32_t n_head;           /* points of headland.path */
    int32_t n_rev[3];         /* reverse-fill points after the three loop-0 turns, mlp3:1214 */
    int32_t n_accel_viol;     /* mlp3:1401 */
    int32_t n_boundary_viol;  /* D3: points outside the field by > 1e-9 m */
    int32_t n_obstacle_viol;  /* D3: points inside an obstacle buffered by W/2 */
    int32_t corner_g;         /* int(2R/0.1), mlp3:1457 */
    int32_t corner_before[4]; /* covered lattice points, turn only, mlp3:1483 */
    int32_t corner_after[4];  /* turn + reverse fill, mlp3:1500 */
    int64_t cov_cells;        /* covered cells of the headland band (A11, D5) */
    int64_t cov_total;        /* cells of the headland band */
    double len_main;          /* m, mlp3:1290 on main_work.path */
    double len_head;
    double time_main;         /* s, mlp3:1298 with the ADJUSTED speeds (mlp3:423-431) */
    double time_head;
    double time_main_pre;     /* s, with the initial speeds (feeds the stale avg_speed_kmh, Q8) */
    double time_head_pre;
    double max_curvature;     /* mlp3:1396 */
    double max_lateral_accel; /* mlp3:1397 */
    double max_jump;          /* mlp3:1404-1406 */
    double reserved;
} fcpp_summary;

typedef struct {
    fcpp_summary *summary; /* [B] */
    /* optional materialised paths (all NULL = summary-only search mode) */
    const int64_t *offsets; /* [B+1] from fcpp_layout: candidate b owns points offsets[b]..offsets[b+1] */
    double *path_xy;        /* [total][2]  main_work.path then headland.path (mlp3:411) */
    double *speeds_kmh;     /* [total]     adjusted speeds (mlp3:415-420) */
    double *curvature;      /* [total] or NULL: kappa per point (0 at both ends) */
    int64_t path_capacity;  /* > 0: points the path buffers hold.  A caller that keeps buffers from an earlier batch
                               (no read-back of the layout's total) sets it: a plan whose points would not fit gets
                               status FCPP_CAND_TOO_LARGE instead of being written; 0 = unchecked */
    uint32_t *corner_bits;  /* optional: the occupancy bits of the four verification corner windows AFTER the reverse
                               fill (the 'grid' of mlp3:1503-1510).  Candidate b, corner c, lattice row j (g =
                               corner_g rows of rw = (g + 31) / 32 words): word corner_bits[b * corner_bits_stride
                               + (c * g + j) * rw + w], bit i & 31 of word i >> 5 = lattice point (i, j).  Written
                               only for candidates whose corner windows are rasterised (every candidate when
                               cover_dedupe = 0). */
    int64_t corner_bits_stride; /* words per candidate, >= 4 * g * rw of the largest window */
} fcpp_outputs;

int fcpp_abi_version(void);

/* Creates a handle on CUDA device `device`.  Fails with FCPP_ERR_NO_DEVICE when CUDA is absent. */
int fcpp_create(int device, fcpp_handle **out);
void fcpp_destroy(fcpp_handle *h);
const char *fcpp_last_error(const fcpp_handle *h);

/* Replaces the library's own libm tables of cos/sin(linspace(0,pi,20)) and
 * cos/sin(linspace(0,pi/2,15)) (mlp3:807-808, :1046-1047) by the host's (numpy's) values so
 * that device arcs are bit-identical to the host reference on the same machine.  Host pointers. */
int fcpp_set_trig_tables(fcpp_handle *h, const double *cos20, const double *sin20,
                         const double *cos15, const double *sin15);

/* FP64 integer-layout pass (P, K, n_rev, point counts: mlp3:739, :916, :1214) for every
 * candidate + exclusive prefix sum.  d_n_pts [B] int32 and d_offsets [B+1] int64 are device
 * buffers; either may be NULL.  Must precede fcpp_plan_batch for the same batch. */
int fcpp_layout(fcpp_handle *h, const fcpp_batch *batch, int32_t *d_n_pts, int64_t *d_offsets,
                void *stream);

/* The hot path: path sampling (mlp3:591-1288), speed planning (mlp3:467-589), kinematic and
 * geofence validation (mlp3:1373-1424 + D3), path metrics (mlp3:1290-1311) and coverage
 * rasterisation (mlp3:1357-1371, :1426-1578) for all candidates. */
int fcpp_plan_batch(fcpp_handle *h, const fcpp_batch *batch, const fcpp_outputs *out, void *stream);

/* ---- per-field top-k under a constraint-aware cost (DESIGN.md §3.8) ---- */
#define FCPP_SELECT_MAX_K 32

/* A candidate is ELIGIBLE when status == 0, every limit that is set holds (n_*_viol <= max_*), and, with
 * min_coverage set, cov_total > 0 and (double)cov_cells >= min_coverage * (double)cov_total.  Its cost, in FP64
 * left to right (the library is built with -fmad=false):
 *   L = len_main + len_head;  T = time_main + time_head;  U = (double)(cov_total - cov_cells) * cell_area;
 *   cost = w_length*L + w_time*T + w_boundary*n_boundary_viol + w_obstacle*n_obstacle_viol
 *        + w_accel*n_accel_viol + w_uncovered*U
 * A PLAIN selection: top_k = 1, no limit set, and the weights (w_length = 1, every other 0) or (w_time = 1, every
 * other 0).  Its cost is L or T exactly (for finite L, T >= 0): the per-field argmin of the length or of the time. */
typedef struct {
    double w_length, w_time, w_boundary, w_obstacle, w_accel, w_uncovered; /* finite, >= 0 */
    double cell_area;          /* m^2 of a headland-band cell: grid_h * grid_h */
    double min_coverage;       /* in [0, 1]; < 0: no limit */
    int32_t max_boundary_viol; /* < 0: no limit */
    int32_t max_obstacle_viol; /* < 0: no limit */
    int32_t max_accel_viol;    /* < 0: no limit */
    int32_t top_k;             /* 1 .. FCPP_SELECT_MAX_K */
} fcpp_selection;

/* Per field, the eligible candidates ranked by (cost, candidate index) ascending, the first top_k of them:
 * d_cost [F][k] double (+inf where fewer than k are eligible), d_cand [F][k] int64 global indices (cand_base added;
 * -1 where none).  Candidates whose field lies outside [0, n_fields) are skipped.  d_cand_field [n_cand] is the field
 * of each candidate; it may be NULL right after fcpp_plan_batch of the same batch on this handle: the fields are
 * then taken from the library's candidate records (factored candidate sets have no cand_field array).
 * Exact and deterministic for any order of the candidates' fields; scratch space is the handle's workspace.
 * A plain selection runs the argmin kernels: one launch up to 16 384 candidates and fields, else four (two without
 * candidates), with no workspace; any other selection runs the ranking pipeline (DESIGN.md §3.8). */
int fcpp_field_select(fcpp_handle *h, const fcpp_summary *d_summary, const int32_t *d_cand_field, int64_t n_cand,
                      int32_t n_fields, const fcpp_selection *sel, int64_t cand_base, double *d_cost,
                      int64_t *d_cand, void *stream);

/* Multi-GPU merge of the ranks' rankings: d_gathered [world][2*F*k] 8-byte words = every rank's d_cost [F][k] (as
 * double bits) then d_cand [F][k], e.g. ONE all-gather of the two arrays laid out back to back.  Per field the k
 * lowest (cost, index) of the union; +inf / -1 pad.  The winners' records of the ranking: fcpp_winner_records
 * with n_fields = F * k on the flattened d_cand. */
int fcpp_field_select_merge(fcpp_handle *h, const int64_t *d_gathered, int32_t world, int32_t n_fields, int32_t k,
                            double *d_cost, int64_t *d_cand, void *stream);

/* Multi-GPU: this rank's contribution to the exchange of the winners' records after the merge: d_out [F][176 bytes]
 * = the summary record of every field whose global winner d_best_cand[f] lies in this rank's candidate range
 * [cand_lo, cand_hi) (d_summary holds that range), zeros for every other field — summing the ranks' buffers as
 * 32-bit words (one all-reduce) gives every rank every winner's record. */
int fcpp_winner_records(fcpp_handle *h, const fcpp_summary *d_summary, int64_t cand_lo, int64_t cand_hi,
                        const int64_t *d_best_cand, int32_t n_fields, void *d_out, void *stream);

/* *d_count = number of candidates whose status has a bit of `mask` (e.g. FCPP_CAND_TOO_LARGE |
 * FCPP_CAND_GRID_TOO_LARGE: a caller that sized a launch from hints of an earlier batch learns on the device —
 * and, summed over the ranks, collectively — whether the sizes were sufficient). */
int fcpp_status_count(fcpp_handle *h, const fcpp_summary *d_summary, int64_t n_cand, int32_t mask, int32_t *d_count,
                      void *stream);

/* Generic A7/A8/A13 on caller-supplied paths (ragged batch, path p = points offsets[p]..offsets[p+1]):
 * speed planning mlp3:467-589 (d_speeds_out may alias d_speeds_in), curvature verification
 * mlp3:1373-1424 and length/time mlp3:1290-1311 into d_summary (fields n_accel_viol, max_*,
 * len_main, time_main, time_main_pre; the split point n_main = whole path).
 * do_speed_plan = 0 verifies the given speeds without adjusting them.
 * max_path_len sizes the per-path staging: paths of up to max_path_len rounded up to a multiple of 256 points (0: up
 * to the largest shared-memory staging, ~9500 points on a B200) are processed; a longer path gets status
 * FCPP_CAND_TOO_LARGE, zero lengths, times, counts and maxima, and no speeds or curvature written. */
int fcpp_speed_verify(fcpp_handle *h, const fcpp_vehicle *veh, const double *d_path_xy,
                      const double *d_speeds_in, const int64_t *d_offsets, int64_t n_paths,
                      int64_t max_path_len, int do_speed_plan, double *d_speeds_out,
                      double *d_curvature, fcpp_summary *d_summary, void *stream);

/* ---- segment-level obstacle sweep (DESIGN.md §3.9) ----
 * The obstacle region O of a field is the set of points D3 counts in n_obstacle_viol: inside an obstacle polygon
 * (even-odd crossing) or at distance < r from one of its edges.  For every segment a -> b of a path, m = metres of
 * the segment inside O (exact up to rounding: the segment is cut at the boundaries of the edges' r-capsules and each
 * piece classified at its midpoint; oracle/sweep.py states the rule).  Per candidate or path: the segments with
 * m > 0 and the sum of m (left to right in segment order) of main_work.path and of headland.path; the segment
 * from the last main point to the first headland point belongs to neither.  24 bytes. */
typedef struct {
    int32_t n_seg_main, n_seg_head; /* segments with m > 0 */
    double len_main, len_head;      /* m, summed left to right */
} fcpp_sweep;

/* The sweep of every candidate of `batch` with r = working_width / 2, from the library's candidate records: must
 * follow fcpp_layout of the same batch (same arrays, same stream) on this handle — before or after its
 * fcpp_plan_batch — else FCPP_ERR_INVALID.  d_out [B].  Candidates whose layout failed (status != 0) and fields
 * without obstacles (or a batch without obstacle tables) get zeros. */
int fcpp_obstacle_sweep(fcpp_handle *h, const fcpp_batch *batch, fcpp_sweep *d_out, void *stream);

/* The sweep of caller-supplied paths (ragged batch, path p = points d_offsets[p] .. d_offsets[p+1]) against ONE
 * obstacle set (polygon q = vertices d_obs_vert_start[q] .. [q+1] of d_obs_verts [NV][2]).  d_n_main [n_paths] (or
 * NULL: the whole path is main work) splits path p into main_work (its first n_main points) and headland.  d_out
 * [n_paths]. */
int fcpp_obstacle_sweep_paths(fcpp_handle *h, const double *d_path_xy, const int64_t *d_offsets, int64_t n_paths,
                              const int32_t *d_n_main, const int32_t *d_obs_vert_start, const double *d_obs_verts,
                              int32_t n_polys, double radius, fcpp_sweep *d_out, void *stream);

/* ---- whole-field and headland-band coverage of polylines in device memory (DESIGN.md §3.10) ----
 * The lattice is A11's: cell centres q(bbox_min) + H/2 + (i H, j H) of the path's field, H = q(grid_h),
 * q(x) = rint(x 1e4).  A cell is covered by a set of segments iff its centre lies strictly within r = W/2 of one of
 * them (the exact 128-bit predicate, D2/D5).  A path is main work (its first n_main points) then headland; the
 * segment from the last main point to the first headland point belongs to neither layer.
 *   field cells: centre inside-or-on the field quad; field_cells counts those covered by the segments of BOTH layers.
 *   band cells: A11's headland band, the field cells not inside-or-on the mitred inset of the field by the headland
 *     width (D1); band_cells counts those covered by the HEADLAND layer only (as fcpp_summary.cov_cells).  An inset
 *     that is empty or has |area| < 1 m^2 makes the band the whole field; a headland width <= 0 means no band (both
 *     band counts 0).
 *   n_boundary_viol / n_obstacle_viol: D3 over every point of the path (the plan kernel's point test).
 * status: FCPP_CAND_GRID_TOO_LARGE | FCPP_CAND_BAND_GRID_TOO_LARGE when the field's lattice does not fit (a lattice
 * row longer than the 32 KB tile, or an extent of 2^30 units); the four cell counts are then 0.
 * FCPP_PATH_OUT_OF_RANGE when a point lies 2^30 lattice units (~107 km) or more from the field's lattice origin, or
 * the path's field index is outside [0, n_fields): every count is 0.  Points are never clamped.
 * The counts are sums of integer atomics over row slabs: deterministic.  48 bytes. */
#define FCPP_PATH_OUT_OF_RANGE 128
typedef struct {
    int32_t status;
    int32_t n_boundary_viol, n_obstacle_viol;
    int32_t reserved;
    int64_t band_total, band_cells;   /* cells of the headland band; of those, covered by the headland layer */
    int64_t field_total, field_cells; /* cells of the field; of those, covered by either layer */
} fcpp_path_cover;

/* Coverage and D3 counts of caller-supplied paths (ragged batch, path p = points d_offsets[p] .. d_offsets[p+1] of
 * d_path_xy [N][2]).  d_n_main [n_paths] splits path p into main work and headland; NULL means n_main = 0: the whole
 * path is the headland layer and counts for both the band and the field.  d_path_field [n_paths] is each path's
 * field (d_field_verts [n_fields][4][2], convex CCW), d_headland_width [n_paths] its headland width in m.  Obstacles
 * as in fcpp_batch, per field (d_obs_poly_start [n_fields + 1], or NULL: none).  radius = W/2; grid_h an even
 * multiple of 1e-4 m.  d_out [n_paths].  Asynchronous: no read-back. */
int fcpp_path_coverage(fcpp_handle *h, const double *d_path_xy, const int64_t *d_offsets, int64_t n_paths,
                       const int32_t *d_n_main, const int32_t *d_path_field, const double *d_headland_width,
                       int32_t n_fields, const double *d_field_verts, const int32_t *d_obs_poly_start,
                       const int32_t *d_obs_vert_start, const double *d_obs_verts, double radius, double grid_h,
                       fcpp_path_cover *d_out, void *stream);

/* The same for the materialised plans of the last fcpp_plan_batch of `batch` on this handle (outputs->path_xy and
 * outputs->offsets are required, else FCPP_ERR_INVALID; the candidate records must be this batch's, as for
 * fcpp_obstacle_sweep): field, headland width R and n_main from the candidate records, r = working_width / 2 and
 * the batch's grid_h and obstacles.  Candidates whose layout failed, that have no points, or whose paths were not
 * written (summary status FCPP_CAND_TOO_LARGE) get zero records.  d_out [B]. */
int fcpp_plan_coverage(fcpp_handle *h, const fcpp_batch *batch, const fcpp_outputs *outputs, fcpp_path_cover *d_out,
                       void *stream);

/* Generic A10 window raster (mlp3:1426-1510): ORs the W/2 round buffer of a polyline into a
 * g x g lattice-point window (bit (j*g+i) of d_bits, row-major, 32-bit words, ceil(g*g/32) words,
 * caller-zeroed or carrying an earlier cover) and writes the number of set bits to d_count.
 * Range contract (as fcpp_path_coverage): FCPP_ERR_INVALID when g * q(h_cell) >= 2^30 lattice units; when a point
 * lies 2^30 units (~107 km) or more from q(origin) in x or y, *d_count = -1 and no bit of d_bits changes.  Points
 * are never clamped. */
int fcpp_raster_window(fcpp_handle *h, const double *d_path_xy, int32_t n_pts, double radius,
                       double origin_x, double origin_y, double h_cell, int32_t g,
                       uint32_t *d_bits, int64_t *d_count, void *stream);

/* A12 closed-tour lengths: d_out[p] = sum_i D[r_i, r_(i+1) mod n] accumulated left to right in
 * FP64 exactly as ga:174-181; d_fitness (optional) = 1/(d + 1e-6) (ga:168-172).
 * D is n x n row-major FP64 (multi_field_planner.py:263-288), pop is pop_size x n int32. */
int fcpp_tour_lengths(fcpp_handle *h, const double *d_D, int32_t n, const int32_t *d_pop,
                      int64_t pop_size, double *d_out, double *d_fitness, void *stream);


/* ---------------------------------------------------------------------------------------------
 * Multi-field glue (SURVEY.md §8(f) N2; "mfp" = multi_field_planner.py)
 * ------------------------------------------------------------------------------------------- */

/* mfp:263-288 _calculate_distance_matrix: d_D[i*n+j] = ||pos_i - pos_j|| (0 on the diagonal);
 * d_pos [n][2], row 0 = depot, row f+1 = centroid of field f. */
int fcpp_distance_matrix(fcpp_handle *h, const double *d_pos, int32_t n, double *d_D, void *stream);

/* mfp:290-320 _find_best_connection for EVERY ordered pair of nodes (node 0 = depot, node f+1 = field
 * f whose four vertices d_field_verts[f][4][2] are its exit and entry points, mfp:123-141):
 * d_C[a*(F+1)+b] = shortest exit-vertex -> entry-vertex distance, d_arg = from_index*4 + to_index of
 * the FIRST minimum in the reference's loop order (strict '<', mfp:308-311). */
int fcpp_connection_matrix(fcpp_handle *h, const double *d_field_verts, int32_t n_fields, double depot_x,
                           double depot_y, double *d_C, int32_t *d_arg, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Multi-vehicle split (SURVEY.md §8(f) N4; "mvp" = multi_vehicle_planner.py)
 * ------------------------------------------------------------------------------------------- */

/* mvp:186-209 _cluster_fields = sklearn.cluster.KMeans(n_clusters=V, random_state=42).fit_predict(centroids):
 * the Lloyd iteration of scikit-learn's `_kmeans_single_lloyd` on 2-D points, batched — problem p owns the points
 * d_xy[d_pt_start[p] .. d_pt_start[p+1]) and the centres d_centers[d_center_start[p] .. d_center_start[p+1])
 * (k-means++ seeds in, final centres out; max_clusters = the largest centre count of a problem, <= 4096).  Per
 * problem: data centred on its mean; E step = first minimum of ||c||^2 - 2 x.c; M step = member mean, an empty
 * cluster takes the point farthest from its centre; stop on unchanged labels, or when the summed squared centre
 * shift <= tol * mean per-axis variance (sklearn: tol = 1e-4), or after max_iter (sklearn: 300) iterations, then
 * one more E step unless the labels were unchanged.  d_labels [sum n] int32, d_n_iter [P], d_inertia [P]
 * (sum of squared distances to the assigned centre).  One CTA per problem, deterministic reductions. */
int fcpp_kmeans_lloyd(fcpp_handle *h, int32_t n_problems, const int64_t *d_pt_start, const double *d_xy,
                      const int64_t *d_center_start, int32_t max_clusters, double *d_centers, int32_t *d_labels,
                      int32_t max_iter, double tol, int32_t *d_n_iter, double *d_inertia, void *stream);

/* `TSPSolver.solve(distance_matrix)` — imported by multi_field_planner.py:176 and multi_vehicle_planner.py:131 from
 * `multi_field_planner_v37`, a module the reference does not ship.  BUILD-DEFINED (no reference source): nearest-
 * neighbour tour from node 0, then best-improvement 2-opt on the closed tour (delta = (D[a][c] + D[b][d]) -
 * (D[a][b] + D[c][d]) for the tour edges (a, b), (c, d); the lowest delta < -1e-9 is applied, ties to the lowest
 * edge pair; node 0 stays first) until no move improves or max_iter moves were made.  Batched: problem p owns the
 * n_p x n_p symmetric FP64 matrix at d_D + d_mat_start[p] (n_p = d_node_start[p+1] - d_node_start[p] <= max_nodes
 * <= 16384) and writes its tour to d_tours + d_node_start[p], the closed-tour length (left-to-right FP64 sum, as
 * fcpp_tour_lengths) to d_lengths[p] and the number of moves to d_iters[p].  One CTA per problem, deterministic. */
int fcpp_tsp_two_opt(fcpp_handle *h, int32_t n_problems, const int64_t *d_mat_start, const double *d_D,
                     const int64_t *d_node_start, int32_t max_nodes, int32_t *d_tours, double *d_lengths,
                     int32_t *d_iters, int32_t max_iter, void *stream);

/* ---------------------------------------------------------------------------------------------
 * GA evolution on the device (SURVEY.md §8(f) N1; "ga" = genetic_algorithm_solver.py)
 * ------------------------------------------------------------------------------------------- */
#define FCPP_GA_MAX_TOURNAMENT 16
#define FCPP_GA_TRACE_INTS 48 /* per offspring pair: [0] parent A, [1] parent B (indices into the old
                                 population), [2] crossed, [3] cut a, [4] cut b, [5..7] child 1 mutated / i / j,
                                 [8..10] child 2 mutated / i / j, [11] tournament size,
                                 [12..28) tournament draws of A, [28..44) tournament draws of B */

/* GAConfig, ga:20-29, + the seed of the counter-based generator (the reference uses Python's
 * unseeded global `random`; parity of whole runs is statistical, of the operators exact) */
typedef struct {
    int32_t population_size;
    int32_t max_generations;
    double crossover_rate;
    double mutation_rate;
    int32_t elite_size;
    int32_t tournament_size;       /* 1 .. FCPP_GA_MAX_TOURNAMENT and <= population (random.sample, ga:189) */
    int32_t convergence_threshold;
    int32_t check_every;           /* generations between host polls of the convergence flag (0: 16) */
    uint64_t seed;
} fcpp_ga_config;

/* stats of ga:122-127 */
typedef struct {
    int32_t generations;
    int32_t convergence_gen;
    int32_t final_population; /* an odd population grows by one individual in its first generation (ga:205) */
    int32_t reserved;
    double best_distance;
    double best_fitness;
} fcpp_ga_result;

/* ga:137-166: 2*(population_size/2) individuals x n into d_pop (int32, row-major). */
int fcpp_ga_init_population(fcpp_handle *h, const fcpp_ga_config *cfg, int32_t n, int32_t *d_pop, void *stream);

/* Individuals after one generation over m_in individuals (python slicing of ga:262-266 included). */
int32_t fcpp_ga_next_size(const fcpp_ga_config *cfg, int32_t m_in);

/* One generation ga:78-88: tournament selection, OX crossover, swap mutation, elitism.  d_pop_in
 * [m_in][n] + d_fitness [m_in] -> d_pop_out [fcpp_ga_next_size][n].  d_trace (optional)
 * [(m_in+1)/2][FCPP_GA_TRACE_INTS] receives every random decision taken. */
int fcpp_ga_generation(fcpp_handle *h, const fcpp_ga_config *cfg, int32_t generation, int32_t n,
                       const int32_t *d_pop_in, const double *d_fitness, int32_t m_in, int32_t *d_pop_out,
                       int32_t *d_trace, void *stream);

/* solve(), ga:44-135, entirely on the device: initial population (d_pop_init [population_size][n] or
 * NULL = fcpp_ga_init_population), fitness, evolution loop with best tracking and the
 * convergence stop, final rotation to node 0.  d_best_route [n] int32; d_history (optional)
 * [max_generations][2] = best_fitness_history / avg_fitness_history.  Synchronises the stream
 * every check_every generations and before returning (host_result is host memory). */
int fcpp_ga_solve(fcpp_handle *h, const fcpp_ga_config *cfg, const double *d_D, int32_t n,
                  const int32_t *d_pop_init, int32_t *d_best_route, double *d_history,
                  fcpp_ga_result *host_result, void *stream);

/* Number of kernels this handle has launched so far (bench.py's gpu_launches). */
int64_t fcpp_launch_count(const fcpp_handle *h);

/* Longest plan / longest headland path (points) seen by the last synchronous fcpp_layout
 * (feed max_points_hint / max_head_points_hint). */
int32_t fcpp_last_max_points(const fcpp_handle *h);
int32_t fcpp_last_max_head_points(const fcpp_handle *h);
/* offsets[n_cand] of the last fcpp_layout that wrote offsets without size hints (it is read back in the
 * same synchronisation as the two maxima); -1 if unknown.  Sizes the path buffers without a second copy. */
int64_t fcpp_last_total_points(const fcpp_handle *h);

/* Per-kernel device times.  With profiling on, every fcpp_plan_batch brackets its kernels with
 * CUDA events on the launching stream; fcpp_kernel_times (call after synchronising the stream)
 * returns the milliseconds of the last call: [0] layout (+scan), [1] plan, [2] coverage. */
int fcpp_set_profiling(fcpp_handle *h, int on);
int fcpp_kernel_times(fcpp_handle *h, float *ms3);

/* Diagnostics: coverage-kernel evaluation mode of the following fcpp_plan_batch calls.  0 = automatic
 * (default): the headland band of a field whose straights are axis-aligned is evaluated "zoned"
 * (bitmap around the corners, closed form elsewhere), any other field row-tiled.  Bit 0 set = always
 * row-tiled.  Bit 1 set = no coverage de-duplication (by default candidates whose coverage inputs are
 * identical — same field, R, start corner; e.g. the headings of a heading search — are rasterised once
 * and share the counts).  Bits 6 / 7 override fcpp_batch.cover_dedupe's choice between one coverage CTA per
 * listed task (bit 6) and the persistent grid over the task list (bit 7).  Any other bit is
 * FCPP_ERR_INVALID and leaves the mode unchanged.  All modes give identical results (tests/test_gpu_parity.py
 * compares them). */
int fcpp_set_cover_mode(fcpp_handle *h, int mode);

#ifdef __cplusplus
}
#endif
#endif /* FCPP_H */
