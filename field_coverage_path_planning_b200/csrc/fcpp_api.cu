// fcpp_api.cu — the extern "C" boundary of libfcpp.so (declared in include/fcpp.h).
// No exceptions cross this boundary; every CUDA error is turned into a negative status and a
// message retrievable with fcpp_last_error().
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "fcpp_internal.cuh"

namespace {

int fail(fcpp_handle *h, int code, const char *fmt, ...)
{
    if (h) {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(h->err, sizeof(h->err), fmt, ap);
        va_end(ap);
    }
    return code;
}

int cuda_fail(fcpp_handle *h, cudaError_t e, const char *what)
{
    return fail(h, FCPP_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
}

// numpy.linspace(0, stop, n): i*step for i < n-1, exactly `stop` at the end
void host_tables(TrigTables &t)
{
    const double pi = 3.141592653589793;
    for (int i = 0; i < FCPP_UTURN_POINTS; ++i) {
        const double a = (i == FCPP_UTURN_POINTS - 1) ? pi : i * (pi / (FCPP_UTURN_POINTS - 1));
        t.cos20[i] = cos(a);
        t.sin20[i] = sin(a);
    }
    for (int i = 0; i < FCPP_CORNER_POINTS; ++i) {
        const double a = (i == FCPP_CORNER_POINTS - 1) ? pi / 2 : i * ((pi / 2) / (FCPP_CORNER_POINTS - 1));
        t.cos15[i] = cos(a);
        t.sin15[i] = sin(a);
    }
}

int ensure_workspace(fcpp_handle *h, int64_t n_cand)
{
    if (n_cand > h->rec_cap) {
        if (h->d_rec) cudaFree(h->d_rec);
        h->d_rec = nullptr;
        h->rec_cap = 0;
        int64_t cap = n_cand + n_cand / 8 + 1024;
        cudaError_t e = cudaMalloc((void **)&h->d_rec, (size_t)cap * sizeof(CandRec));
        if (e != cudaSuccess) return cuda_fail(h, e, "cudaMalloc(candidate records)");
        h->rec_cap = cap;
    }
    const int64_t tiles = n_cand / 4096 + 2;
    if (tiles > h->scan_tmp_cap) {
        if (h->d_scan_tmp) cudaFree(h->d_scan_tmp);
        h->d_scan_tmp = nullptr;
        h->scan_tmp_cap = 0;
        cudaError_t e = cudaMalloc(&h->d_scan_tmp, (size_t)(tiles + 1024) * sizeof(int64_t));
        if (e != cudaSuccess) return cuda_fail(h, e, "cudaMalloc(scan workspace)");
        h->scan_tmp_cap = tiles + 1024;
    }
    return FCPP_OK;
}

int check_batch(fcpp_handle *h, const fcpp_batch *b)
{
    if (!h) return FCPP_ERR_INVALID;
    if (!b) return fail(h, FCPP_ERR_INVALID, "batch is NULL");
    if (b->n_cand < 0 || b->n_fields < 0) return fail(h, FCPP_ERR_INVALID, "negative sizes");
    if (b->n_cand > 0 && (!b->field_verts || !b->field_extent || !b->field_flags))
        return fail(h, FCPP_ERR_INVALID, "a required batch pointer is NULL");
    if (b->n_cand > 0 && b->cand_field && (!b->cand_R || !b->cand_rot || !b->cand_flags))
        return fail(h, FCPP_ERR_INVALID, "a required candidate array is NULL");
    if (b->n_cand > 0 && !b->cand_field) {  // factored candidate set
        if (b->n_ax_headings < 0 || b->n_ax_radii < 0 || b->n_ax_corners < 0 || b->cand_first < 0)
            return fail(h, FCPP_ERR_INVALID, "negative axis size");
        if ((b->n_ax_headings > 0 && (!b->ax_heading_rot || !b->ax_heading_flags)) ||
            (b->n_ax_headings == 0 && (!b->field_rot || !b->field_rot_flags)) ||
            (b->n_ax_radii > 0 && (!b->ax_radii || !b->ax_radius_flags)) || (b->n_ax_corners > 0 && !b->ax_corners))
            return fail(h, FCPP_ERR_INVALID, "a candidate axis array is NULL");
        const int64_t per = (int64_t)(b->n_ax_headings > 0 ? b->n_ax_headings : 1) *
                            (b->n_ax_radii > 0 ? b->n_ax_radii : 1) * (b->n_ax_corners > 0 ? b->n_ax_corners : 1);
        if (b->cand_first + b->n_cand > (int64_t)b->n_fields * per)
            return fail(h, FCPP_ERR_INVALID, "candidate range beyond the product of the axes");
        if (b->cand_start) return fail(h, FCPP_ERR_INVALID, "start points need explicit candidate arrays");
    }
    if (b->obs_poly_start && (!b->obs_vert_start || !b->obs_verts || !b->obs_moments))
        return fail(h, FCPP_ERR_INVALID, "obstacle tables are incomplete");
    if (!(b->vehicle.working_width > 0.0)) return fail(h, FCPP_ERR_INVALID, "working_width must be > 0");
    if (b->turn_model != FCPP_TURN_ARC && b->turn_model != FCPP_TURN_CLOTHOID && b->turn_model != FCPP_TURN_OMEGA)
        return fail(h, FCPP_ERR_INVALID, "turn_model must be 0 (arc), 1 (clothoid) or 2 (omega skip-row pattern)");
    if (b->turn_model == FCPP_TURN_CLOTHOID && !(b->clothoid_share > 0.0 && b->clothoid_share <= 1.0))
        return fail(h, FCPP_ERR_INVALID, "clothoid_share must be in (0, 1]");
    if (b->do_coverage) {
        const double hq = b->grid_h * FCPP_FIXED_UNIT;
        const long long H = llrint(hq);
        if (H < 2 || (H & 1) || fabs(hq - (double)H) > 1e-6)
            return fail(h, FCPP_ERR_INVALID, "grid_h must be an even multiple of 1e-4 m (got %g)", b->grid_h);
    }
    return FCPP_OK;
}

}  // namespace

extern "C" {

int fcpp_abi_version(void) { return FCPP_ABI_VERSION; }

int fcpp_create(int device, fcpp_handle **out)
{
    if (!out) return FCPP_ERR_INVALID;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) {
        cudaGetLastError();
        return FCPP_ERR_NO_DEVICE;
    }
    if (cudaSetDevice(device) != cudaSuccess) return FCPP_ERR_NO_DEVICE;
    fcpp_handle *h = (fcpp_handle *)calloc(1, sizeof(fcpp_handle));
    if (!h) return FCPP_ERR_INVALID;
    h->device = device;
    cudaDeviceGetAttribute(&h->max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device);
    cudaDeviceGetAttribute(&h->max_smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, device);
    TrigTables t;
    host_tables(t);
    cudaError_t e = cudaMalloc((void **)&h->d_trig, sizeof(TrigTables));
    if (e == cudaSuccess) e = cudaMemcpy(h->d_trig, &t, sizeof(t), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc((void **)&h->d_maxn, 2 * sizeof(int));
    if (e == cudaSuccess) e = cudaMallocHost((void **)&h->h_maxn, 4 * sizeof(int));  // + int64 total points
    if (e != cudaSuccess) {
        fcpp_destroy(h);
        return FCPP_ERR_CUDA;
    }
    *out = h;
    return FCPP_OK;
}

void fcpp_destroy(fcpp_handle *h)
{
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->d_trig) cudaFree(h->d_trig);
    if (h->d_rec) cudaFree(h->d_rec);
    if (h->d_scan_tmp) cudaFree(h->d_scan_tmp);
    if (h->d_big) cudaFree(h->d_big);
    if (h->d_maxn) cudaFree(h->d_maxn);
    if (h->h_maxn) cudaFreeHost(h->h_maxn);
    if (h->d_ga) cudaFree(h->d_ga);
    if (h->d_dedupe) cudaFree(h->d_dedupe);
    if (h->d_sel) cudaFree(h->d_sel);
    if (h->d_pcov) cudaFree(h->d_pcov);
    if (h->h_ga_state) cudaFreeHost(h->h_ga_state);
    if (h->ga_stream) cudaStreamDestroy(h->ga_stream);
    for (int k = 0; k < 4; ++k)
        if (h->ev[k]) cudaEventDestroy(h->ev[k]);
    free(h);
}

const char *fcpp_last_error(const fcpp_handle *h) { return h ? h->err : "invalid handle"; }

int64_t fcpp_launch_count(const fcpp_handle *h) { return h ? h->launches : 0; }

int32_t fcpp_last_max_points(const fcpp_handle *h) { return h ? h->last_maxn : 0; }
int32_t fcpp_last_max_head_points(const fcpp_handle *h) { return h ? h->last_maxhead : 0; }
int64_t fcpp_last_total_points(const fcpp_handle *h) { return h ? h->last_total : -1; }

int fcpp_set_cover_mode(fcpp_handle *h, int mode)
{
    constexpr int known = 1 | 2 | 64 | 128;  // the bits documented in fcpp.h
    if (!h) return FCPP_ERR_INVALID;
    if (mode & ~known) return fail(h, FCPP_ERR_INVALID, "fcpp_set_cover_mode: unknown mode bits 0x%x", mode & ~known);
    h->cover_mode = mode;
    return FCPP_OK;
}

int fcpp_set_profiling(fcpp_handle *h, int on)
{
    if (!h) return FCPP_ERR_INVALID;
    cudaSetDevice(h->device);
    if (on && !h->ev[0]) {
        for (int k = 0; k < 4; ++k)
            if (cudaEventCreate(&h->ev[k]) != cudaSuccess) return cuda_fail(h, cudaGetLastError(), "cudaEventCreate");
    }
    h->profiling = on != 0;
    return FCPP_OK;
}

int fcpp_kernel_times(fcpp_handle *h, float *ms3)
{
    if (!h || !ms3 || !h->ev[0]) return fail(h, FCPP_ERR_INVALID, "profiling is off");
    for (int k = 0; k < 3; ++k) {
        cudaError_t e = cudaEventElapsedTime(&ms3[k], h->ev[k], h->ev[k + 1]);
        if (e != cudaSuccess) return cuda_fail(h, e, "cudaEventElapsedTime");
    }
    return FCPP_OK;
}

int fcpp_set_trig_tables(fcpp_handle *h, const double *cos20, const double *sin20, const double *cos15,
                         const double *sin15)
{
    if (!h || !cos20 || !sin20 || !cos15 || !sin15) return fail(h, FCPP_ERR_INVALID, "NULL table");
    TrigTables t;
    memcpy(t.cos20, cos20, sizeof(t.cos20));
    memcpy(t.sin20, sin20, sizeof(t.sin20));
    memcpy(t.cos15, cos15, sizeof(t.cos15));
    memcpy(t.sin15, sin15, sizeof(t.sin15));
    cudaSetDevice(h->device);
    cudaError_t e = cudaMemcpy(h->d_trig, &t, sizeof(t), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return cuda_fail(h, e, "fcpp_set_trig_tables");
    return FCPP_OK;
}

int fcpp_layout(fcpp_handle *h, const fcpp_batch *batch, int32_t *d_n_pts, int64_t *d_offsets, void *stream)
{
    int rc = check_batch(h, batch);
    if (rc) return rc;
    cudaSetDevice(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    h->rec_valid = false;
    rc = ensure_workspace(h, batch->n_cand);
    if (rc) return rc;
    cudaError_t e = fcpp_launch_layout(h, *batch, d_n_pts, d_offsets, st);
    if (e != cudaSuccess) return cuda_fail(h, e, "layout kernel");
    // the plan and coverage kernels size their shared-memory staging by the longest headland of the batch
    int maxn = batch->max_points_hint, maxhead = batch->max_head_points_hint;
    if (maxn <= 0 || maxhead <= 0) {
        h->h_maxn[0] = h->h_maxn[1] = 0;
        if (batch->n_cand > 0) {
            e = cudaMemcpyAsync(h->h_maxn, h->d_maxn, 2 * sizeof(int), cudaMemcpyDeviceToHost, st);
            // the same synchronisation also brings back the total number of points (sizes the path buffers)
            if (e == cudaSuccess && d_offsets)
                e = cudaMemcpyAsync(h->h_maxn + 2, d_offsets + batch->n_cand, sizeof(int64_t), cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) return cuda_fail(h, e, "layout readback");
        }
        maxn = h->h_maxn[0];
        maxhead = h->h_maxn[1];
        h->last_maxn = maxn;
        h->last_maxhead = maxhead;
        h->last_total = -1;
        if (d_offsets && batch->n_cand > 0) memcpy(&h->last_total, h->h_maxn + 2, sizeof(int64_t));
    } else {
        h->last_total = -1;  // asynchronous pass: nothing was read back
    }
    h->cover_pcap = maxhead;
    h->layout_valid = true;
    h->rec_valid = true;
    h->layout_ncand = batch->n_cand;
    h->layout_id[0] = batch->cand_field ? (const void *)batch->cand_R : (const void *)batch->ax_radii;
    h->layout_id[1] = batch->cand_field ? (const void *)batch->cand_flags : (const void *)(intptr_t)batch->cand_first;
    h->layout_id[2] = batch->field_verts;
    h->layout_id[3] = stream;
    return FCPP_OK;
}

int fcpp_plan_batch(fcpp_handle *h, const fcpp_batch *batch, const fcpp_outputs *out, void *stream)
{
    int rc = check_batch(h, batch);
    if (rc) return rc;
    if (!out || !out->summary) return fail(h, FCPP_ERR_INVALID, "outputs.summary is required");
    const bool paths = out->path_xy || out->speeds_kmh || out->curvature;
    if (paths && !out->offsets)
        return fail(h, FCPP_ERR_INVALID, "materialised paths need outputs.offsets from fcpp_layout");
    cudaSetDevice(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    const bool prof = h->profiling;
    if (prof) cudaEventRecord(h->ev[0], st);
    if (out->offsets) {
        // the layout is stamped with the batch it was computed for (candidate / field arrays, stream): a
        // layout of another batch of the same size would hand stale records and offsets to the kernels
        const void *id0 = batch->cand_field ? (const void *)batch->cand_R : (const void *)batch->ax_radii;
        const void *id1 = batch->cand_field ? (const void *)batch->cand_flags : (const void *)(intptr_t)batch->cand_first;
        if (!h->layout_valid || h->layout_ncand != batch->n_cand || h->layout_id[0] != id0 || h->layout_id[1] != id1 ||
            h->layout_id[2] != batch->field_verts || h->layout_id[3] != stream)
            return fail(h, FCPP_ERR_INVALID, "fcpp_layout must be called for this batch (same arrays, same stream) "
                                             "before fcpp_plan_batch");
    } else {
        rc = fcpp_layout(h, batch, nullptr, nullptr, stream);
        if (rc) return rc;
    }
    if (prof) cudaEventRecord(h->ev[1], st);
    cudaError_t e = fcpp_launch_plan(h, *batch, *out, st);
    if (e != cudaSuccess) return cuda_fail(h, e, "plan kernel");
    if (prof) cudaEventRecord(h->ev[2], st);
    if (batch->do_coverage) {
        e = fcpp_launch_cover(h, *batch, *out, st);
        if (e != cudaSuccess) return cuda_fail(h, e, "coverage kernels");
    }
    if (prof) cudaEventRecord(h->ev[3], st);
    h->layout_valid = false;  // one layout per plan call
    return FCPP_OK;
}

int fcpp_obstacle_sweep(fcpp_handle *h, const fcpp_batch *batch, fcpp_sweep *d_out, void *stream)
{
    int rc = check_batch(h, batch);
    if (rc) return rc;
    if (batch->n_cand > 0 && !d_out) return fail(h, FCPP_ERR_INVALID, "fcpp_obstacle_sweep: d_out is NULL");
    // the records must be those of this batch: the stamp of its layout pass, which fcpp_plan_batch leaves in place
    const void *id0 = batch->cand_field ? (const void *)batch->cand_R : (const void *)batch->ax_radii;
    const void *id1 = batch->cand_field ? (const void *)batch->cand_flags : (const void *)(intptr_t)batch->cand_first;
    if (!h->rec_valid || h->layout_ncand != batch->n_cand || h->layout_id[0] != id0 || h->layout_id[1] != id1 ||
        h->layout_id[2] != batch->field_verts || h->layout_id[3] != stream)
        return fail(h, FCPP_ERR_INVALID, "fcpp_layout must be called for this batch (same arrays, same stream) "
                                         "before fcpp_obstacle_sweep");
    cudaSetDevice(h->device);
    cudaError_t e = fcpp_launch_sweep(h, *batch, d_out, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(h, e, "obstacle sweep kernel");
    return FCPP_OK;
}

int fcpp_obstacle_sweep_paths(fcpp_handle *h, const double *d_path_xy, const int64_t *d_offsets, int64_t n_paths,
                              const int32_t *d_n_main, const int32_t *d_obs_vert_start, const double *d_obs_verts,
                              int32_t n_polys, double radius, fcpp_sweep *d_out, void *stream)
{
    if (!h) return FCPP_ERR_INVALID;
    if (n_paths < 0 || n_paths > 0x7fffffff || n_polys < 0 || !(radius >= 0.0) || !isfinite(radius) ||
        (n_paths > 0 && (!d_path_xy || !d_offsets || !d_out)) || (n_polys > 0 && (!d_obs_vert_start || !d_obs_verts)))
        return fail(h, FCPP_ERR_INVALID, "fcpp_obstacle_sweep_paths: bad argument");
    cudaSetDevice(h->device);
    cudaError_t e = fcpp_launch_sweep_paths(h, d_path_xy, d_offsets, n_paths, d_n_main, d_obs_vert_start, d_obs_verts,
                                            n_polys, radius, d_out, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(h, e, "obstacle sweep kernel (paths)");
    return FCPP_OK;
}

static bool grid_h_ok(double grid_h)
{
    const double hq = grid_h * FCPP_FIXED_UNIT;
    const long long H = llrint(hq);
    return isfinite(hq) && H >= 2 && !(H & 1) && fabs(hq - (double)H) <= 1e-6;
}

int fcpp_path_coverage(fcpp_handle *h, const double *d_path_xy, const int64_t *d_offsets, int64_t n_paths,
                       const int32_t *d_n_main, const int32_t *d_path_field, const double *d_headland_width,
                       int32_t n_fields, const double *d_field_verts, const int32_t *d_obs_poly_start,
                       const int32_t *d_obs_vert_start, const double *d_obs_verts, double radius, double grid_h,
                       fcpp_path_cover *d_out, void *stream)
{
    if (!h) return FCPP_ERR_INVALID;
    if (n_paths < 0 || n_paths > 0x7fffffff || n_fields < 0 || !(radius >= 0.0) || !isfinite(radius) ||
        (n_paths > 0 && (!d_path_xy || !d_offsets || !d_path_field || !d_headland_width || !d_out)) ||
        (n_paths > 0 && n_fields > 0 && !d_field_verts) || (d_obs_poly_start && (!d_obs_vert_start || !d_obs_verts)))
        return fail(h, FCPP_ERR_INVALID, "fcpp_path_coverage: bad argument");
    if (!grid_h_ok(grid_h))
        return fail(h, FCPP_ERR_INVALID, "fcpp_path_coverage: grid_h must be an even multiple of 1e-4 m (got %g)", grid_h);
    cudaSetDevice(h->device);
    PathCoverSrc src{};
    src.path = d_path_xy;
    src.offsets = d_offsets;
    src.n = n_paths;
    src.path_field = d_path_field;
    src.headland_width = d_headland_width;
    src.n_main = d_n_main;
    src.n_fields = n_fields;
    src.field_verts = d_field_verts;
    src.obs_poly_start = d_obs_poly_start;
    src.obs_vert_start = d_obs_vert_start;
    src.obs_verts = d_obs_verts;
    src.radius = radius;
    src.grid_h = grid_h;
    cudaError_t e = fcpp_launch_path_cover(h, src, d_out, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(h, e, "path coverage kernels");
    return FCPP_OK;
}

int fcpp_plan_coverage(fcpp_handle *h, const fcpp_batch *batch, const fcpp_outputs *outputs, fcpp_path_cover *d_out,
                       void *stream)
{
    int rc = check_batch(h, batch);
    if (rc) return rc;
    if (!outputs || !outputs->summary || !outputs->path_xy || !outputs->offsets)
        return fail(h, FCPP_ERR_INVALID, "fcpp_plan_coverage: needs materialised paths (outputs.path_xy, offsets)");
    if (batch->n_cand > 0 && !d_out) return fail(h, FCPP_ERR_INVALID, "fcpp_plan_coverage: d_out is NULL");
    if (!grid_h_ok(batch->grid_h))
        return fail(h, FCPP_ERR_INVALID, "fcpp_plan_coverage: grid_h must be an even multiple of 1e-4 m (got %g)",
                    batch->grid_h);
    // the records must be those of this batch (the stamp of its layout pass, as fcpp_obstacle_sweep)
    const void *id0 = batch->cand_field ? (const void *)batch->cand_R : (const void *)batch->ax_radii;
    const void *id1 = batch->cand_field ? (const void *)batch->cand_flags : (const void *)(intptr_t)batch->cand_first;
    if (!h->rec_valid || h->layout_ncand != batch->n_cand || h->layout_id[0] != id0 || h->layout_id[1] != id1 ||
        h->layout_id[2] != batch->field_verts || h->layout_id[3] != stream)
        return fail(h, FCPP_ERR_INVALID, "fcpp_layout and fcpp_plan_batch must be called for this batch (same arrays, "
                                         "same stream) before fcpp_plan_coverage");
    cudaSetDevice(h->device);
    PathCoverSrc src{};
    src.path = outputs->path_xy;
    src.offsets = outputs->offsets;
    src.n = batch->n_cand;
    src.recs = h->d_rec;
    src.summary = outputs->summary;
    src.n_fields = batch->n_fields;
    src.field_verts = batch->field_verts;
    src.obs_poly_start = batch->obs_poly_start;
    src.obs_vert_start = batch->obs_vert_start;
    src.obs_verts = batch->obs_verts;
    src.radius = batch->vehicle.working_width / 2;
    src.grid_h = batch->grid_h;
    cudaError_t e = fcpp_launch_path_cover(h, src, d_out, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(h, e, "plan coverage kernels");
    return FCPP_OK;
}

int fcpp_field_select(fcpp_handle *h, const fcpp_summary *d_summary, const int32_t *d_cand_field, int64_t n_cand,
                      int32_t n_fields, const fcpp_selection *sel, int64_t cand_base, double *d_cost, int64_t *d_cand,
                      void *stream)
{
    if (!h) return FCPP_ERR_INVALID;
    if (!sel || n_cand < 0 || n_fields < 0 || cand_base < 0 || (n_fields > 0 && (!d_cost || !d_cand)) ||
        (n_cand > 0 && !d_summary))
        return fail(h, FCPP_ERR_INVALID, "fcpp_field_select: bad argument");
    if (sel->top_k < 1 || sel->top_k > FCPP_SELECT_MAX_K)
        return fail(h, FCPP_ERR_INVALID, "fcpp_field_select: top_k must be in 1..%d (got %d)", FCPP_SELECT_MAX_K,
                    sel->top_k);
    const double w[7] = {sel->w_length, sel->w_time, sel->w_boundary, sel->w_obstacle, sel->w_accel, sel->w_uncovered,
                         sel->cell_area};
    for (double x : w)
        if (!(x >= 0.0 && isfinite(x)))
            return fail(h, FCPP_ERR_INVALID, "fcpp_field_select: weights and cell_area must be finite and >= 0");
    if (!(sel->min_coverage <= 1.0))  // NaN too; < 0 = no limit
        return fail(h, FCPP_ERR_INVALID, "fcpp_field_select: min_coverage must be <= 1");
    if (n_cand > 0 && !d_cand_field && (n_cand > h->rec_cap || !h->d_rec))
        return fail(h, FCPP_ERR_INVALID, "fcpp_field_select: no cand_field and no candidate records of this batch");
    cudaSetDevice(h->device);
    cudaError_t e = fcpp_launch_select(h, d_summary, d_cand_field, n_cand, n_fields, *sel, cand_base, d_cost, d_cand,
                                       (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(h, e, "selection kernels");
    return FCPP_OK;
}

int fcpp_field_select_merge(fcpp_handle *h, const int64_t *d_gathered, int32_t world, int32_t n_fields, int32_t k,
                            double *d_cost, int64_t *d_cand, void *stream)
{
    if (!h) return FCPP_ERR_INVALID;
    if (world < 1 || n_fields < 0 || k < 1 || k > FCPP_SELECT_MAX_K ||
        (n_fields > 0 && (!d_gathered || !d_cost || !d_cand)))
        return fail(h, FCPP_ERR_INVALID, "fcpp_field_select_merge: bad argument");
    cudaSetDevice(h->device);
    cudaError_t e = fcpp_launch_select_merge(h, d_gathered, world, n_fields, k, d_cost, d_cand, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(h, e, "selection merge kernel");
    return FCPP_OK;
}

int fcpp_winner_records(fcpp_handle *h, const fcpp_summary *d_summary, int64_t cand_lo, int64_t cand_hi,
                        const int64_t *d_best_cand, int32_t n_fields, void *d_out, void *stream)
{
    if (!h) return FCPP_ERR_INVALID;
    if (n_fields < 0 || cand_hi < cand_lo || (n_fields > 0 && (!d_best_cand || !d_out)) || (cand_hi > cand_lo && !d_summary))
        return fail(h, FCPP_ERR_INVALID, "fcpp_winner_records: bad argument");
    cudaSetDevice(h->device);
    cudaError_t e = fcpp_launch_winner_records(h, d_summary, cand_lo, cand_hi, d_best_cand, n_fields, d_out,
                                               (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(h, e, "winner records kernel");
    return FCPP_OK;
}

int fcpp_status_count(fcpp_handle *h, const fcpp_summary *d_summary, int64_t n_cand, int32_t mask, int32_t *d_count,
                      void *stream)
{
    if (!h) return FCPP_ERR_INVALID;
    if (n_cand < 0 || !d_count || (n_cand > 0 && !d_summary)) return fail(h, FCPP_ERR_INVALID, "fcpp_status_count: bad argument");
    cudaSetDevice(h->device);
    cudaError_t e = fcpp_launch_status_count(h, d_summary, n_cand, mask, d_count, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(h, e, "status count kernel");
    return FCPP_OK;
}

int fcpp_speed_verify(fcpp_handle *h, const fcpp_vehicle *veh, const double *d_path_xy, const double *d_speeds_in,
                      const int64_t *d_offsets, int64_t n_paths, int64_t max_path_len, int do_speed_plan,
                      double *d_speeds_out, double *d_curvature, fcpp_summary *d_summary, void *stream)
{
    if (!h) return FCPP_ERR_INVALID;
    if (!veh || n_paths < 0 || (n_paths > 0 && (!d_path_xy || !d_speeds_in || !d_offsets)))
        return fail(h, FCPP_ERR_INVALID, "fcpp_speed_verify: bad argument");
    cudaSetDevice(h->device);
    cudaError_t e = fcpp_launch_speed_verify(h, *veh, d_path_xy, d_speeds_in, d_offsets, n_paths, max_path_len,
                                             do_speed_plan, d_speeds_out, d_curvature, d_summary,
                                             (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(h, e, "speed/verify kernel");
    return FCPP_OK;
}

int fcpp_raster_window(fcpp_handle *h, const double *d_path_xy, int32_t n_pts, double radius, double origin_x,
                       double origin_y, double h_cell, int32_t g, uint32_t *d_bits, int64_t *d_count, void *stream)
{
    if (!h) return FCPP_ERR_INVALID;
    if (!d_path_xy || n_pts < 0 || g < 1 || g > 8192 || !d_bits || !d_count || !(h_cell > 0) || !(radius >= 0))
        return fail(h, FCPP_ERR_INVALID, "fcpp_raster_window: bad argument");
    if (llrint(h_cell * FCPP_FIXED_UNIT) < 1) return fail(h, FCPP_ERR_INVALID, "h_cell below the 1e-4 m lattice");
    if (!(h_cell * FCPP_FIXED_UNIT < 1e15) || (int64_t)g * llrint(h_cell * FCPP_FIXED_UNIT) >= (1ll << 30))
        return fail(h, FCPP_ERR_INVALID, "fcpp_raster_window: g * q(h_cell) must be below 2^30 lattice units");
    cudaSetDevice(h->device);
    cudaError_t e = fcpp_launch_raster_window(h, d_path_xy, n_pts, radius, origin_x, origin_y, h_cell, g, d_bits,
                                              d_count, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(h, e, "window raster kernel");
    return FCPP_OK;
}

int fcpp_tour_lengths(fcpp_handle *h, const double *d_D, int32_t n, const int32_t *d_pop, int64_t pop_size,
                      double *d_out, double *d_fitness, void *stream)
{
    if (!h) return FCPP_ERR_INVALID;
    if (n < 1 || pop_size < 0 || !d_out || (pop_size > 0 && (!d_D || !d_pop)))
        return fail(h, FCPP_ERR_INVALID, "fcpp_tour_lengths: bad argument");
    cudaSetDevice(h->device);
    cudaError_t e = fcpp_launch_tours(h, d_D, n, d_pop, pop_size, d_out, d_fitness, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(h, e, "tour kernel");
    return FCPP_OK;
}

}  // extern "C"

extern "C" {

int fcpp_distance_matrix(fcpp_handle *h, const double *d_pos, int32_t n, double *d_D, void *stream)
{
    if (!h) return FCPP_ERR_INVALID;
    if (n < 0 || n > 65535 || (n > 0 && (!d_pos || !d_D))) return fail(h, FCPP_ERR_INVALID, "fcpp_distance_matrix: bad argument");
    cudaSetDevice(h->device);
    cudaError_t e = fcpp_launch_distance_matrix(h, d_pos, n, d_D, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(h, e, "distance matrix kernel");
    return FCPP_OK;
}

int fcpp_connection_matrix(fcpp_handle *h, const double *d_field_verts, int32_t n_fields, double depot_x,
                           double depot_y, double *d_C, int32_t *d_arg, void *stream)
{
    if (!h) return FCPP_ERR_INVALID;
    if (n_fields < 0 || n_fields > 65534 || !d_C || !d_arg || (n_fields > 0 && !d_field_verts))
        return fail(h, FCPP_ERR_INVALID, "fcpp_connection_matrix: bad argument");
    cudaSetDevice(h->device);
    cudaError_t e = fcpp_launch_connection_matrix(h, d_field_verts, n_fields, depot_x, depot_y, d_C, d_arg,
                                                  (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(h, e, "connection matrix kernel");
    return FCPP_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// GA evolution on the device (fcpp_ga.cu)
// ---------------------------------------------------------------------------------------------
namespace {

int check_ga(fcpp_handle *h, const fcpp_ga_config *c, int n, int m_in)
{
    if (!h) return FCPP_ERR_INVALID;
    if (!c) return fail(h, FCPP_ERR_INVALID, "GA config is NULL");
    if (n < 1 || n > 12288) return fail(h, FCPP_ERR_INVALID, "GA: n must be in 1..12288 (got %d)", n);
    if (m_in < 1) return fail(h, FCPP_ERR_INVALID, "GA: empty population");
    if (c->tournament_size < 1 || c->tournament_size > FCPP_GA_MAX_TOURNAMENT)
        return fail(h, FCPP_ERR_INVALID, "GA: tournament_size must be in 1..%d", FCPP_GA_MAX_TOURNAMENT);
    if (c->tournament_size > m_in)  // random.sample raises ValueError (ga:189)
        return fail(h, FCPP_ERR_INVALID, "GA: tournament_size %d larger than the population %d", c->tournament_size,
                    m_in);
    if (c->elite_size < 0) return fail(h, FCPP_ERR_INVALID, "GA: negative elite_size");
    return FCPP_OK;
}

struct GaWs {
    int32_t *pop[2];
    double *len, *fit;
    int *rank;
    void *state;
    int32_t *best;
};

size_t al256(size_t x) { return (x + 255) & ~size_t(255); }

int ga_workspace(fcpp_handle *h, int cap, int n, GaWs &w)
{
    const size_t pop_b = al256((size_t)cap * n * 4), vec_b = al256((size_t)cap * 8), rank_b = al256((size_t)cap * 4);
    const size_t st_b = al256(fcpp_ga_state_bytes()), best_b = al256((size_t)n * 4);
    const size_t total = 2 * pop_b + 2 * vec_b + rank_b + st_b + best_b;
    if (total > h->ga_bytes) {
        if (h->d_ga) cudaFree(h->d_ga);
        h->d_ga = nullptr;
        h->ga_bytes = 0;
        cudaError_t e = cudaMalloc(&h->d_ga, total);
        if (e != cudaSuccess) return cuda_fail(h, e, "cudaMalloc(GA workspace)");
        h->ga_bytes = total;
    }
    if (!h->h_ga_state) {
        cudaError_t e = cudaMallocHost(&h->h_ga_state, fcpp_ga_state_bytes());
        if (e != cudaSuccess) return cuda_fail(h, e, "cudaMallocHost(GA state)");
    }
    unsigned char *p = (unsigned char *)h->d_ga;
    w.pop[0] = (int32_t *)p;
    p += pop_b;
    w.pop[1] = (int32_t *)p;
    p += pop_b;
    w.len = (double *)p;
    p += vec_b;
    w.fit = (double *)p;
    p += vec_b;
    w.rank = (int *)p;
    p += rank_b;
    w.state = p;
    p += st_b;
    w.best = (int32_t *)p;
    return FCPP_OK;
}

}  // namespace

extern "C" {

int32_t fcpp_ga_next_size(const fcpp_ga_config *cfg, int32_t m_in)
{
    if (!cfg || m_in < 1) return 0;
    int keep, e_take, m_out;
    fcpp_ga_sizes(*cfg, m_in, keep, e_take, m_out);
    return m_out;
}

int fcpp_ga_init_population(fcpp_handle *h, const fcpp_ga_config *cfg, int32_t n, int32_t *d_pop, void *stream)
{
    if (!h) return FCPP_ERR_INVALID;
    if (!cfg || !d_pop || n < 1 || cfg->population_size < 0)
        return fail(h, FCPP_ERR_INVALID, "fcpp_ga_init_population: bad argument");
    cudaSetDevice(h->device);
    cudaError_t e = fcpp_launch_ga_init(h, *cfg, n, d_pop, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(h, e, "GA init kernel");
    return FCPP_OK;
}

int fcpp_ga_generation(fcpp_handle *h, const fcpp_ga_config *cfg, int32_t generation, int32_t n,
                       const int32_t *d_pop_in, const double *d_fitness, int32_t m_in, int32_t *d_pop_out,
                       int32_t *d_trace, void *stream)
{
    int rc = check_ga(h, cfg, n, m_in);
    if (rc) return rc;
    if (!d_pop_in || !d_fitness || !d_pop_out || generation < 0)
        return fail(h, FCPP_ERR_INVALID, "fcpp_ga_generation: bad argument");
    cudaSetDevice(h->device);
    GaWs w;
    rc = ga_workspace(h, m_in + 2, n, w);
    if (rc) return rc;
    cudaError_t e = fcpp_launch_ga_generation(h, *cfg, generation, n, d_pop_in, d_fitness, m_in, d_pop_out, w.rank,
                                              d_trace, nullptr, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(h, e, "GA generation kernels");
    return FCPP_OK;
}

int fcpp_ga_solve(fcpp_handle *h, const fcpp_ga_config *cfg, const double *d_D, int32_t n, const int32_t *d_pop_init,
                  int32_t *d_best_route, double *d_history, fcpp_ga_result *host_result, void *stream)
{
    if (!h) return FCPP_ERR_INVALID;
    if (!cfg || !d_D || !d_best_route || !host_result) return fail(h, FCPP_ERR_INVALID, "fcpp_ga_solve: NULL argument");
    int m = d_pop_init ? cfg->population_size : 2 * (cfg->population_size / 2);  // ga:141-151
    int rc = check_ga(h, cfg, n, m);
    if (rc) return rc;
    if (cfg->max_generations < 0) return fail(h, FCPP_ERR_INVALID, "GA: negative max_generations");
    cudaSetDevice(h->device);
    cudaStream_t st = (cudaStream_t)stream;
    GaWs w;
    rc = ga_workspace(h, cfg->population_size + 2, n, w);
    if (rc) return rc;
    cudaError_t e = cudaSuccess;
#define GA_CK(call, what)                          \
    do {                                           \
        e = (call);                                \
        if (e != cudaSuccess) {                    \
            if (exec) cudaGraphExecDestroy(exec);  \
            return cuda_fail(h, e, what);          \
        }                                          \
    } while (0)
    cudaGraphExec_t exec = nullptr;
    if (d_pop_init)
        GA_CK(cudaMemcpyAsync(w.pop[0], d_pop_init, (size_t)m * n * 4, cudaMemcpyDeviceToDevice, st), "GA copy");
    else
        GA_CK(fcpp_launch_ga_init(h, *cfg, n, w.pop[0], st), "GA init kernel");
    GA_CK(fcpp_launch_tours(h, d_D, n, w.pop[0], m, w.len, w.fit, st), "tour kernel");                       // ga:68
    GA_CK(fcpp_launch_ga_track(h, w.fit, w.len, w.pop[0], m, n, cfg->convergence_threshold, 1, w.state, w.best,
                               nullptr, st),
          "GA track kernel");                                                                                // ga:70-72
    int cur = 0, launched = 0;
    const int G = cfg->max_generations;
    int check = cfg->check_every > 0 ? cfg->check_every : 16;
    check += check & 1;
    auto one_generation = [&](cudaStream_t s) -> cudaError_t {
        int keep, e_take, m_out;
        fcpp_ga_sizes(*cfg, m, keep, e_take, m_out);
        cudaError_t err = fcpp_launch_ga_generation(h, *cfg, -1, n, w.pop[cur], w.fit, m, w.pop[cur ^ 1], w.rank,
                                                    nullptr, w.state, s);                                     // ga:78-88
        if (err != cudaSuccess) return err;
        cur ^= 1;
        m = m_out;
        err = fcpp_launch_tours(h, d_D, n, w.pop[cur], m, w.len, w.fit, s);                                   // ga:91
        if (err != cudaSuccess) return err;
        return fcpp_launch_ga_track(h, w.fit, w.len, w.pop[cur], m, n, cfg->convergence_threshold, 0, w.state,
                                    w.best, d_history, s);                                                    // ga:94-116
    };
    auto poll = [&](int &done) -> cudaError_t {
        cudaError_t err = cudaMemcpyAsync(h->h_ga_state, w.state, fcpp_ga_state_bytes(), cudaMemcpyDeviceToHost, st);
        if (err == cudaSuccess) err = cudaStreamSynchronize(st);
        int g, sg, lg;
        double bf, bl;
        fcpp_ga_read_state(h->h_ga_state, g, sg, done, lg, bf, bl);
        return err;
    };
    int done = 0;
    // generations whose population size still changes (an odd population grows once) run directly
    while (launched < G && fcpp_ga_next_size(cfg, m) != m) {
        GA_CK(one_generation(st), "GA generation");
        ++launched;
    }
    if (launched > 0) GA_CK(poll(done), "GA poll");
    // steady state: a CUDA graph of two generations (ping-pong returns to the same buffer)
    if (!done && G - launched >= 2) {
        if (!h->ga_stream) GA_CK(cudaStreamCreateWithFlags(&h->ga_stream, cudaStreamNonBlocking), "cudaStreamCreate");
        cudaGraph_t graph = nullptr;
        const int64_t l0 = h->launches;
        GA_CK(cudaStreamBeginCapture(h->ga_stream, cudaStreamCaptureModeThreadLocal), "cudaStreamBeginCapture");
        cudaError_t e1 = one_generation(h->ga_stream);
        cudaError_t e2 = (e1 == cudaSuccess) ? one_generation(h->ga_stream) : e1;
        cudaError_t e3 = cudaStreamEndCapture(h->ga_stream, &graph);
        const int64_t per_unit = h->launches - l0;
        h->launches = l0;
        if (e2 != cudaSuccess || e3 != cudaSuccess) {
            if (graph) cudaGraphDestroy(graph);
            return cuda_fail(h, e2 != cudaSuccess ? e2 : e3, "GA graph capture");
        }
        e = cudaGraphInstantiate(&exec, graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) {
            exec = nullptr;
            return cuda_fail(h, e, "cudaGraphInstantiate");
        }
        int since = 0;
        while (!done && G - launched >= 2) {
            GA_CK(cudaGraphLaunch(exec, st), "cudaGraphLaunch");
            h->launches += per_unit;
            launched += 2;
            since += 2;
            if (since >= check) {
                GA_CK(poll(done), "GA poll");
                since = 0;
            }
        }
        if (!done) GA_CK(poll(done), "GA poll");
        cudaGraphExecDestroy(exec);
        exec = nullptr;
    }
    while (!done && launched < G) {
        GA_CK(one_generation(st), "GA generation");
        ++launched;
        GA_CK(poll(done), "GA poll");
    }
    GA_CK(fcpp_launch_ga_rotate(h, w.best, n, d_best_route, st), "GA rotate kernel");                        // ga:119-120
    GA_CK(poll(done), "GA poll");
#undef GA_CK
    int g, sg, lg;
    double bf, bl;
    fcpp_ga_read_state(h->h_ga_state, g, sg, done, lg, bf, bl);
    host_result->generations = g;                 // ga:123 generation + 1
    host_result->convergence_gen = lg - sg;       // ga:126
    host_result->final_population = m;
    host_result->reserved = 0;
    host_result->best_distance = bl;
    host_result->best_fitness = bf;
    return FCPP_OK;
}

}  // extern "C"
