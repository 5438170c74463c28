// fcpp_misc.cu — batched GA tour-length fitness (A12), the multi-GPU exchange of the winners' records and the
// multi-field distance / connection matrices.
//
// Reference code replaced:
//   genetic_algorithm_solver.py:168-181  _calculate_fitness / _calculate_distance
//   (distance-matrix layout: multi_field_planner.py:263-288, node 0 = depot)
#include "fcpp_internal.cuh"

namespace {

constexpr int TOUR_THREADS = 128;
constexpr int TOUR_CHUNK = 32;

// One thread per tour: the FP64 sum runs left to right exactly like the reference's Python
// loop, so tour lengths are bit-identical to genetic_algorithm_solver.py:174-181.  Tour rows
// are staged through shared memory in 32-column chunks (coalesced 128-B row segments in,
// conflict-free padded columns out); D (n*n FP64, 323 KB at n=201) is gathered through the
// read-only path and stays L1/L2 resident.
__global__ void __launch_bounds__(TOUR_THREADS) tour_kernel(const double *__restrict__ D, int n,
                                                            const int32_t *__restrict__ pop, int64_t pop_size,
                                                            double *__restrict__ out, double *__restrict__ fit)
{
    __shared__ int32_t tile[TOUR_THREADS][TOUR_CHUNK + 1];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t t0 = (int64_t)blockIdx.x * TOUR_THREADS;
    const int64_t me = t0 + tid;
    double s = 0.0;
    int first = 0, prev = 0;
    for (int c0 = 0; c0 < n; c0 += TOUR_CHUNK) {
        const int nc = min(TOUR_CHUNK, n - c0);
        for (int rr = warp; rr < TOUR_THREADS; rr += TOUR_THREADS / 32) {
            const int64_t t = t0 + rr;
            if (t < pop_size && lane < nc) tile[rr][lane] = pop[t * n + c0 + lane];
        }
        __syncthreads();
        if (me < pop_size) {
            int k = 0;
            if (c0 == 0) {
                first = prev = tile[tid][0];
                k = 1;
            }
            for (; k < nc; ++k) {
                const int cur = tile[tid][k];
                s += __ldg(&D[(int64_t)prev * n + cur]);
                prev = cur;
            }
        }
        __syncthreads();
    }
    if (me < pop_size) {
        s += __ldg(&D[(int64_t)prev * n + first]);  // closing edge (ga:178 `(i + 1) % len(route)`)
        out[me] = s;
        if (fit) fit[me] = 1.0 / (s + 1e-6);  // ga:172
    }
}

// multi-GPU: this rank's contribution to the all-gather of the winners' summary records — the 176-byte record of
// every field whose global winner lies in [lo, hi), zeros elsewhere (a SUM over the ranks then is the record)
__global__ void winner_records_kernel(const fcpp_summary *__restrict__ sm, int64_t lo, int64_t hi,
                                      const long long *__restrict__ best_cand, int n_fields, int4 *__restrict__ out)
{
    constexpr int W = sizeof(fcpp_summary) / 16;  // 11 int4 words per record
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)n_fields * W) return;
    const int f = (int)(t / W), k = (int)(t - (int64_t)f * W);
    const long long b = best_cand[f];
    out[t] = (b >= lo && b < hi) ? reinterpret_cast<const int4 *>(sm + (b - lo))[k] : make_int4(0, 0, 0, 0);
}

// multi_field_planner.py:263-288 ("mfp"): D[i][j] = ||pos_i - pos_j||, 0 on the diagonal
__global__ void distance_matrix_kernel(const double *__restrict__ pos, int n, double *__restrict__ D)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (j >= n) return;
    const double dx = pos[2 * i] - pos[2 * j], dy = pos[2 * i + 1] - pos[2 * j + 1];
    D[(int64_t)i * n + j] = (i == j) ? 0.0 : sqrt(dx * dx + dy * dy);
}

// mfp:290-320 for every ordered pair of nodes at once.  Node 0 is the depot (one candidate point),
// node f+1 is field f (its four vertices are both exit and entry points, mfp:140-141).
// C[a][b] = min over (from point of a) x (to point of b) of the distance, from points in the outer
// loop, strict '<' so the FIRST minimum wins; arg[a][b] = from_index * 4 + to_index.
__global__ void connection_matrix_kernel(const double *__restrict__ verts, int n_fields, double depot_x,
                                         double depot_y, double *__restrict__ Cm, int32_t *__restrict__ arg)
{
    const int n = n_fields + 1;
    const int b = blockIdx.x * blockDim.x + threadIdx.x, a = blockIdx.y;
    if (b >= n) return;
    double fx[4], fy[4], tx[4], ty[4];
    const int nf = a == 0 ? 1 : 4, nt = b == 0 ? 1 : 4;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        fx[k] = a == 0 ? depot_x : verts[(int64_t)(a - 1) * 8 + 2 * k];
        fy[k] = a == 0 ? depot_y : verts[(int64_t)(a - 1) * 8 + 2 * k + 1];
        tx[k] = b == 0 ? depot_x : verts[(int64_t)(b - 1) * 8 + 2 * k];
        ty[k] = b == 0 ? depot_y : verts[(int64_t)(b - 1) * 8 + 2 * k + 1];
    }
    double best = INFINITY;
    int bi = 0;
    for (int p = 0; p < nf; ++p)
        for (int q = 0; q < nt; ++q) {
            const double dx = fx[p] - tx[q], dy = fy[p] - ty[q];
            const double d = sqrt(dx * dx + dy * dy);
            if (d < best) {
                best = d;
                bi = p * 4 + q;
            }
        }
    Cm[(int64_t)a * n + b] = best;
    arg[(int64_t)a * n + b] = bi;
}

}  // namespace

// number of candidates whose status has one of the bits of `mask`
__global__ void status_count_kernel(const fcpp_summary *__restrict__ sm, int64_t n, int mask, int32_t *__restrict__ count)
{
    int hits = 0;
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (int64_t)gridDim.x * blockDim.x)
        hits += (sm[c].status & mask) != 0;
    hits = __reduce_add_sync(0xffffffffu, hits);
    if ((threadIdx.x & 31) == 0 && hits) atomicAdd(count, hits);
}

cudaError_t fcpp_launch_status_count(fcpp_handle *h, const fcpp_summary *d_summary, int64_t n, int mask, int32_t *d_count,
                                     cudaStream_t st)
{
    cudaError_t e = cudaMemsetAsync(d_count, 0, sizeof(int32_t), st);
    if (e != cudaSuccess || n == 0) return e;
    int64_t blocks = (n + 255) / 256;
    if (blocks > 4 * (int64_t)h->sm_count) blocks = 4 * (int64_t)h->sm_count;
    status_count_kernel<<<(unsigned)blocks, 256, 0, st>>>(d_summary, n, mask, d_count);
    h->launches++;
    return cudaGetLastError();
}

cudaError_t fcpp_launch_winner_records(fcpp_handle *h, const fcpp_summary *d_summary, int64_t lo, int64_t hi,
                                       const int64_t *d_best_cand, int32_t n_fields, void *d_out, cudaStream_t st)
{
    if (n_fields == 0) return cudaSuccess;
    static_assert(sizeof(fcpp_summary) % 16 == 0, "records are copied as int4 words");
    const int64_t n = (int64_t)n_fields * (sizeof(fcpp_summary) / 16);
    winner_records_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_summary, lo, hi, (const long long *)d_best_cand,
                                                                       n_fields, (int4 *)d_out);
    h->launches++;
    return cudaGetLastError();
}

cudaError_t fcpp_launch_distance_matrix(fcpp_handle *h, const double *d_pos, int32_t n, double *d_D, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    distance_matrix_kernel<<<dim3((n + 127) / 128, n), 128, 0, st>>>(d_pos, n, d_D);
    h->launches++;
    return cudaGetLastError();
}

cudaError_t fcpp_launch_connection_matrix(fcpp_handle *h, const double *d_verts, int32_t n_fields, double depot_x,
                                          double depot_y, double *d_C, int32_t *d_arg, cudaStream_t st)
{
    const int n = n_fields + 1;
    connection_matrix_kernel<<<dim3((n + 127) / 128, n), 128, 0, st>>>(d_verts, n_fields, depot_x, depot_y, d_C, d_arg);
    h->launches++;
    return cudaGetLastError();
}

cudaError_t fcpp_launch_tours(fcpp_handle *h, const double *d_D, int32_t n, const int32_t *d_pop,
                              int64_t pop_size, double *d_out, double *d_fit, cudaStream_t st)
{
    if (pop_size == 0) return cudaSuccess;
    const unsigned blocks = (unsigned)((pop_size + TOUR_THREADS - 1) / TOUR_THREADS);
    tour_kernel<<<blocks, TOUR_THREADS, 0, st>>>(d_D, n, d_pop, pop_size, d_out, d_fit);
    h->launches++;
    return cudaGetLastError();
}
