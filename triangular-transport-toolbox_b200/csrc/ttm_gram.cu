// K-gram: G = Psi^T Psi with Psi = [Psi_non | Psi_mon] (N x M), the one dense contraction of the path
// (reference: worker_task_monotone, transport_map.py:2966-2975 QR / A_sqrt^T A_sqrt and :3031-3050 ridge
// normal equations).  FP64 tensor cores: DMMA `mma.sync.aligned.m8n8k4.f64` -- tcgen05 has no f64 kind,
// so the warp-level MMA is the sm_100a tensor path for double precision.
//
// Two stages per chunk of samples:
//   1. the basis kernel materialises Psi for the chunk once (row-major, row stride Mp) in scratch;
//   2. a tiled SYRK: each block owns one 64x64 tile of the upper triangle of G and one split of the
//      chunk's rows, stages 32-row slabs of the two column panels in shared memory (coalesced 512-byte
//      rows, conflict-free fragment reads) and accumulates with 8 warps x (2x4) m8n8k4 tiles.
// Per-split partial Grams are summed in fixed order by gram_reduce_kernel (bit-reproducible).
// Flops 2*N*M^2 (upper triangle only: N*M*(M+64)); bytes: Psi is written once and read ~M/64 times from L2.

#include "ttm_common.cuh"
#include "ttm_kernels.h"

namespace {

constexpr int GT = 64;        // output tile
constexpr int GK = 32;        // rows per staged slab
constexpr int GLD = GT + 4;   // shared-memory row stride (doubles): conflict-free m8n8k4 fragment reads
constexpr int T_GRAM = 256;

// blockIdx.x = tile pair (ti <= tj, tj >= tj0), blockIdx.y = row split.  tj0 > 0: only the tile columns from tj0 on
// (the "tail" Gram: Psi^T [last columns], all a component needs when the leading block comes from a donor).
__global__ void __launch_bounds__(T_GRAM) syrk_dmma_kernel(const double* __restrict__ Psi, int64_t n, int Mp,
                                                           int nsplit, int accumulate, int tj0,
                                                           double* __restrict__ partial) {
    __shared__ double As[GK][GLD];
    __shared__ double Bs[GK][GLD];
    const int nt = (Mp + GT - 1) / GT;
    int tj = tj0, rem = blockIdx.x;                  // column tile tj holds the pairs ti = 0..tj
    while (rem > tj) { rem -= tj + 1; ++tj; }
    const int ti = rem;
    const int split = blockIdx.y;
    const int64_t rows_per = ((n + nsplit - 1) / nsplit + GK - 1) / GK * GK;
    const int64_t r_lo = (int64_t)split * rows_per;
    const int64_t r_hi = (r_lo + rows_per < n) ? r_lo + rows_per : n;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int wm = warp >> 1, wn = warp & 1;     // 4 x 2 warps: warp tile 16 rows x 32 columns
    double c[2][4][2];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) c[i][j][0] = c[i][j][1] = 0.0;
    const int ca = ti * GT, cb = tj * GT;
    for (int64_t s0 = r_lo; s0 < r_hi; s0 += GK) {
        __syncthreads();
        // stage 32 rows x 64 columns of both panels as double2 (32 consecutive threads = one 512-byte row)
        for (int e = threadIdx.x; e < GK * (GT / 2); e += T_GRAM) {
            const int row = e / (GT / 2), c2 = (e % (GT / 2)) * 2;
            const int64_t r = s0 + row;
            double2 va = make_double2(0.0, 0.0), vb = make_double2(0.0, 0.0);
            if (r < r_hi) {
                if (ca + c2 < Mp) va = *reinterpret_cast<const double2*>(Psi + r * Mp + ca + c2);
                if (cb + c2 < Mp) vb = *reinterpret_cast<const double2*>(Psi + r * Mp + cb + c2);
            }
            As[row][c2] = va.x; As[row][c2 + 1] = va.y;
            Bs[row][c2] = vb.x; Bs[row][c2 + 1] = vb.y;
        }
        __syncthreads();
#pragma unroll
        for (int k0 = 0; k0 < GK; k0 += 4) {
            const int kk = k0 + (lane & 3), q = lane >> 2;
            double a[2], b[4];
#pragma unroll
            for (int i = 0; i < 2; ++i) a[i] = As[kk][wm * 16 + i * 8 + q];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Bs[kk][wn * 32 + j * 8 + q];
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) dmma_m8n8k4(c[i][j][0], c[i][j][1], a[i], b[j]);
        }
    }
    double* out = partial + (int64_t)split * Mp * Mp;
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int row = ca + wm * 16 + i * 8 + (lane >> 2), col = cb + wn * 32 + j * 8 + 2 * (lane & 3);
            if (row < Mp && col < Mp) {     // Mp is a multiple of 8 and col is even: col + 1 < Mp as well
                double* o = out + (int64_t)row * Mp + col;
                if (accumulate) { o[0] += c[i][j][0]; o[1] += c[i][j][1]; }
                else { o[0] = c[i][j][0]; o[1] = c[i][j][1]; }
            }
        }
}

// G[i][j] = sum over splits (fixed order) of the stored element: element (r, c) of the upper block triangle
__global__ void gram_reduce_kernel(const double* __restrict__ partial, int nsplit, int Mp, int M, int tj0,
                                   double* __restrict__ G) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= M * M) return;
    const int i = e / M, j = e % M;
    if (max(i, j) / GT < tj0) { G[e] = 0.0; return; }   // tail Gram: the leading block is not computed
    // tile (i/64, j/64) is stored if its row tile <= column tile; otherwise use the transposed element
    const int r = (i / GT <= j / GT) ? i : j, c = (i / GT <= j / GT) ? j : i;
    double s = 0.0;
    for (int b = 0; b < nsplit; ++b) s += partial[(int64_t)b * Mp * Mp + (int64_t)r * Mp + c];
    G[e] = s;
}

}  // namespace

cudaError_t ttm_launch_gram(const PlanView& P, const double* Xt, int64_t ld, int64_t N, int first_col, double* G,
                            double* scratch, int64_t scratch_doubles, int sm_count, cudaStream_t st) {
    const int M = P.m_non + P.m_mon;
    if (M == 0 || N == 0) return cudaSuccess;
    const int Mp = (M + 7) / 8 * 8;
    const int nt = (Mp + GT - 1) / GT;
    const int tj0 = first_col / GT;                  // entries (i, j) with max(i, j) >= tj0 * 64 are computed
    const int npairs = nt * (nt + 1) / 2 - tj0 * (tj0 + 1) / 2;
    int nsplit = (2 * sm_count + npairs - 1) / npairs;
    if (nsplit > 64) nsplit = 64;
    if ((int64_t)nsplit * GK > N) nsplit = (int)((N + GK - 1) / GK);
    if (nsplit < 1) nsplit = 1;
    const int64_t part = (int64_t)nsplit * Mp * Mp;
    int64_t chunk = (scratch_doubles - part) / Mp;
    if (chunk > N) chunk = N;
    if (chunk > (1 << 18)) chunk = 1 << 18;
    if (chunk < GK && chunk < N) return cudaErrorInvalidValue;   // scratch too small
    double* partial = scratch;
    double* Psi = scratch + part;
    for (int64_t n0 = 0, it = 0; n0 < N; n0 += chunk, ++it) {
        const int64_t n = (n0 + chunk < N) ? chunk : N - n0;
        cudaError_t e = cudaMemsetAsync(Psi, 0, sizeof(double) * (size_t)n * Mp, st);
        if (e != cudaSuccess) return e;
        e = ttm_launch_basis_concat(P, Xt + n0, ld, n, Psi, Mp, st);
        if (e != cudaSuccess) return e;
        dim3 grid((unsigned)npairs, (unsigned)nsplit);
        syrk_dmma_kernel<<<grid, T_GRAM, 0, st>>>(Psi, n, Mp, nsplit, it > 0 ? 1 : 0, tj0, partial);
    }
    gram_reduce_kernel<<<(M * M + 255) / 256, 256, 0, st>>>(partial, nsplit, Mp, M, tj0, G);
    return cudaGetLastError();
}
