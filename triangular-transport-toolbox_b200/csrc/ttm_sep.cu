// Separable-monotonicity kernels: K-sep-eval (S_k, d_k S_k), K-sepobj, density bookkeeping (K-gram: ttm_gram.cu).
//
// Reference: s (separable arm) transport_map.py:2550-2558; log-determinants :2618-2641, :2686-2709;
// worker_task_monotone :2903-3172 (Gram-type contractions :2966-2975, :3031-3050; reduced objective
// fun_mon_objective :2978-3018).

#include "ttm_common.cuh"
#include "ttm_kernels.h"
#include "ttm_sweep.cuh"

namespace {

constexpr int T_SEP = 128;

// S_i = sum_j a_j psi^non_j(Xt_i) + sum_j b_j psi^mon_j(Xt_i);  dS_i = sum_j b_j dpsi^mon_j(Xd_i)
__global__ void __launch_bounds__(T_SEP) sep_eval_kernel(const PlanView P, const double* __restrict__ Xt, int64_t ld,
                                                         int64_t N, const double* __restrict__ coeffs,
                                                         double* __restrict__ S_out, const double* __restrict__ Xd,
                                                         int64_t ldd, double* __restrict__ dS_out,
                                                         const double* __restrict__ base, double a0) {
    // base != NULL: the nonmonotone part comes from K-inv-rect's GEMM (base_i + a0), only the monotone terms are
    // evaluated here
    extern __shared__ double s_coef[];
    const int m = P.m_non + P.m_mon;
    for (int j = threadIdx.x; j < m; j += T_SEP) s_coef[j] = coeffs[j];
    const DenseSmem DS = stage_dense_tables(P, coeffs, m, threadIdx.x, T_SEP);
    __syncthreads();
    const double* acoef = s_coef;
    const double* bcoef = s_coef + P.m_non;
    const int64_t rows = (N + T_SEP - 1) / T_SEP;
    for (int64_t row0 = (int64_t)blockIdx.x * R_OBJ; row0 < rows; row0 += (int64_t)gridDim.x * R_OBJ) {
        int64_t idx[R_OBJ];
        bool ok[R_OBJ];
        double S[R_OBJ];
#pragma unroll
        for (int r = 0; r < R_OBJ; ++r) {
            const int64_t i = (row0 + r) * T_SEP + threadIdx.x;
            ok[r] = (row0 + r < rows) && (i < N);
            idx[r] = ok[r] ? i : N - 1;
            S[r] = 0.0;
        }
        if (S_out) {
            if (base) {
#pragma unroll
                for (int r = 0; r < R_OBJ; ++r) S[r] = __ldcs(base + idx[r]) + a0;
            } else {
                dense_value_smem_rt<R_OBJ>(P, DS, Xt, ld, row0 * T_SEP + threadIdx.x, T_SEP, ok, S);
                nonmon_slow_rt<false>(P, Xt, ld, idx, acoef, S, nullptr, 0);
            }
            for (int j = 0; j < P.m_mon; ++j) {
                const double b = bcoef[j];
#pragma unroll
                for (int r = 0; r < R_OBJ; ++r)
                    S[r] = fma(b, plan_term(P, P.o_mon_ptr, P.o_mon_fac, j, Xt, ld, idx[r]), S[r]);
            }
#pragma unroll
            for (int r = 0; r < R_OBJ; ++r)
                if (ok[r]) S_out[idx[r]] = S[r];
        }
        if (dS_out) {
            double dS[R_OBJ];
#pragma unroll
            for (int r = 0; r < R_OBJ; ++r) dS[r] = 0.0;
            for (int j = 0; j < P.m_dmon; ++j) {
                const double b = bcoef[j];
#pragma unroll
                for (int r = 0; r < R_OBJ; ++r)
                    dS[r] = fma(b, plan_term(P, P.o_dmon_ptr, P.o_dmon_fac, j, Xd, ldd, idx[r]), dS[r]);
            }
#pragma unroll
            for (int r = 0; r < R_OBJ; ++r)
                if (ok[r]) dS_out[idx[r]] = dS[r];
        }
    }
}

// -------------------------------------------------------------------------------------------------
// K-sepobj: out[0] = sum_i log dS_i, out[1+j] = sum_i dpsi_ij / dS_i,
//           dS_i = sum_j (b_j + delta) dpsi_ij      (transport_map.py:2990-3006)
// -------------------------------------------------------------------------------------------------
// b may live in mapped pinned host memory (read once per block); the last block mirrors the result to host memory
// and publishes the launch's sequence number after a system fence (no D2H copy, no stream synchronisation)
__device__ __forceinline__ void sepobj_body(const PlanView& P, const double* __restrict__ Xt, int64_t ld, int64_t N,
                                            const double* __restrict__ b, double* __restrict__ d_b, double delta,
                                            double* __restrict__ partials, unsigned int* counter,
                                            double* __restrict__ out, double* out_host,
                                            unsigned long long* flag_host, unsigned long long seq,
                                            const unsigned int bx, const unsigned int gx) {
    extern __shared__ double sm[];
    const int mm = P.m_dmon;
    double* s_b = sm;                 // [mm]
    double* s_acc = sm + mm;          // [mm][T_SEP]
    double* s_red = s_acc + mm * T_SEP;  // [T_SEP/32][1+mm]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int j = tid; j < mm; j += T_SEP) {
        const double bj = b[j];
        s_b[j] = bj + delta;
        if (bx == 0 && d_b) d_b[j] = bj;       // device copy of the coefficients (map / inverse use it)
    }
    for (int j = 0; j < mm; ++j) s_acc[j * T_SEP + tid] = 0.0;
    __syncthreads();
    double lacc = 0.0;
    for (int64_t i = (int64_t)bx * T_SEP + tid; i < N; i += (int64_t)gx * T_SEP) {
        double dS = 0.0;
        for (int j = 0; j < mm; ++j) dS = fma(s_b[j], plan_term(P, P.o_dmon_ptr, P.o_dmon_fac, j, Xt, ld, i), dS);
        lacc += log(dS);
        const double inv = 1.0 / dS;
        for (int j = 0; j < mm; ++j)
            s_acc[j * T_SEP + tid] += plan_term(P, P.o_dmon_ptr, P.o_dmon_fac, j, Xt, ld, i) * inv;
    }
    lacc = warp_sum(lacc);
    if (lane == 0) s_red[warp * (1 + mm)] = lacc;
    for (int j = 0; j < mm; ++j) {
        const double v = warp_sum(s_acc[j * T_SEP + tid]);
        if (lane == 0) s_red[warp * (1 + mm) + 1 + j] = v;
    }
    __syncthreads();
    double* part = partials + (int64_t)bx * (1 + mm);
    for (int j = tid; j < 1 + mm; j += T_SEP) {
        double v = 0.0;
        for (int w = 0; w < T_SEP / 32; ++w) v += s_red[w * (1 + mm) + j];
        part[j] = v;
    }
    __threadfence();
    __shared__ unsigned int s_last;
    __syncthreads();
    if (tid == 0) s_last = (atomicAdd(counter, 1u) == gx - 1) ? 1u : 0u;
    __syncthreads();
    if (s_last) {
        __threadfence();
        for (int j = tid; j < 1 + mm; j += T_SEP) {
            double v = 0.0;
            for (unsigned int bk = 0; bk < gx; ++bk) v += __ldcg(partials + (int64_t)bk * (1 + mm) + j);
            out[j] = v;
            if (out_host) out_host[j] = v;
        }
        if (out_host) {
            __threadfence_system();
            __syncthreads();
            if (tid == 0) *reinterpret_cast<volatile unsigned long long*>(flag_host) = seq;
        }
        if (tid == 0) *counter = 0u;
    }
}


__global__ void __launch_bounds__(T_SEP) sepobj_kernel(const PlanView P, const double* __restrict__ Xt, int64_t ld,
                                                       int64_t N, const double* __restrict__ b, double* __restrict__ d_b,
                                                       double delta, double* __restrict__ partials, unsigned int* counter,
                                                       double* __restrict__ out, double* out_host,
                                                       unsigned long long* flag_host, unsigned long long seq) {
    sepobj_body(P, Xt, ld, N, b, d_b, delta, partials, counter, out, out_host, flag_host, seq, blockIdx.x, gridDim.x);
}

// the same for several components in ONE launch (blockIdx.y selects the component): the lockstep L-BFGS-B rounds of a
// separable fit evaluate every component that asked for (f, g) together; descriptors live in device memory, only the
// launch's sequence numbers and the list of active components travel as kernel parameters
__global__ void __launch_bounds__(T_SEP) sepobj_batch_kernel(const SepBatchItem* __restrict__ items,
                                                             const __grid_constant__ SepBatchLaunch L,
                                                             const double* __restrict__ Xt, int64_t ld, int64_t N,
                                                             double delta) {
    const SepBatchItem& it = items[L.item[blockIdx.y]];
    sepobj_body(it.P, Xt, ld, N, it.b, it.d_b, delta, it.partials, it.counter, it.out, it.out_host, it.flag_host,
                L.seq[blockIdx.y], blockIdx.x, gridDim.x);
}

// change-of-variables bookkeeping of the density evaluators (transport_map.py:2618-2644, :2680-2712)
__global__ void density_acc_kernel(double* __restrict__ acc, const double* __restrict__ S,
                                   const double* __restrict__ dS, double sigma, int mode, int64_t N) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const double ld = log(dS[i] / sigma);
    if (mode == 0) acc[i] += -0.5 * S[i] * S[i] - 0.91893853320467274178 + ld;   // log N(z;0,1) + log dS/sigma
    else acc[i] -= ld;
}

__global__ void density_finish_kernel(const double* __restrict__ acc, const double* __restrict__ logt,
                                      double* __restrict__ out, int64_t N) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    out[i] = exp(acc[i] + (logt ? logt[i] : 0.0));
}

}  // namespace

cudaError_t ttm_launch_density_acc(double* acc, const double* S, const double* dS, double sigma, int mode, int64_t N,
                                   cudaStream_t st) {
    density_acc_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(acc, S, dS, sigma, mode, N);
    return cudaGetLastError();
}

cudaError_t ttm_launch_density_finish(const double* acc, const double* logt, double* out, int64_t N, cudaStream_t st) {
    density_finish_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(acc, logt, out, N);
    return cudaGetLastError();
}

cudaError_t ttm_launch_sep_eval(const PlanView& P, const double* Xt, int64_t ld, int64_t N, const double* coeffs,
                                double* S_out, const double* Xd, int64_t ldd, double* dS_out, int sm_count,
                                cudaStream_t st, const double* base, double a0) {
    if (N == 0) return cudaSuccess;
    const int64_t rows = (N + T_SEP - 1) / T_SEP;
    int64_t grid = (rows + R_OBJ - 1) / R_OBJ;
    if (grid > (int64_t)sm_count * 16) grid = (int64_t)sm_count * 16;
    const size_t smem = sizeof(double) * (size_t)(P.m_non + P.m_mon + dense_smem_doubles(P.ndense, P.dense_maxord));
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(sep_eval_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    sep_eval_kernel<<<(unsigned)grid, T_SEP, smem, st>>>(P, Xt, ld, N, coeffs, S_out, Xd, ldd, dS_out, base, a0);
    return cudaGetLastError();
}

cudaError_t ttm_launch_sepobj(const PlanView& P, const double* Xt, int64_t ld, int64_t N, const double* b,
                              double* d_b, double delta, double* partials, unsigned int* counter, double* out,
                              double* out_host, unsigned long long* flag_host, unsigned long long seq, int max_grid,
                              int sm_count, cudaStream_t st) {
    const int mm = P.m_dmon;
    int64_t grid = (N + T_SEP - 1) / T_SEP;
    if (grid > (int64_t)sm_count * 8) grid = (int64_t)sm_count * 8;
    if (grid > max_grid) grid = max_grid;
    if (grid < 1) grid = 1;
    const size_t smem = sizeof(double) * (size_t)(mm + mm * T_SEP + (T_SEP / 32) * (1 + mm));
    if (smem > 227 * 1024) return cudaErrorInvalidValue;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(sepobj_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    sepobj_kernel<<<(unsigned)grid, T_SEP, smem, st>>>(P, Xt, ld, N, b, d_b, delta, partials, counter, out, out_host,
                                                       flag_host, seq);
    return cudaGetLastError();
}

cudaError_t ttm_launch_sepobj_batch(const SepBatchItem* d_items, const SepBatchLaunch& L, int nact, int max_mm,
                                    const double* Xt, int64_t ld, int64_t N, double delta, int max_grid, int sm_count,
                                    cudaStream_t st) {
    if (nact <= 0) return cudaSuccess;
    int64_t gx = (N + T_SEP - 1) / T_SEP;
    const int64_t share = (int64_t)sm_count * 8 / nact;
    if (gx > share) gx = share;
    if (gx > max_grid) gx = max_grid;
    if (gx < 1) gx = 1;
    const size_t smem = sizeof(double) * (size_t)(max_mm + max_mm * T_SEP + (T_SEP / 32) * (1 + max_mm));
    if (smem > 227 * 1024) return cudaErrorInvalidValue;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(sepobj_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    sepobj_batch_kernel<<<dim3((unsigned)gx, (unsigned)nact), T_SEP, smem, st>>>(d_items, L, Xt, ld, N, delta);
    return cudaGetLastError();
}

// -------------------------------------------------------------------------------------------------
// K-map-fused / K-pullback (small separable maps): ALL components of the map on a tile of samples in one launch,
// reading the caller's row-major samples directly (float64 or float32, any row stride; standardisation on the fly) and writing row-major Z and/or the
// density -- no transposes, no per-component launches, no S / dS / accumulator round trips through HBM.
//   map                 tm.py:2391-2437 (separable arm of s, :2550-2558)
//   pullback density    tm.py:2646-2712:  exp( sum_k [-S_k^2/2 - log(2 pi)/2] + sum_k log(dS_k / sigma_k) )
//   pushforward density tm.py:2618-2644:  exp( log_target - sum_k log(dS_k / sigma_k) )
// dS_k = der_Psi_mon . coeffs_mon is evaluated on the UNstandardised samples like the reference does (:2627, :2695).
//   modes 3 / 4: the log pullback / log pushforward density of the fitted map (no exp; dS_k on the standardised
//   samples, sigma_k = X_std[k+skip] from the host) -- evaluate_log_pullback_density / _pushforward_density.
// HBM traffic: 8 n Dtot in, 8 n (D | 1) out.  The per-term work goes through the generic factor evaluator, so the
// host uses this kernel for maps with a few hundred terms in total (Example 05 / 06 shapes) and the per-component
// kernels with their dense sweeps for the large ones.
// -------------------------------------------------------------------------------------------------
namespace {

constexpr int T_FUSE = 128;

template <typename T>
__global__ void __launch_bounds__(T_FUSE) map_fused_kernel(const FusedMapArgs a) {
    extern __shared__ double sm[];
    const int ldt = T_FUSE + 1;
    double* t_std = sm;                         // [Dtot][129] standardised samples of the tile, column-major
    double* t_raw = sm + a.Dtot * ldt;          // [Dtot][129] raw samples
    const int tid = threadIdx.x;
    const int64_t base = (int64_t)blockIdx.x * T_FUSE;
    const int rows = (int)min((int64_t)T_FUSE, a.n - base);
    const T* __restrict__ X = static_cast<const T*>(a.X);
    for (int e = tid; e < rows * a.Dtot; e += T_FUSE) {
        const int r = e / a.Dtot, v = e - r * a.Dtot;
        const double x = (double)X[(base + r) * a.ldx + v];
        t_raw[v * ldt + r] = x;
        t_std[v * ldt + r] = a.mean ? (x - a.mean[v]) / a.sd[v] : x;
    }
    __syncthreads();
    if (tid >= rows) return;
    const bool pull = a.mode == 0 || a.mode == 3, push = a.mode == 1 || a.mode == 4, logm = a.mode >= 3;
    const double* t_der = logm ? t_std : t_raw;   // the log modes differentiate the map they evaluate
    double acc = 0.0;
    for (int k = 0; k < a.D; ++k) {
        const PlanView P = a.comps[k].P;
        const double* coef = a.comps[k].coeffs;
        const double* bcoef = coef + P.m_non;
        if (!push) {
            double S = 0.0;
            for (int j = 0; j < P.m_non; ++j) S = fma(coef[j], plan_term(P, P.o_non_ptr, P.o_non_fac, j, t_std, ldt, tid), S);
            for (int j = 0; j < P.m_mon; ++j) S = fma(bcoef[j], plan_term(P, P.o_mon_ptr, P.o_mon_fac, j, t_std, ldt, tid), S);
            if (a.Z) a.Z[(base + tid) * a.D + k] = S;
            acc += -0.5 * S * S - 0.91893853320467274178;
        }
        if (a.mode != 2) {
            double dS = 0.0;
            for (int j = 0; j < P.m_dmon; ++j) dS = fma(bcoef[j], plan_term(P, P.o_dmon_ptr, P.o_dmon_fac, j, t_der, ldt, tid), dS);
            const double ld = log(dS / a.comps[k].sigma);
            acc += pull ? ld : -ld;
        }
    }
    if (a.mode != 2) {
        const double v = acc + ((push && a.logt) ? a.logt[base + tid] : 0.0);
        a.out[base + tid] = logm ? v : exp(v);
    }
}

}  // namespace

template <typename T>
static cudaError_t launch_map_fused(const FusedMapArgs& a, size_t smem, cudaStream_t st) {
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(map_fused_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    map_fused_kernel<T><<<(unsigned)((a.n + T_FUSE - 1) / T_FUSE), T_FUSE, smem, st>>>(a);
    return cudaGetLastError();
}

cudaError_t ttm_launch_map_fused(const FusedMapArgs& a, cudaStream_t st) {
    if (a.n == 0) return cudaSuccess;
    const size_t smem = sizeof(double) * (size_t)(2 * a.Dtot * (T_FUSE + 1));
    if (smem > 200 * 1024) return cudaErrorInvalidValue;
    return a.dtype == TTM_DTYPE_F32 ? launch_map_fused<float>(a, smem, st) : launch_map_fused<double>(a, smem, st);
}
