// K-inv-fused: the whole triangular solve of inverse_map for a tile of samples in ONE launch
// (separable monotonicity, table root finder).
//
// Reference: inverse_map transport_map.py:3639-3796 loops over the components k on the host and calls
//            vectorized_root_search_alternate :3987-4084 for each: offset_k = Psi_non(x_<c) a_k  (:4039-4043),
//            x_c = interp1d(table_k)(z_k - offset_k)                                             (:4047-4076).
// The per-component kernel (ttm_inverse.cu) re-reads every solved column for every component: sum_k 8 n (k+2)
// bytes, 64x the algorithmic 8 n (E + 2 (D - E)) at C5 (D = 256, E = 128).  Here a thread keeps its samples and walks
// the components itself, in blocks of 16:
//   rectangular part   offsets of the block's 16 components from all variables before the block: per variable the
//                      Hermite-function features {x, He2 e^{-x^2/4}, He3 e^{-x^2/4}} (one exp) are formed once and
//                      contracted with the 16 x 3 coefficients, which are staged through shared memory
//                      (cp.async, double buffered) and read as broadcast LDS.128;
//   diagonal part      component by component: table look-up (numpy.searchsorted + scipy's interp1d formula),
//                      store x_c, features of x_c, update of the remaining offsets of the block.
// Two samples per thread share every coefficient load.  The contraction is FP64-pipe work: 3 FMA per
// (sample, variable, component) pair, ~73 k FMA per sample at C5; measured FP64 tensor-core (DMMA) peak on B200
// equals the vector peak (tools/pipe_probe.cu: 37.0 vs 36.4 TFLOP/s), so the contraction stays on the vector pipe
// where it needs no operand staging of the features.
//
// Class: every component in the range has nonmonotone terms = constants + per-variable Hermite-function groups of
// order <= 3 (the host packs their coefficients, slot mask = the tile kernel's); anything else takes the
// per-component path.
#include <cuda_runtime.h>

#include <cstdint>

#include "ttm_common.cuh"
#include "ttm_exp.cuh"
#include "ttm_kernels.h"

namespace ttm_invf {

constexpr int TB = 128;       // threads per block
constexpr int SPT = 2;        // samples per thread
constexpr int CB = 16;        // components per block
constexpr int VC = 32;        // variables (coefficient rows) per staged chunk

// features of one variable value, in slot order (NS = 3: {He1, He2 e, He3 e}; NS = 6: {He1, He1 e, He2, He2 e, He3, He3 e})
template <int NS>
__device__ __forceinline__ void features(double x, const unsigned int* __restrict__ tab, double (&f)[NS]) {
    const double xx = x * x;
    const double ga = ttm_exp32::exp_neg_1(-0.25 * xx, tab);
    const double P2 = xx - 1.0, P3 = x * (xx - 3.0);
    if (NS == 3) {
        f[0] = x; f[1] = P2 * ga; f[2] = P3 * ga;
    } else {
        f[0] = x; f[1] = x * ga; f[2] = P2; f[3] = P2 * ga; f[4] = P3; f[NS - 1] = P3 * ga;
    }
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

// Apack: component block b holds rows v = 0 .. c0 + CB*b + CB - 1, each row CB*NS doubles [jj][slot];
// entries with v >= c0 + CB*b + jj (not a predecessor of component jj) are zero
__host__ __device__ inline int64_t block_row0(int b, int c0) { return (int64_t)b * (c0 + CB) + (int64_t)CB * b * (b - 1) / 2; }

// The component's table travels through shared memory (cp.async, double buffered, one barrier per component) and the
// binary search runs there: ten dependent LDS instead of dependent L2 round trips -- ncu attributed 37 % of the walk's
// issue slots to long-scoreboard waits of the search in place.  The entry points reject tables longer than
// TTM_INVERSE_FUSED_MAX_NTAB, whose two buffers would not fit next to the operands.  (A four-level search over a
// bank-skewed table image -- 21 independent comparisons instead of 10 dependent halvings -- was measured 2 % SLOWER: the
// walk is bound by the dependent FP64 chains of the whole component step, not by the search.)
template <int NS>
__global__ void __launch_bounds__(TB, 3) inverse_fused_kernel(const InvFusedArgs a) {
    extern __shared__ double smem[];
    constexpr int ROW = CB * NS;                 // doubles per coefficient row
    unsigned int* s_tab = reinterpret_cast<unsigned int*>(smem);   // exp table (64 words)
    double* s_coef = smem + ttm_exp32::TAB_DOUBLES;   // [2][VC][ROW]
    double* s_diag = s_coef + 2 * VC * ROW;      // [CB][ROW]
    double* s_table = s_diag + CB * ROW;         // [2][2 ntab]
    const int tbuf = 2 * a.ntab;
    const int tid = threadIdx.x;
    constexpr int PF = 8;                        // variables ahead of use for the L2 prefetch of the sample columns
    ttm_exp32::stage_table(s_tab, tid, TB);
    __syncthreads();
    const int nblk = (a.ncomp + CB - 1) / CB;
    const int64_t tiles = (a.N + TB * SPT - 1) / (TB * SPT);
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        int64_t i[SPT];
        bool ok[SPT];
#pragma unroll
        for (int s = 0; s < SPT; ++s) {
            i[s] = tile * (TB * SPT) + s * TB + tid;
            ok[s] = i[s] < a.N;
            if (!ok[s]) i[s] = a.N - 1;
        }
#pragma unroll 1
        for (int b = 0; b < nblk; ++b) {
            const int nrect = a.c0 + CB * b;                      // variables before the block
            const double* Ab = a.Apack + block_row0(b, a.c0) * ROW;
            // with the conditioning block contracted by K-inv-rect (a.base), the walk starts at variable c0
            const int vfirst = a.base ? a.c0 : 0;
            double acc[SPT][CB];
#pragma unroll
            for (int s = 0; s < SPT; ++s)
#pragma unroll
                for (int jj = 0; jj < CB; ++jj)
                    acc[s][jj] = (a.base && CB * b + jj < a.ncomp) ? __ldcs(a.base + (int64_t)(CB * b + jj) * a.ldb + i[s]) : 0.0;
            // ---- stage chunk 0 (and the diagonal rows) ----
            const int nchunk = (nrect - vfirst + VC - 1) / VC;
            auto stage = [&](int ch, int buf) {
                const int r0 = vfirst + ch * VC;
                const int nr = min(VC, nrect - r0);
                const double* src = Ab + (int64_t)r0 * ROW;
                double* dst = s_coef + buf * VC * ROW;
                for (int e = tid; e < nr * ROW / 2; e += TB) cp_async16(dst + 2 * e, src + 2 * e);
            };
            __syncthreads();                                      // previous block's readers are done
            {
                const double* src = Ab + (int64_t)nrect * ROW;
                for (int e = tid; e < CB * ROW / 2; e += TB) cp_async16(s_diag + 2 * e, src + 2 * e);
            }
            if (nchunk > 0) stage(0, 0);
            auto stage_table = [&](int jj) {                      // table of component CB b + jj -> buffer jj & 1
                const int j = CB * b + jj;
                if (j < a.ncomp) {
                    const double* src = a.tables + (int64_t)j * 2 * a.ntab;
                    double* dst = s_table + (jj & 1) * tbuf;
                    for (int e = tid; e < a.ntab; e += TB) cp_async16(dst + 2 * e, src + 2 * e);
                }
            };
            stage_table(0);                                       // buffer 0 was last read two barriers ago
            cp_async_commit();
            {                                                     // reference samples of the block -> L2
                const int j0 = CB * b, j1 = min(a.ncomp, j0 + CB);
                for (int j = j0; j < j1; ++j)
#pragma unroll
                    for (int s = 0; s < SPT; ++s) prefetch_l2(a.Zt + (int64_t)j * a.ldz + i[s]);
            }
            // ---- rectangular part ----
            // software pipeline over the variables: while the FMAs of variable v issue, the features of v + 1 (an
            // exp: a long dependent chain) are formed and the column of v + 2 is in flight
            double xn[SPT], fn[SPT][NS];
            if (nrect > vfirst) {
#pragma unroll
                for (int s = 0; s < SPT; ++s) features<NS>(a.Xw[(int64_t)vfirst * a.ld + i[s]], s_tab, fn[s]);
                if (vfirst + 1 < nrect) {
#pragma unroll
                    for (int s = 0; s < SPT; ++s) xn[s] = a.Xw[(int64_t)(vfirst + 1) * a.ld + i[s]];
                }
                for (int v = vfirst + 2; v < min(vfirst + PF, nrect); ++v)
#pragma unroll
                    for (int s = 0; s < SPT; ++s) prefetch_l2(a.Xw + (int64_t)v * a.ld + i[s]);
            }
#pragma unroll 1
            for (int ch = 0; ch < nchunk; ++ch) {
                if (ch + 1 < nchunk) stage(ch + 1, (ch + 1) & 1);
                cp_async_commit();
                cp_async_wait<1>();
                __syncthreads();
                const double* cbuf = s_coef + (ch & 1) * VC * ROW;
                const int r0 = vfirst + ch * VC, nr = min(VC, nrect - r0);
#pragma unroll 1
                for (int vv = 0; vv < nr; ++vv) {
                    const int v = r0 + vv;
                    double f[SPT][NS];
#pragma unroll
                    for (int s = 0; s < SPT; ++s)
#pragma unroll
                        for (int q = 0; q < NS; ++q) f[s][q] = fn[s][q];
                    if (v + 1 < nrect) {
#pragma unroll
                        for (int s = 0; s < SPT; ++s) features<NS>(xn[s], s_tab, fn[s]);
                    }
                    if (v + 2 < nrect) {
#pragma unroll
                        for (int s = 0; s < SPT; ++s) xn[s] = a.Xw[(int64_t)(v + 2) * a.ld + i[s]];
                    }
                    if (v + PF < nrect) {
#pragma unroll
                        for (int s = 0; s < SPT; ++s) prefetch_l2(a.Xw + (int64_t)(v + PF) * a.ld + i[s]);
                    }
                    // coefficients of two components at a time: 2 NS doubles = NS broadcast LDS.128 (48 / 96 B aligned)
                    const double2* c2 = reinterpret_cast<const double2*>(cbuf + vv * ROW);
#pragma unroll
                    for (int pr = 0; pr < CB / 2; ++pr) {
                        double cf[2 * NS];
#pragma unroll
                        for (int e = 0; e < NS; ++e) {
                            const double2 t = c2[pr * NS + e];
                            cf[2 * e] = t.x;
                            cf[2 * e + 1] = t.y;
                        }
#pragma unroll
                        for (int h = 0; h < 2; ++h)
#pragma unroll
                            for (int q = 0; q < NS; ++q)
#pragma unroll
                                for (int s = 0; s < SPT; ++s)
                                    acc[s][2 * pr + h] = fma(cf[h * NS + q], f[s][q], acc[s][2 * pr + h]);
                    }
                }
                __syncthreads();                                  // buffer (ch & 1) may be overwritten by chunk ch + 2
            }
            cp_async_wait<0>();
            __syncthreads();                                      // diagonal rows landed (nchunk == 0 included)
            // ---- diagonal part ----
            double zn[SPT];                                       // reference samples, one component ahead of use
#pragma unroll
            for (int s = 0; s < SPT; ++s) zn[s] = __ldcs(a.Zt + (int64_t)(CB * b) * a.ldz + i[s]);
#pragma unroll
            for (int jj = 0; jj < CB; ++jj) {
                const int j = CB * b + jj;
                if (jj > 0) {                                     // (jj = 0 landed with the diagonal rows)
                    cp_async_wait<0>();
                    __syncthreads();                              // table jj visible; everyone is done with table jj - 1
                }
                if (jj + 1 < CB) {
                    stage_table(jj + 1);
                    cp_async_commit();
                }
                if (j < a.ncomp) {
                    const double a0 = __ldg(a.a0 + j);
                    double xs[SPT], zc[SPT];
#pragma unroll
                    for (int s = 0; s < SPT; ++s) zc[s] = zn[s];
                    if (jj + 1 < CB && j + 1 < a.ncomp) {
#pragma unroll
                        for (int s = 0; s < SPT; ++s) zn[s] = __ldcs(a.Zt + (int64_t)(j + 1) * a.ldz + i[s]);
                    }
#pragma unroll
                    for (int s = 0; s < SPT; ++s) {
                        const double S = acc[s][jj] + a0;                        // offset (:4039-4043)
                        const double t = __dadd_rn(-S, zc[s]);                   // target = -offset + Zk (:4071)
                        xs[s] = interp_sorted_table(s_table + (jj & 1) * tbuf, a.ntab, a.truncate, t);
                        if (ok[s]) a.Xw[(int64_t)(a.c0 + j) * a.ld + i[s]] = xs[s];
                    }
                    if (jj + 1 < CB && j + 1 < a.ncomp) {
                        double f[SPT][NS];
#pragma unroll
                        for (int s = 0; s < SPT; ++s) features<NS>(xs[s], s_tab, f[s]);
                        const double* crow = s_diag + jj * ROW;
#pragma unroll
                        for (int j2 = jj + 1; j2 < CB; ++j2)
#pragma unroll
                            for (int q = 0; q < NS; ++q) {
                                const double c = crow[j2 * NS + q];
#pragma unroll
                                for (int s = 0; s < SPT; ++s) acc[s][j2] = fma(c, f[s][q], acc[s][j2]);
                            }
                    }
                }
            }
        }
    }
}

}  // namespace ttm_invf

// ---------------------------------------------------------------------------------------------------------------------
// K-inv-rect: the conditioning block's share of every offset as one tall-skinny FP64 GEMM
//
//   base[j][i] = sum_{v < c0} sum_q  f_q(x_iv) * A[v][q][j]          (i: sample, j: component)
//
// In a conditional inverse (X_star given, tm.py:3684-3698) the first c0 columns are known for every component, so their
// contribution does not belong in the sequential walk: K-inv-fused alone recomputes their features once per block
// of 16 components and re-reads the columns as often (ncu at C5: 17.7 GB of DRAM traffic for 3.1 GB of operands,
// long-scoreboard stalls on top).  Here a thread block owns 64 samples x 128 components; per chunk of variables the
// features are formed ONCE into shared memory, the coefficient rows arrive by cp.async (double buffered), and every
// warp updates a 32-sample x 32-component tile with DMMA m8n8k4 (16 per 8 fragment loads).  FP64 tensor-core peak
// equals the vector peak on B200 (37.1 vs 36.5 TFLOP/s), so DMMA is not chosen for rate but for operand traffic: a first
// version with a 4 x 8 register tile per thread on DFMA was co-limited by shared memory (ncu: FP64 pipe 64 %,
// shared-memory wavefronts 66 % of cycles, every LDS.128 costing >= 2 wavefronts even when broadcast), the fragment
// layout needs 4.5x fewer wavefronts per FMA.  K-inv-fused then starts its accumulators from `base` and walks only the
// columns it solves itself.
// ---------------------------------------------------------------------------------------------------------------------
namespace ttm_invr {

constexpr int TB = 256;       // 8 warps: 2 (sample halves) x 4 (component quarters), warp tile 32 x 32
constexpr int TS = 64;        // samples per tile
constexpr int TC = 128;       // components per tile
constexpr int FS = TS + 4;    // shared-memory row strides (doubles): conflict-free m8n8k4 fragment reads
constexpr int AS = TC + 4;

template <int NS>
__global__ void __launch_bounds__(TB, 2) inverse_rect_kernel(const InvRectArgs a) {
    constexpr int VC = (NS == 3) ? 8 : 4;        // variables per staged chunk
    constexpr int KR = VC * NS;                  // feature rows per chunk (24: six k = 4 steps)
    constexpr int PPT = TS * VC / TB;            // (sample, variable) pairs per thread in the feature step
    extern __shared__ double smem[];
    unsigned int* s_tab = reinterpret_cast<unsigned int*>(smem);
    double* sA = smem + ttm_exp32::TAB_DOUBLES;  // [2][KR][AS]
    double* sF = sA + 2 * KR * AS;               // [2][KR][FS]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ws = warp & 1, wc = warp >> 1;
    const int fs = tid & (TS - 1), fv = tid / TS;            // feature step: sample, first variable of the chunk
    ttm_exp32::stage_table(s_tab, tid, TB);
    const int64_t tiles = (a.N + TS - 1) / TS;
    const int nsb = (a.ncomp + TC - 1) / TC;
    const int c0p = (a.c0 + 7) / 8 * 8;                      // packed rows per component tile (zero padded)
    const int nchunk_all = (a.c0 + VC - 1) / VC;
    __syncthreads();
    for (int64_t w = blockIdx.x; w < tiles * nsb; w += gridDim.x) {
        const int64_t tile = w / nsb;
        const int sb = (int)(w - tile * nsb);
        const int64_t i0 = tile * TS;
        const int64_t irow = min(i0 + fs, a.N - 1);
        const double* Ab = a.Rpack + (int64_t)sb * c0p * NS * TC;
        const int nchunk = (a.tri < 0) ? nchunk_all
                                       : (min(a.c0, a.tri + TC * (sb + 1)) + VC - 1) / VC;   // rows beyond are zero
        auto stage = [&](int ch, int buf) {
            const double* src = Ab + (int64_t)ch * KR * TC;
            double* dst = sA + buf * KR * AS;
            for (int e = tid; e < KR * (TC / 2); e += TB) {
                const int r = e / (TC / 2), c2 = (e - r * (TC / 2)) * 2;
                ttm_invf::cp_async16(dst + r * AS + c2, src + r * TC + c2);
            }
        };
        auto load_x = [&](int ch, double (&x)[PPT]) {
#pragma unroll
            for (int p = 0; p < PPT; ++p) {
                const int v = min(ch * VC + fv + p * (TB / TS), a.c0 - 1);   // padded rows carry zero coefficients
                x[p] = __ldcs(a.Xw + (int64_t)v * a.ld + irow);
            }
        };
        auto put_features = [&](const double (&x)[PPT], int buf) {
#pragma unroll
            for (int p = 0; p < PPT; ++p) {
                double f[NS];
                ttm_invf::features<NS>(x[p], s_tab, f);
                double* dst = sF + (buf * KR + (fv + p * (TB / TS)) * NS) * FS + fs;
#pragma unroll
                for (int q = 0; q < NS; ++q) dst[q * FS] = f[q];
            }
        };
        double c[4][4][2];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) c[i][j][0] = c[i][j][1] = 0.0;
        double xr[PPT];
        __syncthreads();                                      // the previous work item's readers are done
        stage(0, 0);
        ttm_invf::cp_async_commit();
        load_x(0, xr);
        put_features(xr, 0);
        ttm_invf::cp_async_wait<0>();
        __syncthreads();
#pragma unroll 1
        for (int ch = 0; ch < nchunk; ++ch) {
            const int buf = ch & 1;
            if (ch + 1 < nchunk) {
                stage(ch + 1, buf ^ 1);
                load_x(ch + 1, xr);
            }
            ttm_invf::cp_async_commit();
            const double* F = sF + buf * KR * FS + ws * 32 + (lane >> 2);
            const double* A = sA + buf * KR * AS + wc * 32 + (lane >> 2);
#pragma unroll
            for (int k0 = 0; k0 < KR; k0 += 4) {
                const int kk = k0 + (lane & 3);
                double fa[4], cb[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) fa[i] = F[kk * FS + i * 8];
#pragma unroll
                for (int j = 0; j < 4; ++j) cb[j] = A[kk * AS + j * 8];
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) dmma_m8n8k4(c[i][j][0], c[i][j][1], fa[i], cb[j]);
            }
            if (ch + 1 < nchunk) put_features(xr, buf ^ 1);
            ttm_invf::cp_async_wait<0>();
            __syncthreads();
        }
        // ---- store: fragment (i, j) holds samples 32 ws + 8 i + lane/4, components 32 wc + 8 j + 2 (lane%4) + {0, 1} ----
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t ii = i0 + ws * 32 + i * 8 + (lane >> 2);
            if (ii < a.N) {
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int jc = sb * TC + wc * 32 + j * 8 + 2 * (lane & 3) + e;
                        if (jc < a.ncomp) __stcs(a.base + (int64_t)jc * a.ldb + ii, c[i][j][e]);
                    }
            }
        }
    }
}

}  // namespace ttm_invr

size_t ttm_inverse_rect_rpack_doubles(int ncomp, int c0, int ns) {
    const int nsb = (ncomp + ttm_invr::TC - 1) / ttm_invr::TC;
    return (size_t)nsb * ((c0 + 7) / 8 * 8) * ns * ttm_invr::TC;
}

cudaError_t ttm_launch_inverse_rect(const InvRectArgs& a, int sm_count, cudaStream_t st) {
    using namespace ttm_invr;
    if (a.N == 0 || a.ncomp == 0 || a.c0 == 0) return cudaSuccess;
    if (a.ns != 3 && a.ns != 6) return cudaErrorInvalidValue;
    const int64_t work = (a.N + TS - 1) / TS * ((a.ncomp + TC - 1) / TC);
    const int kr = (a.ns == 3 ? 8 : 4) * a.ns;
    const size_t smem = sizeof(double) * (size_t)(ttm_exp32::TAB_DOUBLES + 2 * kr * (AS + FS));
    cudaError_t e;
    auto launch = [&](auto kernel) -> cudaError_t {
        if ((e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
        int per_sm = 0;
        if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, TB, smem)) != cudaSuccess) return e;
        int64_t grid = (int64_t)sm_count * (per_sm > 0 ? per_sm : 1);
        if (grid > work) grid = work;
        kernel<<<(unsigned)grid, TB, smem, st>>>(a);
        return cudaGetLastError();
    };
    return a.ns == 3 ? launch(inverse_rect_kernel<3>) : launch(inverse_rect_kernel<6>);
}

size_t ttm_inverse_fused_apack_doubles(int ncomp, int c0, int ns) {
    const int nblk = (ncomp + ttm_invf::CB - 1) / ttm_invf::CB;
    return (size_t)ttm_invf::block_row0(nblk, c0) * ttm_invf::CB * ns;
}

cudaError_t ttm_launch_inverse_fused(const InvFusedArgs& a, int sm_count, cudaStream_t st) {
    using namespace ttm_invf;
    if (a.N == 0 || a.ncomp == 0) return cudaSuccess;
    if ((a.ns != 3 && a.ns != 6) || a.ntab > TTM_INVERSE_FUSED_MAX_NTAB) return cudaErrorInvalidValue;
    const int64_t tiles = (a.N + TB * SPT - 1) / (TB * SPT);
    // exp table, coefficient chunks, diagonal rows, 2 x [values | abscissae]
    const size_t smem = sizeof(double) * (size_t)(ttm_exp32::TAB_DOUBLES + (2 * VC + CB) * CB * a.ns + 4 * a.ntab);
    cudaError_t e;
    // persistent grid = resident blocks (a block past residency would run alone on its SM at the end)
    auto launch = [&](auto kernel) -> cudaError_t {
        if ((e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
        int per_sm = 0;
        if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, TB, smem)) != cudaSuccess) return e;
        int64_t grid = (int64_t)sm_count * (per_sm > 0 ? per_sm : 1);
        if (grid > tiles) grid = tiles;
        kernel<<<(unsigned)grid, TB, smem, st>>>(a);
        return cudaGetLastError();
    };
    return a.ns == 3 ? launch(inverse_fused_kernel<3>) : launch(inverse_fused_kernel<6>);
}
