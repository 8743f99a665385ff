// Internal launcher interface between the kernel translation units and the C ABI (ttm_api.cu).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/ttm.h"
#include "ttm_common.cuh"

struct ObjArgs {
    PlanView P;
    const double* Xt;      // standardised samples, column-major: column v at Xt + v*ld
    int64_t ld, N;
    const double* coeffs;  // device [m_non + m_mon]
    const double* xis;     // device [Q] Gauss-Legendre nodes
    const double* ws;      // device [Q] weights
    int Q;
    double wsum;           // sum of the weights (host, same summation order as the nodes)
    int rect;
    double delta;
    double* partials;      // device [max_grid][1+m]
    unsigned int* counter; // device, zero on entry, zero on exit
    double* out;           // device [1+m]: J, grad
    double* out_host;      // pinned host mirror of `out` (mapped): written by the last block together with `out`,
    unsigned long long* flag_host;   // followed by a system fence and the sequence number of the launch, so that the
    unsigned long long seq;          // host can wait for the result without a D2H copy and a stream synchronisation
    double* S_out;         // device [N] (value-only mode)
    int max_grid;
    int gram_mode;         // 1: nonmonotone gradient slots return h_j = sum_i M_i psi_ij / N (host adds G a)
    int ch_rows;           // rows per chunk (set by the dispatcher)
    int blocks_per_sm;     // resident blocks per SM of one launch (0: default); smaller grids let launches on
                           // different streams co-reside on an SM so that their phases overlap
    // tile kernel (ttm_objgrad_tile.cu): eligibility and table facts computed from the host blob at plan creation
    int tile_ok;           // 1: order <= 3 Hermite-function component without special/multivariate nonmonotone terms
    int dense_mask;        // union over the dense groups of the used slots, bit 2*order+hf
    int n_out_terms;       // monotone terms with an outer product over x_<c
    const double* h_xis;   // HOST copies of the quadrature rule: the tile kernel's launcher turns them into the
    const double* h_ws;    // node-constant table it passes as a kernel parameter
    int lay[16];           // shared-memory layout of the launched kernel (offsets in doubles), computed by its launcher
};

#define TTM_TILE_MAXMON 8   // monotone terms per component handled by the tile kernel
#define TTM_TILE_MAXOUT 4   // ... of which with an outer product
#define TTM_TILE_MAXQ 128   // quadrature nodes (6 constants per node travel as a 6 KB kernel parameter)

cudaError_t ttm_launch_objgrad(const ObjArgs& a, bool grad, int sm_count, cudaStream_t st);
// tile kernel; cudaErrorNotSupported if the plan is outside its class
cudaError_t ttm_launch_objgrad_tile(const ObjArgs& a, bool grad, int sm_count, cudaStream_t st);

// column statistics + standardise + transpose (reference: standardize, transport_map.py:750-787).
// X: row-major (N, >= D) samples of dtype TTM_DTYPE_F64 / TTM_DTYPE_F32 with row stride ldx
cudaError_t ttm_launch_colstats(const void* X, int dtype, int64_t ldx, int64_t N, int D, double* mean, double* std,
                                double* scratch, int sm_count, cudaStream_t st);
cudaError_t ttm_launch_standardize_transpose(const void* X, int dtype, int64_t ldx, int64_t N, int D,
                                             const double* mean, const double* std, double* Xt, int64_t ld,
                                             cudaStream_t st);
cudaError_t ttm_launch_transpose_back(const double* Xt, int64_t ld, int64_t N, int D, const double* mean,
                                      const double* std, double* X, int64_t ldx, int col0, cudaStream_t st);

// basis matrices (reference: generated fun_mon_k / fun_nonmon_k / der_fun_mon_k + precalculate :789-821)
cudaError_t ttm_launch_basis(const PlanView& P, int which, const double* Xt, int64_t ld, int64_t N, double* Psi,
                             cudaStream_t st);

cudaError_t ttm_launch_basis_concat(const PlanView& P, const double* Xt, int64_t ld, int64_t n, double* Psi,
                                    int64_t ldp, cudaStream_t st);

// separable-monotonicity evaluation: S_k and d_k S_k per sample (reference: s :2550-2558, densities :2620-2641)
cudaError_t ttm_launch_sep_eval(const PlanView& P, const double* Xt, int64_t ld, int64_t N, const double* coeffs,
                                double* S_out, const double* Xd, int64_t ldd, double* dS_out, int sm_count,
                                cudaStream_t st, const double* base = nullptr, double a0 = 0.0);

cudaError_t ttm_launch_density_acc(double* acc, const double* S, const double* dS, double sigma, int mode, int64_t N,
                                   cudaStream_t st);
cudaError_t ttm_launch_density_finish(const double* acc, const double* logt, double* out, int64_t N, cudaStream_t st);

// all components of a small separable map in one launch (ttm_sep.cu: K-map-fused / K-pullback)
struct FusedComp {
    PlanView P;
    const double* coeffs;  // device [m_non + m_mon]
    double sigma;          // X_std entry dividing d_k S_k in the densities
};
struct FusedMapArgs {
    const FusedComp* comps;  // device [D]
    int D, Dtot;
    const void* X;           // device row-major (n, >= Dtot) UNstandardised samples, row stride ldx
    int dtype;               // TTM_DTYPE_F64 / TTM_DTYPE_F32 (widened on load)
    int64_t ldx;
    int64_t n;
    const double* mean;      // device [Dtot] or NULL (no standardisation)
    const double* sd;
    const double* logt;      // device [n] or NULL (mode 1)
    int mode;                // 0 pullback density (+ Z if given), 1 pushforward density, 2 map only,
                             // 3 / 4 log pullback / log pushforward density (derivative basis on the standardised samples)
    double* Z;               // device row-major (n, D) or NULL
    double* out;             // device [n] (modes 0, 1)
};
cudaError_t ttm_launch_map_fused(const FusedMapArgs& a, cudaStream_t st);

// Gram matrix of [Psi_non | Psi_mon] (reference: worker_task_monotone :2966-2975, :3031-3050)
cudaError_t ttm_launch_gram(const PlanView& P, const double* Xt, int64_t ld, int64_t N, int first_col, double* G,
                            double* scratch, int64_t scratch_doubles, int sm_count, cudaStream_t st);

// reduced separable objective: sum log dS, colsum(dPsi/dS) (reference: fun_mon_objective :2978-3018)
// K-sepobj for several components in one launch
#define TTM_SEP_BATCH_MAX 64
struct SepBatchItem {
    PlanView P;
    const double* b;               // coefficients (mapped host memory, written by the host before the launch)
    double* d_b;
    double* partials;
    unsigned int* counter;
    double* out;
    double* out_host;
    unsigned long long* flag_host;
};
struct SepBatchLaunch {
    unsigned long long seq[TTM_SEP_BATCH_MAX];
    int item[TTM_SEP_BATCH_MAX];
};
cudaError_t ttm_launch_sepobj_batch(const SepBatchItem* d_items, const SepBatchLaunch& L, int nact, int max_mm,
                                    const double* Xt, int64_t ld, int64_t N, double delta, int max_grid, int sm_count,
                                    cudaStream_t st);
cudaError_t ttm_launch_sepobj(const PlanView& P, const double* Xt, int64_t ld, int64_t N, const double* b,
                              double* d_b, double delta, double* partials, unsigned int* counter, double* out,
                              double* out_host, unsigned long long* flag_host, unsigned long long seq, int max_grid,
                              int sm_count, cudaStream_t st);

struct InvArgs {
    PlanView P;
    double* Xt;            // working sample matrix (columns < c already solved); column c is written
    int64_t ld, N;
    const double* z;       // device [N] target values of this component
    const double* coeffs;  // device [m_non + m_mon]
    // integrated rectifier
    const double* xis;
    const double* ws;
    int Q;
    double wsum;
    int rect;
    double delta;
    int separable;
    // table mode
    const double* table;   // device [ntab] sorted monotone-part values, abscissae in table + ntab
    int ntab;
    int truncate;
    // bisection quirk bookkeeping (transport_map.py:3952): iterations used by samples >= 1
    int64_t first, count;  // sample range handled by this launch
    int max_iter;
    int* iter_max;         // device scalar
    int* not_converged;    // device counter of samples stopped at max_iter
};

// fused multi-component table inverse (ttm_inverse_fused.cu)
struct InvFusedArgs {
    double* Xw;            // working sample matrix, column-major: columns < c0 filled (conditioning block), c0.. written
    int64_t ld, N;
    const double* Zt;      // reference samples of component j at Zt + j*ldz
    int64_t ldz;
    int ncomp, c0;         // component j solves column c0 + j from the columns < c0 + j
    int ns;                // slots per (variable, component): 3 = {He1, He2 e, He3 e}, 6 = all plain/HF slots of order 1..3
    const double* Apack;   // packed coefficient*scale, see ttm_inverse_fused.cu
    const double* a0;      // [ncomp] constant part of the offset
    const double* tables;  // [ncomp][2*ntab] sorted values | abscissae
    int ntab, truncate;
    const double* base;    // NULL, or [ncomp][ldb]: offsets' share of the columns < c0 (K-inv-rect); the walk then starts at c0
    int64_t ldb;
};
// K-inv-rect: base[j][i] = sum_{v<c0} sum_q f_q(Xw[v][i]) Rpack[j/128][v][q][j%128]
struct InvRectArgs {
    const double* Xw;
    int64_t ld, N;
    int ncomp, c0, ns;
    const double* Rpack;   // [ceil(ncomp/128)][c0 rounded up to 8][ns][128], zero padded
    double* base;          // [ncomp][ldb]
    int64_t ldb;
    int tri;               // -1: every component uses all c0 rows; >= 0: component j uses the rows v < tri + j only (the
                           // forward map: all columns known, Rpack is triangular) -- tile sb stops at tri + 128 (sb + 1)
};
cudaError_t ttm_launch_inverse_rect(const InvRectArgs& a, int sm_count, cudaStream_t st);
size_t ttm_inverse_rect_rpack_doubles(int ncomp, int c0, int ns);
cudaError_t ttm_launch_inverse_fused(const InvFusedArgs& a, int sm_count, cudaStream_t st);
size_t ttm_inverse_fused_apack_doubles(int ncomp, int c0, int ns);

cudaError_t ttm_launch_inverse_table(const InvArgs& a, int sm_count, cudaStream_t st);
cudaError_t ttm_launch_inverse_bisect(const InvArgs& a, int sm_count, cudaStream_t st);
cudaError_t ttm_launch_mon_table(const PlanView& P, const double* coeffs, int ntab, double* table, cudaStream_t st);
// K-logdet-IR (ttm_inverse.cu); cudaErrorInvalidValue if the plan has more slots than MonEval holds
cudaError_t ttm_launch_ir_logdet(const PlanView& P, const double* coeffs, const double* Xt, int64_t ld, int64_t N,
                                 const double* S, double sigma, int rect, double delta, int mode, double* acc,
                                 cudaStream_t st);

// FP64 pipe micro-benchmark (dependent-free DFMA chains); returns flop count per launch
cudaError_t ttm_launch_fp64_peak(double* sink, int iters, int grid, int block, cudaStream_t st);
