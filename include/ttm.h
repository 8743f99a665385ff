/*
 * libttm -- C ABI of the B200-native triangular-transport hot path.
 *
 * Drop-in boundary for the data-parallel path of MaxRamgraber/Triangular-Transport-Toolbox
 * (`transport_map.py`, "tm.py" below): basis assembly, integrated-rectifier objective + gradient,
 * separable-monotonicity least-squares contractions, forward map, inverse map and the
 * log-determinants of the density evaluators.  The reference has no FFI of its own (it is one
 * pure-Python file); each entry point below names the reference function(s) it replaces, and
 * INTEGRATION.md shows the ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 on success and a negative code on failure; the message is
 *     available from ttm_last_error() (thread local).  No exceptions cross the ABI, and the
 *     caller allocates every output buffer.
 *   - pointers are DEVICE pointers unless the parameter name starts with `host_`.
 *   - sample matrices on the device are column-major ("Xt"): column v starts at Xt + v*ld,
 *     ld >= N.  ttm_standardize_transpose builds that layout from a row-major (N, D) array.
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream).  Calls on one
 *     ttm_plan must not overlap in time (the plan owns its reduction workspace).
 *   - there is no CPU fallback: every entry point launches sm_100a kernels.
 */
#ifndef TTM_H
#define TTM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ttm_ctx ttm_ctx;   /* per-map constants: device, quadrature rule, rectifier */
typedef struct ttm_plan ttm_plan; /* one compiled map component (term tables + workspace)  */

#define TTM_OK 0
#define TTM_ERR_CUDA -1
#define TTM_ERR_ARG -2
#define TTM_ERR_LIMIT -3 /* plan exceeds a compiled limit (order > 20, > 8 special inner terms), or a table is longer
                          * than TTM_INVERSE_FUSED_MAX_NTAB (ttm_inverse_fused, ttm_inverse_fused_split) */

/* longest table ttm_inverse_fused and ttm_inverse_fused_split accept: each block stages two [values | abscissae]
 * tables (4 ntab doubles = 64 KB at the limit) in shared memory next to its coefficient operands */
#define TTM_INVERSE_FUSED_MAX_NTAB 2048

/* element type of a caller's row-major sample array (the *_ld entry points); float32 is widened on load */
#define TTM_DTYPE_F64 0
#define TTM_DTYPE_F32 1

#define TTM_WHICH_NONMON 0
#define TTM_WHICH_MON 1
#define TTM_WHICH_DMON 2

const char* ttm_last_error(void);
int ttm_version(void);

/* 1 if host_ptr lies in page-locked (pinned / registered) host memory: such inputs are copied to the device directly,
 * pageable ones through the library's pinned staging buffers */
int ttm_host_is_pinned(const void* host_ptr, int* host_out);
/* device query used by the host to size grids and scratch buffers */
int ttm_device_sm_count(int device, int* host_sm_count);

/* ---- map-level constants -------------------------------------------------------------------
 * replaces: transport_map.__init__ option handling, tm.py:186-225 (rectifier, delta, GL nodes) */
int ttm_ctx_create(int device, ttm_ctx** host_out);
int ttm_ctx_destroy(ttm_ctx* ctx);
/* xis/ws are computed on the host exactly as tm.py:211-221 and uploaded once */
int ttm_ctx_set_quadrature(ttm_ctx* ctx, const double* host_xis, const double* host_ws, int Q);
/* rect: 0 exponential, 1 softplus, 2 squared, 3 expneg, 4 explinearunit (tm.py:4981-5018) */
int ttm_ctx_set_rectifier(ttm_ctx* ctx, int rect, double delta);
/* resident blocks per SM of one K-objgrad launch (0 = default 4).  With 2, launches issued on two streams
 * (two components fitted by two host threads) share every SM and their phases overlap (+16 % throughput). */
int ttm_ctx_set_blocks_per_sm(ttm_ctx* ctx, int blocks_per_sm);

/* K-objgrad kernel selection: 0 (default) = the tile kernel (csrc/ttm_objgrad_tile.cu) whenever the component is in
 * its class (order <= 3 Hermite functions, exponential rectifier; ttm_plan_info), 1 = always the general kernel.
 * Both compute the same (J, grad); the switch exists for A/B parity runs. */
int ttm_ctx_set_objgrad_kernel(ttm_ctx* ctx, int mode);

/* ---- component plans -----------------------------------------------------------------------
 * replaces: function_constructor_alternative / function_derivative_constructor_alternative
 * (tm.py:1263-2134): instead of exec'ing generated source, the host compiles the term lists into
 * an int32 blob + a double blob (layout: csrc/ttm_common.cuh, enum H_*), uploaded here.          */
int ttm_plan_create(ttm_ctx* ctx, const int32_t* host_iblob, int64_t n_int, const double* host_dblob,
                    int64_t n_double, ttm_plan** host_out);
/* host_info[4] = {in the tile kernel's class (0/1), union of used nonmonotone slots (bit 2*order+hf),
 *                 monotone terms with an outer product over x_<c, m = m_non + m_mon} */
int ttm_plan_info(ttm_plan* plan, int* host_info);
/* re-upload the double blob only (special-term centres/scales move on reset(), tm.py:800) */
int ttm_plan_update_doubles(ttm_plan* plan, const double* host_dblob, int64_t n_double);
int ttm_plan_destroy(ttm_plan* plan);

/* ---- K-std -----------------------------------------------------------------------------------
 * replaces: standardize, tm.py:750-787 ('standard' mode: mean and population std per column).
 * X is row-major (N, D) on the device; scratch holds >= 4*sm_count*256 doubles.                 */
int ttm_colstats(ttm_ctx* ctx, const double* X, int64_t N, int D, double* mean, double* std, double* scratch,
                 void* stream);
/* Xt[v*ld + i] = (X[i*D + v] - mean[v]) / std[v]   (mean == NULL: plain transpose)              */
int ttm_standardize_transpose(ttm_ctx* ctx, const double* X, int64_t N, int D, const double* mean,
                              const double* std, double* Xt, int64_t ld, void* stream);
/* The same two for a caller's row-major array read in place: row i at (char*)X + i*ldx*elemsize, ldx >= D (e.g. a
 * column slice X[:, a:b] of a wider array), elements of type `dtype` (TTM_DTYPE_F64 / TTM_DTYPE_F32, widened to double
 * as they are loaded, so a float32 array gives the bits its float64 copy gives).  The entry points above are these with
 * (TTM_DTYPE_F64, ldx = D).  TTM_ERR_ARG on ldx < D or an unknown dtype. */
int ttm_colstats_ld(ttm_ctx* ctx, const void* X, int dtype, int64_t ldx, int64_t N, int D, double* mean, double* std,
                    double* scratch, void* stream);
int ttm_standardize_transpose_ld(ttm_ctx* ctx, const void* X, int dtype, int64_t ldx, int64_t N, int D,
                                 const double* mean, const double* std, double* Xt, int64_t ld, void* stream);
/* X[i*ldx + v] = Xt[v*ld + i] * std[v] + mean[v]   (un-standardise, tm.py:3700-3704; NULL: transpose) */
int ttm_transpose_back(ttm_ctx* ctx, const double* Xt, int64_t ld, int64_t N, int D, const double* mean,
                       const double* std, double* X, int64_t ldx, void* stream);

/* ---- K-basis ---------------------------------------------------------------------------------
 * replaces: generated fun_mon_k / fun_nonmon_k / der_fun_mon_k and precalculate, tm.py:789-821.
 * Psi is row-major (N, m) like the reference's Psi_mon[k] / Psi_nonmon[k] / der_Psi_mon[k].      */
int ttm_basis_eval(ttm_plan* plan, int which, const double* Xt, int64_t ld, int64_t N, double* Psi, void* stream);

/* ---- K-objgrad (integrated rectifier) --------------------------------------------------------
 * replaces: objective_function tm.py:3300-3433 + objective_function_jacobian :3435-3635 (the two
 * scipy callbacks of worker_task :3252-3257), incl. s :2439-2547 and GaussQuadrature :4202-4278.
 * host_coeffs = [coeffs_nonmon | coeffs_mon] (m doubles); host_out = [J, dJ/dcoeffs] (1+m doubles),
 * WITHOUT the regularisation terms (the host adds them, tm.py:3382-3431 / :3575-3633).
 * ttm_objgrad_ir = set_coeffs + launch + get_out (synchronises `stream`).                        */
/* Gram mode: dJ/da = G a + h with G = Psi_non^T Psi_non / N (ttm_gram, once per ensemble, like the reference's
 * precalculate()).  When on, the nonmonotone slots of host_out hold h_j = mean_i M_i psi_ij only and the caller
 * adds G a; the kernel then needs one sweep over the columns x_<c instead of two.  Fails with TTM_ERR_LIMIT if
 * a nonmonotone polynomial order exceeds 3. */
int ttm_plan_set_gram_mode(ttm_plan* plan, int on);
int ttm_plan_set_coeffs(ttm_plan* plan, const double* host_coeffs, void* stream);
int ttm_objgrad_ir_launch(ttm_plan* plan, const double* Xt, int64_t ld, int64_t N, void* stream);
int ttm_plan_get_out(ttm_plan* plan, double* host_out, int n, void* stream);
int ttm_objgrad_ir(ttm_plan* plan, const double* Xt, int64_t ld, int64_t N, const double* host_coeffs,
                   double* host_out, void* stream);

/* ---- K-S --------------------------------------------------------------------------------------
 * replaces: s, tm.py:2439-2567, called per component by map :2428-2435.
 * Uses the coefficients last set with ttm_plan_set_coeffs.  S_out: N doubles.                    */
int ttm_eval_s_ir(ttm_plan* plan, const double* Xt, int64_t ld, int64_t N, double* S_out, void* stream);
/* separable arm (tm.py:2550-2558) and the derivative d_k S_k = der_Psi_mon . coeffs_mon used by the
 * density evaluators (tm.py:2627-2633, :2695-2701).  Xd is the matrix the derivative basis is
 * evaluated on (the reference passes the UNstandardised samples there).  Either output may be NULL. */
int ttm_sep_eval(ttm_plan* plan, const double* Xt, int64_t ld, int64_t N, double* S_out, const double* Xd,
                 int64_t ldd, double* dS_out, void* stream);

/* ---- K-pullback / K-logdet ----------------------------------------------------------------------
 * replaces: the change-of-variables bookkeeping of evaluate_pullback_density tm.py:2680-2712 and
 * evaluate_pushforward_density :2618-2644, one component at a time (S, dS from ttm_sep_eval):
 *   mode 0 (pullback):    acc[i] += -S_i^2/2 - log(2 pi)/2 + log(dS_i / sigma)
 *   mode 1 (pushforward): acc[i] -= log(dS_i / sigma)
 * ttm_density_finish: out[i] = exp(acc[i] + log_target[i])  (log_target may be NULL).             */
int ttm_density_accumulate(ttm_ctx* ctx, double* acc, const double* S, const double* dS, double sigma, int mode,
                           int64_t N, void* stream);
int ttm_density_finish(ttm_ctx* ctx, const double* acc, const double* log_target, double* out, int64_t N,
                       void* stream);

/* ---- K-logdet-IR ------------------------------------------------------------------------------
 * replaces: nothing -- the reference's density evaluators assert separable monotonicity (tm.py:2569, :2646).  The
 * log-determinant term of an integrated-rectifier component for evaluate_log_pullback_density /
 * evaluate_log_pushforward_density: l_i = log d_c S_k(x_i) = log(g(r_i) + delta), r_i = sum_j b_j psi^mon_j(x_i)
 * (l_i = r_i for the exponential rectifier with delta = 0), the same per-sample quantity as the objective's -log
 * term.  Xt: standardised samples (column-major, all columns <= c); S: K-S output (ttm_eval_s_ir), read in mode 0 only.
 *   mode 0 (pullback):    acc[i] += -S_i^2/2 - log(2 pi)/2 + l_i - log(sigma)
 *   mode 1 (pushforward): acc[i] -= l_i - log(sigma)
 * Coefficients as last set with ttm_plan_set_coeffs.  One thread per sample, no atomics (bit-reproducible).
 * TTM_ERR_LIMIT for polynomial order > 32 or > 16 special inner terms (as ttm_inverse_bisect). */
int ttm_ir_logdet_accumulate(ttm_plan* plan, const double* Xt, int64_t ld, int64_t N, const double* S, double sigma,
                             int mode, double* acc, void* stream);

/* K-map-fused / K-pullback: all D components of a (small) separable map on row-major samples in ONE launch.
 * replaces: map tm.py:2391-2437 + the whole of evaluate_pullback_density :2646-2712 / the log-determinant loop of
 * evaluate_pushforward_density :2618-2644 (the per-component entry points above remain for large maps).
 * host_plans[D]: the components, coefficients as last set with ttm_plan_set_coeffs; host_sigma[D]: the X_std entry
 * dividing d_k S_k (the reference uses X_std[k] in the pullback and X_std[k+skip] in the pushforward);
 * X: device row-major (n, Dtot) UNstandardised samples; mean/std: device [Dtot] or both NULL.
 *   mode 0: out[i] = pullback density, Z (optional, row-major (n, D)) = map output
 *   mode 1: out[i] = exp(log_target[i] - sum_k log(d_k S_k / sigma_k))
 *   mode 2: Z = map output only
 *   mode 3: out[i] = log pullback density of the fitted map (Z optional as in mode 0)
 *   mode 4: out[i] = log_target[i] - sum_k log(d_k S_k / sigma_k)
 * Modes 3 and 4 evaluate d_k S_k on the STANDARDISED samples and return the log (no exp); host_sigma[k] =
 * X_std[k+skip] there (evaluate_log_pullback_density / evaluate_log_pushforward_density). */
int ttm_map_fused(ttm_ctx* ctx, ttm_plan* const* host_plans, int D, const double* host_sigma, const double* X, int64_t n,
                  int Dtot, const double* mean, const double* std, const double* log_target, int mode, double* Z,
                  double* out, void* stream);
/* the same on a caller's row-major array read in place (row stride ldx >= Dtot, dtype as for ttm_colstats_ld) */
int ttm_map_fused_ld(ttm_ctx* ctx, ttm_plan* const* host_plans, int D, const double* host_sigma, const void* X, int dtype,
                     int64_t ldx, int64_t n, int Dtot, const double* mean, const double* std, const double* log_target,
                     int mode, double* Z, double* out, void* stream);

/* ---- K-gram (FP64 tensor-core DMMA) ----------------------------------------------------------
 * replaces: the dense contractions of worker_task_monotone, tm.py:2966-2975 (QR / A_sqrt) and
 * :3031-3050 (ridge normal equations).  G = [Psi_non | Psi_mon]^T [Psi_non | Psi_mon], row-major
 * (M, M), M = m_non + m_mon.  scratch: as many (M8*M8) blocks as fit are used for split-N partials. */
int ttm_gram(ttm_plan* plan, const double* Xt, int64_t ld, int64_t N, double* G, double* scratch,
             int64_t scratch_doubles, void* stream);
/* the same, but only the entries G[i][j] with max(i, j) >= 64*(first_col/64) are computed (the others are set to 0):
 * Psi^T [Psi_mon] and the neighbouring tiles.  When the components of a map share their nonmonotone basis (the term
 * list of one is a prefix of another's), the leading block Psi_non^T Psi_non and its Cholesky factor come from ONE
 * full Gram of the longest list, and every component only needs this tail. */
int ttm_gram_tail(ttm_plan* plan, const double* Xt, int64_t ld, int64_t N, int first_col, double* G, double* scratch,
                  int64_t scratch_doubles, void* stream);

/* ---- forward map of a wide separable map as a GEMM --------------------------------------------
 * replaces: the nonmonotone sums of `s` (tm.py:2550-2558) for ALL components of `map` (:2391-2437) at once.  With
 * every column known, sum_{v<c} sum_q f_q(x_iv) a[v][q][c] is a (block-triangular) FP64 GEMM: ttm_map_rect runs
 * K-inv-rect over `rows` variables with component j using the rows v < first + j (Rpack as for
 * ttm_inverse_fused_split, zero elsewhere; tiles skip the rows no component of theirs uses), base = [ncomp][ldb].
 * ttm_sep_eval_base then adds the constant a0 and the monotone terms of one component: S = base + a0 + mon(x_c).
 * The per-component path (ttm_sep_eval) re-reads every predecessor column for every component: 8 n D^2 / 2 bytes. */
int ttm_map_rect(ttm_ctx* ctx, const double* Xt, int64_t ld, int64_t N, int ncomp, int rows, int ns, int first,
                 const double* Rpack, double* base, int64_t ldb, void* stream);
int ttm_sep_eval_base(ttm_plan* plan, const double* Xt, int64_t ld, int64_t N, const double* base, double a0,
                      double* S_out, void* stream);

/* ---- K-sepobj ---------------------------------------------------------------------------------
 * replaces: the sample-dependent part of fun_mon_objective, tm.py:2990-3006.
 * host_out[0] = sum_i log dS_i, host_out[1+j] = sum_i dPsi_ij / dS_i with
 * dS_i = sum_j (b_j + delta) dPsi_ij.  The m_mon x m_mon algebra with A stays on the host.       */
int ttm_sep_objgrad(ttm_plan* plan, const double* Xt, int64_t ld, int64_t N, const double* host_b,
                    double* host_out, void* stream);
/* the same in two halves, so that the independent components' L-BFGS-B iterations (Pool.map over worker_task_monotone,
 * tm.py:2837-2845) advance in lockstep: launch every component that wants (f, g), then collect them all.  One launch
 * per plan may be outstanding. */
int ttm_sep_objgrad_launch(ttm_plan* plan, const double* Xt, int64_t ld, int64_t N, const double* host_b, void* stream);
int ttm_sep_objgrad_wait(ttm_plan* plan, double* host_out, void* stream);
/* fun_mon_objective (tm.py:2978-3006) whole, for n components in one call: ONE batched K-sepobj launch per 64
 * components (blockIdx.y = component; the plans' descriptors are registered in a device array on first use), then each
 * result is collected and the reduced objective assembled on the host,
 *   fg[i][0]   = b^T A b / 2 - (sum_s log dS_s) / n_total + b^T c,
 *   fg[i][1+j] = (A b)_j - (sum_s dPsi_sj / dS_s) / n_total + c_j,
 * with A = host_A[i] (m_mon x m_mon, row-major, symmetric), c = host_c[i] = delta * rowsum(A), b = host_b[i].
 * n_total = number of samples of the whole ensemble.  A plan may appear once per call. */
int ttm_sep_reduced_batch(int n, ttm_plan* const* plans, const double* Xt, int64_t ld, int64_t N, double n_total,
                          const double* const* host_b, const double* const* host_A, const double* const* host_c,
                          double* const* host_fg, void* stream);

/* ---- K-inv -----------------------------------------------------------------------------------
 * replaces: vectorized_root_search_alternate tm.py:3987-4084 (table) and
 * vectorized_root_search_bisection :3798-3985, called per component by inverse_map :3639-3796.
 * Xt is the working matrix: columns < c hold the solved (standardised) values, column c is written. */
/* table[ntab..2*ntab) = abscissae (in); table[0..ntab) = monotone part at fakeX (out), tm.py:4047-4058 */
int ttm_mon_table(ttm_plan* plan, int ntab, double* table, void* stream);
/* table = [sorted values | abscissae in the same order] (scipy interp1d sorts, assume_sorted=False) */
int ttm_inverse_table(ttm_plan* plan, double* Xt, int64_t ld, int64_t N, const double* z, const double* table,
                      int ntab, int truncate, void* stream);
/* K-inv-fused: the whole component loop of inverse_map (tm.py:3684-3698 calling :3987-4084) in one launch for maps
 * whose nonmonotone terms are constants + per-variable Hermite-function groups of order <= 3 (every other map takes
 * ttm_inverse_table per component).  Component j = 0..ncomp-1 solves column c0 + j of Xw from the columns before it;
 * Zt holds its reference samples at Zt + j*ldz; tables = [ncomp][2*ntab] as for ttm_inverse_table; a0[j] = sum of
 * the constant terms' coefficients.  Apack (ttm_inverse_fused_apack_size doubles) holds coefficient*scale in blocks
 * of 16 components: block b = rows v = 0 .. c0 + 16 b + 15, row = [16 components][ns slots], zero where variable v is
 * not a predecessor of the component; ns = 3: slots {He1, He2 e^{-x^2/4}, He3 e^{-x^2/4}}, ns = 6: {He1, He1 e, He2,
 * He2 e, He3, He3 e}.  ntab > TTM_INVERSE_FUSED_MAX_NTAB fails with TTM_ERR_LIMIT before any launch. */
int ttm_inverse_fused_apack_size(int ncomp, int c0, int ns, int64_t* host_doubles);
int ttm_inverse_fused(ttm_ctx* ctx, double* Xw, int64_t ld, int64_t N, const double* Zt, int64_t ldz, int ncomp, int c0,
                      int ns, const double* Apack, const double* a0, const double* tables, int ntab, int truncate,
                      void* stream);
/* The same result in two launches for a conditional inverse with a wide conditioning block (X_star given, c0 > 0):
 * K-inv-rect first contracts the c0 known columns with every component's coefficients as one tall-skinny FP64 GEMM,
 * base[j][i] = sum_{v<c0} sum_q f_q(x_iv) Rpack[j/128][v][q][j%128] (features formed once per sample and variable
 * instead of once per block of 16 components), then K-inv-fused starts from `base` and walks only the columns it
 * solves.  Rpack (ttm_inverse_rect_rpack_size doubles) = [ceil(ncomp/128)][c0 rounded up to 8][ns][128], zero padded;
 * base = device scratch [ncomp][ldb], 16-byte aligned, ldb even and >= N.  ntab > TTM_INVERSE_FUSED_MAX_NTAB fails
 * with TTM_ERR_LIMIT before either launch. */
int ttm_inverse_rect_rpack_size(int ncomp, int c0, int ns, int64_t* host_doubles);
int ttm_inverse_fused_split(ttm_ctx* ctx, double* Xw, int64_t ld, int64_t N, const double* Zt, int64_t ldz, int ncomp,
                            int c0, int ns, const double* Apack, const double* Rpack, const double* a0,
                            const double* tables, int ntab, int truncate, double* base, int64_t ldb, void* stream);
/* separable != 0: monotone part is linear in the coefficients; else Gauss-Legendre of the rectifier.
 * host_not_converged receives the number of samples stopped at max_iter (the reference warns).   */
int ttm_inverse_bisect(ttm_plan* plan, double* Xt, int64_t ld, int64_t N, const double* z, int separable,
                       int max_iter, int* host_not_converged, void* stream);

/* ---- measurement ------------------------------------------------------------------------------
 * dependent-free DFMA chains on every SM; writes the achieved FP64 TFLOP/s (2 flop per DFMA).    */
int ttm_fp64_peak(ttm_ctx* ctx, double* host_tflops);

#ifdef __cplusplus
}
#endif
#endif /* TTM_H */
