// K-inv-table / K-inv-bisect: per-sample inversion of one map component, S_k(x_<c, x_c) = z_k.
// K-logdet-IR (end of file): log d_c S_k of an integrated-rectifier component for the log-density evaluators.
//
// Reference: inverse_map transport_map.py:3639-3796 (host loop over k, sequential);
//            vectorized_root_search_alternate :3987-4084 (1001-point table + scipy interp1d linear);
//            vectorized_root_search_bisection :3798-3985 (bracket +-2, widen x2, bisect on |S-z| <= 1e-9).
// One thread per sample (R_OBJ samples per thread for the nonmonotone offset sweep); the launch for
// component k reads the already solved columns < c of the working matrix Xt and writes column c.

#include "ttm_common.cuh"
#include "ttm_kernels.h"
#include "ttm_sweep.cuh"

namespace {

constexpr int T_INV = 128;
constexpr int MAX_SLOTS = 2 * 33 + 16;  // polynomial orders <= 32 (plain + HF) and <= 16 special terms

// monotone part as a function of x_c for one sample; slot coefficients prepared once per sample
struct MonEval {
    const PlanView* P;
    const InvArgs* a;
    const double* xis;
    const double* ws;
    double C[MAX_SLOTS];

    __device__ void prepare(const double* __restrict__ bcoef, const double* Xt, int64_t ld, int64_t i) {
        const PlanView& p = *P;
        const int ns = 2 * (p.maxord + 1) + p.nst;
        for (int s = 0; s < ns; ++s) {
            const int j0 = __ldg(p.ib + p.o_slot_ptr + s), j1 = __ldg(p.ib + p.o_slot_ptr + s + 1);
            double acc = 0.0;
            for (int jj = j0; jj < j1; ++jj) {
                const int j = __ldg(p.ib + p.o_slot_term + jj);
                const int b = __ldg(p.ib + p.o_out_ptr + j), e = __ldg(p.ib + p.o_out_ptr + j + 1);
                double u = 1.0;
                for (int q = b; q < e; ++q) u *= plan_factor(p, __ldg(p.ib + p.o_out_fac + q), Xt, ld, i);
                acc = fma(bcoef[j], u, acc);
            }
            C[s] = acc * __ldg(p.db + p.o_d_slot_scale + s);
        }
    }

    // r(t) = sum_s C_s phi_s(t)
    __device__ double lin(double t) const {
        const PlanView& p = *P;
        const double ga = p.has_hf ? exp(-0.25 * t * t) : 1.0;
        double A, B, Cc;
        rec_coef(p.family, 0, A, B, Cc);
        double pm = 1.0, pc = fma(A, t, B);
        double r = C[0];
        for (int o = 1; o <= p.maxord; ++o) {
            r = fma(pc, fma(ga, C[2 * o + 1], C[2 * o]), r);
            rec_coef(p.family, o, A, B, Cc);
            const double pn = fma(fma(A, t, B), pc, -Cc * pm);
            pm = pc;
            pc = pn;
        }
        const int sb = 2 * (p.maxord + 1);
        for (int q = 0; q < p.nst; ++q) {
            const int f = __ldg(p.ib + p.o_st_fac + q);
            const int4 fi = __ldg(reinterpret_cast<const int4*>(p.ib + p.o_fac_i) + f);
            const double4 fd = ldg_d4(reinterpret_cast<const double4*>(p.db + p.o_d_fac) + f);
            r = fma(C[sb + q], eval_factor(fi.y, fi.z, fd.x, fd.y, fd.z, fd.w, p.family, t), r);
        }
        return r;
    }

    // monotone part M(x): separable -> r(x); integrated rectifier -> Gauss-Legendre of g(r(t)) + delta on [0, x]
    __device__ double mon(double x) const {
        if (a->separable) return lin(x);
        const double hx = 0.5 * x;
        double acc = 0.0;
        for (int q = 0; q < a->Q; ++q) acc = fma(ws[q], rect_eval(a->rect, lin(fma(hx, xis[q], hx))), acc);
        return hx * fma(a->delta, a->wsum, acc);
    }
};

// Prologue shared by K-inv-table and K-inv-bisect, which both handle the samples [a.first, a.first + a.count), grid
// striding over groups of R_OBJ rows of T_INV samples.  Dynamic shared memory holds the coefficients, the kernel's own
// arrays, then the dense-group tables DS (each kernel stages them itself: with the staging in a helper, ptxas spills
// more in K-inv-bisect).  Here: the thread's R_OBJ samples of row group row0 (rows past the range read sample a.first
// and are not ok) and their nonmonotone offsets (:4039-4043).
__device__ __forceinline__ void inv_offsets(const InvArgs& a, const DenseSmem& DS, int64_t row0, int64_t (&idx)[R_OBJ],
                                            bool (&ok)[R_OBJ], double (&S)[R_OBJ]) {
    const int64_t rows = (a.count + T_INV - 1) / T_INV;
#pragma unroll
    for (int r = 0; r < R_OBJ; ++r) {
        const int64_t i = a.first + (row0 + r) * T_INV + threadIdx.x;
        ok[r] = (row0 + r < rows) && (i < a.first + a.count);
        idx[r] = ok[r] ? i : a.first;
        S[r] = 0.0;
    }
    dense_value_smem_rt<R_OBJ>(a.P, DS, a.Xt, a.ld, a.first + row0 * T_INV + threadIdx.x, T_INV, ok, S);
    nonmon_slow_rt<false>(a.P, a.Xt, a.ld, idx, ttm_dyn_smem, S, nullptr, 0);
}

__global__ void __launch_bounds__(T_INV) inverse_table_kernel(const InvArgs a) {
    const PlanView& P = a.P;
    const int m = P.m_non + P.m_mon;
    double* s_table = ttm_dyn_smem + m;  // [sorted values | abscissae]
    for (int j = threadIdx.x; j < m; j += T_INV) ttm_dyn_smem[j] = a.coeffs[j];
    for (int j = threadIdx.x; j < 2 * a.ntab; j += T_INV) s_table[j] = a.table[j];
    const DenseSmem DS = stage_dense_tables(P, a.coeffs, m + 2 * a.ntab, threadIdx.x, T_INV);
    __syncthreads();
    const int64_t rows = (a.count + T_INV - 1) / T_INV;
    double* xc_col = a.Xt + (int64_t)P.c * a.ld;
    for (int64_t row0 = (int64_t)blockIdx.x * R_OBJ; row0 < rows; row0 += (int64_t)gridDim.x * R_OBJ) {
        int64_t idx[R_OBJ];
        bool ok[R_OBJ];
        double S[R_OBJ];
        inv_offsets(a, DS, row0, idx, ok, S);
#pragma unroll
        for (int r = 0; r < R_OBJ; ++r)
            if (ok[r])   // target = -offset + Zk (:4071)
                xc_col[idx[r]] = interp_sorted_table(s_table, a.ntab, a.truncate, __dadd_rn(-S[r], a.z[idx[r]]));
    }
}

__global__ void __launch_bounds__(T_INV) inverse_bisect_kernel(const InvArgs a) {
    const PlanView& P = a.P;
    const int m = P.m_non + P.m_mon;
    double* s_xis = ttm_dyn_smem + m;
    double* s_ws = s_xis + a.Q;
    for (int j = threadIdx.x; j < m; j += T_INV) ttm_dyn_smem[j] = a.coeffs[j];
    for (int q = threadIdx.x; q < a.Q; q += T_INV) {
        s_xis[q] = a.xis[q];
        s_ws[q] = a.ws[q];
    }
    const DenseSmem DS = stage_dense_tables(P, a.coeffs, m + 2 * a.Q, threadIdx.x, T_INV);
    __syncthreads();
    const int64_t rows = (a.count + T_INV - 1) / T_INV;
    double* xc_col = a.Xt + (int64_t)P.c * a.ld;
    int limit = a.max_iter;
    if (a.first == 0 && a.count == 1 && a.iter_max) limit = min(limit, *a.iter_max);  // sample-0 quirk (:3952)
    int it_used_max = 0, n_stalled = 0;
    for (int64_t row0 = (int64_t)blockIdx.x * R_OBJ; row0 < rows; row0 += (int64_t)gridDim.x * R_OBJ) {
        int64_t idx[R_OBJ];
        bool ok[R_OBJ];
        double S[R_OBJ];
        inv_offsets(a, DS, row0, idx, ok, S);
#pragma unroll 1
        for (int r = 0; r < R_OBJ; ++r) {
            if (!ok[r]) continue;
            const int64_t i = idx[r];
            if (isnan(xc_col[i])) continue;                                  // marked for removal (:3846)
            MonEval ev;
            ev.P = &P; ev.a = &a; ev.xis = s_xis; ev.ws = s_ws;
            ev.prepare(ttm_dyn_smem + P.m_non, a.Xt, a.ld, i);
            const double off = S[r], z = a.z[i];
            auto resid = [&](double x) { return (off + ev.mon(x)) - z; };
            double lo = -2.0, hi = 2.0;                                      // start_distance (:3850-3864)
            double flo = resid(lo), fhi = resid(hi);
            double xlast = hi;
            if (flo > fhi) { double t = lo; lo = hi; hi = t; t = flo; flo = fhi; fhi = t; }
            while (flo * fhi > 0.0) {                                        // window shifting (:3894-3941)
                if (flo > fhi) { double t = lo; lo = hi; hi = t; t = flo; flo = fhi; fhi = t; }
                const double diff = hi - lo;
                if (flo > 0.0) { hi = lo; lo -= diff * 2.0; fhi = flo; flo = resid(lo); xlast = lo; }
                else if (flo < 0.0) { lo = hi; hi += diff * 2.0; flo = fhi; fhi = resid(hi); xlast = hi; }
                else break;
            }
            int it = 0;
            bool conv = false;
            while (it < limit) {                                             // bisection (:3952-3976)
                ++it;
                const double mid = (lo + hi) * 0.5;
                const double f = resid(mid);
                xlast = mid;
                if (f < 0.0) lo = mid;
                if (f > 0.0) hi = mid;
                if (!(fabs(f) > 1e-9)) { conv = true; break; }
            }
            xc_col[i] = xlast;
            it_used_max = max(it_used_max, it);
            if (!conv && it >= a.max_iter) ++n_stalled;
        }
    }
    if (a.iter_max && a.first > 0 && it_used_max > 0) atomicMax(a.iter_max, it_used_max);
    if (a.not_converged && n_stalled) atomicAdd(a.not_converged, n_stalled);
}

// table[q] = sum_j b_j psi^mon_j(fakeX_q), fakeX = 0 except column c = pts[q]   (:4047-4058)
__global__ void mon_table_kernel(const PlanView P, const double* __restrict__ coeffs, int ntab,
                                 const double* __restrict__ pts, double* __restrict__ table) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= ntab) return;
    const double x = pts[q];
    double acc = 0.0;
    for (int j = 0; j < P.m_mon; ++j) {
        const int b = __ldg(P.ib + P.o_mon_ptr + j), e = __ldg(P.ib + P.o_mon_ptr + j + 1);
        double v = 1.0;
        for (int f = b; f < e; ++f) {
            const int fidx = __ldg(P.ib + P.o_mon_fac + f);
            const int4 fi = __ldg(reinterpret_cast<const int4*>(P.ib + P.o_fac_i) + fidx);
            const double4 fd = ldg_d4(reinterpret_cast<const double4*>(P.db + P.o_d_fac) + fidx);
            const double fv = eval_factor(fi.y, fi.z, fd.x, fd.y, fd.z, fd.w, P.family, fi.x == P.c ? x : 0.0);
            v = (f == b) ? fv : v * fv;
        }
        acc = fma(coeffs[P.m_non + j], v, acc);
    }
    table[q] = acc;
}

// K-logdet-IR: l = log d_c S_k = log(g(r(x_c)) + delta) per sample, r(t) = sum_j b_j psi^mon_j(x_<c, t) -- the
// quantity the objective's -log term uses (ttm_objgrad_impl.cuh) -- accumulated into the log density:
//   mode 0 (pullback):    acc += -S^2/2 - log(2 pi)/2 + l - log sigma
//   mode 1 (pushforward): acc -= l - log sigma
// exponential with delta = 0 gives l = r exactly (rect_log); every other case log(g + delta), the integrand of the
// quadrature in K-S.  One thread per sample, no atomics: the result does not depend on the launch shape.
__global__ void __launch_bounds__(T_INV) ir_logdet_kernel(const PlanView P, const double* __restrict__ coeffs,
                                                          const double* __restrict__ Xt, int64_t ld, int64_t N,
                                                          const double* __restrict__ S, double log_sigma, int rect,
                                                          double delta, int mode, double* __restrict__ acc) {
    extern __shared__ double s_b[];
    for (int j = threadIdx.x; j < P.m_mon; j += T_INV) s_b[j] = coeffs[P.m_non + j];
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * T_INV + threadIdx.x;
    if (i >= N) return;
    MonEval ev;
    ev.P = &P; ev.a = nullptr; ev.xis = nullptr; ev.ws = nullptr;
    ev.prepare(s_b, Xt, ld, i);
    const double r = ev.lin(Xt[(int64_t)P.c * ld + i]);
    const double l = (rect == RECT_EXP && delta == 0.0) ? r : log(rect_eval(rect, r) + delta);
    const double t = l - log_sigma;
    if (mode == 0) acc[i] += -0.5 * S[i] * S[i] - 0.91893853320467274178 + t;
    else acc[i] -= t;
}

}  // namespace

// K-inv-table / K-inv-bisect: at most 16 blocks per SM, each striding over groups of R_OBJ rows of T_INV samples;
// shared memory: coefficients, the kernel's `own` doubles, dense-group tables
static cudaError_t inv_launch(void (*kernel)(InvArgs), const InvArgs& a, int own, int sm_count, cudaStream_t st) {
    if (a.count == 0) return cudaSuccess;
    const int64_t rows = (a.count + T_INV - 1) / T_INV;
    int64_t grid = (rows + R_OBJ - 1) / R_OBJ;
    if (grid > (int64_t)sm_count * 16) grid = (int64_t)sm_count * 16;
    const size_t smem = sizeof(double) * (size_t)(a.P.m_non + a.P.m_mon + own + dense_smem_doubles(a.P.ndense, a.P.dense_maxord));
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    kernel<<<(unsigned)grid, T_INV, smem, st>>>(a);
    return cudaGetLastError();
}

cudaError_t ttm_launch_inverse_table(const InvArgs& a, int sm_count, cudaStream_t st) {
    return inv_launch(inverse_table_kernel, a, 2 * a.ntab, sm_count, st);
}

cudaError_t ttm_launch_inverse_bisect(const InvArgs& a, int sm_count, cudaStream_t st) {
    if (a.count > 0 && 2 * (a.P.maxord + 1) + a.P.nst > MAX_SLOTS) return cudaErrorInvalidValue;
    return inv_launch(inverse_bisect_kernel, a, 2 * a.Q, sm_count, st);
}

cudaError_t ttm_launch_mon_table(const PlanView& P, const double* coeffs, int ntab, double* table, cudaStream_t st) {
    // `table` holds the abscissae in table[ntab .. 2*ntab) on entry; values are written to table[0 .. ntab)
    mon_table_kernel<<<(ntab + 127) / 128, 128, 0, st>>>(P, coeffs, ntab, table + ntab, table);
    return cudaGetLastError();
}

cudaError_t ttm_launch_ir_logdet(const PlanView& P, const double* coeffs, const double* Xt, int64_t ld, int64_t N,
                                 const double* S, double sigma, int rect, double delta, int mode, double* acc,
                                 cudaStream_t st) {
    if (N == 0) return cudaSuccess;
    if (2 * (P.maxord + 1) + P.nst > MAX_SLOTS) return cudaErrorInvalidValue;
    const size_t smem = sizeof(double) * (size_t)(P.m_mon > 0 ? P.m_mon : 1);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(ir_logdet_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    ir_logdet_kernel<<<(unsigned)((N + T_INV - 1) / T_INV), T_INV, smem, st>>>(P, coeffs, Xt, ld, N, S, log(sigma),
                                                                              rect, delta, mode, acc);
    return cudaGetLastError();
}
