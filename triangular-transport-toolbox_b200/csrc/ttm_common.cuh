// Shared device-side definitions for libttm (sm_100a, FP64).
//
// A map component k (reference: generated fun_mon_k / fun_nonmon_k / der_fun_mon_k,
// transport_map.py:1263-2134) is compiled on the host into a *term table*:
//   factor  = univariate function of one sample column  (polynomial family member, optional
//             Hermite-function Gaussian weight, or one of the RBF-type special terms)
//   term    = product of factors (CSR lists)
// The tables live in two device blobs (int32 + double); `PlanView` is the parsed view.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#define TTM_PLAN_MAGIC 0x54544d31  // "TTM1"

// ---- factor kinds (reference: write_basis_function, transport_map.py:823-1261) ----
enum {
    F_POLY = 0,       // scale * P_n(x)
    F_POLY_HF = 1,    // scale * P_n(x) * exp(-x^2/4)                      (:1148-1150)
    F_RBF = 2,        // exp(-((x-mu)/s)^2/2)/(s*sqrt(2pi))                 (:976)
    F_IRBF = 3,       // (1+erf((x-mu)/(sqrt2 s)))/2                        (:1002)
    F_LET = 4,        // ((x-mu)(1-erf(u)) - s*sqrt(2/pi)exp(-u^2))/2       (:924)
    F_RET = 5,        // ((x-mu)(1+erf(u)) + s*sqrt(2/pi)exp(-u^2))/2       (:950)
    F_DPOLY = 6,      // scale * P_n'(x)                                    (:1178-1206)
    F_DPOLY_HF = 7,   // -1/2 exp(-x^2/4) (x*scale*P_n - 2*scale2*P_n')     (:1245)
    F_DRBF = 8,       // (:985)
    F_DIRBF = 9,      // (:1012)
    F_DLET = 10,      // (:933)
    F_DRET = 11,      // (:959)
    F_ZERO = 12,      // identically zero (derivative of a term without x_c, :1255-1258)
    F_ONE = 13        // constant 1 (reference: np.ones, :890)
};

// ---- polynomial families (reference: transport_map.py:271-304) ----
enum { FAM_POWER = 0, FAM_HERMITE = 1, FAM_HERMITE_E = 2, FAM_CHEBYSHEV = 3, FAM_LAGUERRE = 4, FAM_LEGENDRE = 5 };

// ---- rectifiers (reference: class rectifier, transport_map.py:4956-5213) ----
enum { RECT_EXP = 0, RECT_SOFTPLUS = 1, RECT_SQUARED = 2, RECT_EXPNEG = 3, RECT_ELU = 4 };

// ---- int blob header (offsets are in int32 elements from the blob start) ----
enum {
    H_MAGIC = 0, H_DTOT, H_C, H_FAMILY, H_NFAC, H_FAC_I,
    H_M_NON, H_NON_PTR, H_NON_FAC,
    H_M_MON, H_MON_PTR, H_MON_FAC,
    H_M_DMON, H_DMON_PTR, H_DMON_FAC,
    // integrated-rectifier objective plan
    H_NCONST, H_CONST_IDX,
    H_NVARS, H_VAR_IDX, H_VAR_PTR, H_ENT_I,
    H_NMULTI, H_MULTI_IDX,
    H_MAXORD, H_HAS_PLAIN, H_HAS_HF, H_NST, H_NSLOT,
    H_SLOT_PTR, H_SLOT_TERM, H_OUT_PTR, H_OUT_FAC, H_ST_FAC,
    // double blob offsets (in doubles)
    H_D_FAC, H_D_ENT, H_D_SLOT_SCALE, H_D_REC,
    H_NON_MAXVAR,   // 1 + largest column index touched by the nonmonotone terms
    // dense nonmonotone groups: per variable, polynomial coefficients addressed by slot 2*order+hf
    H_NDENSE, H_DENSE_VAR, H_DENSE_IDX, H_DENSE_MAXORD, H_D_DENSE_SCALE,
    H_NACTIVE,      // number of non-empty monotone slots
    H_NOUTFAC,      // total number of outer-factor entries of the monotone terms
    H_SIZE = 48
};

struct PlanView {
    const int32_t* ib;   // device int blob
    const double* db;    // device double blob
    int dtot, c, family, nfac;
    int m_non, m_mon, m_dmon;
    int nconst, nvars, nmulti;
    int ndense, dense_maxord, nactive, n_outfac;
    int maxord, has_plain, has_hf, nst, nslot;
    // offsets
    int o_fac_i, o_non_ptr, o_non_fac, o_mon_ptr, o_mon_fac, o_dmon_ptr, o_dmon_fac;
    int o_const_idx, o_var_idx, o_var_ptr, o_ent_i, o_multi_idx;
    int o_slot_ptr, o_slot_term, o_out_ptr, o_out_fac, o_st_fac;
    int o_d_fac, o_d_ent, o_d_slot_scale, o_d_rec;
    int o_dense_var, o_dense_idx, o_d_dense_scale;
};

// ---------------------------------------------------------------------------------------
// Orthogonal-polynomial three-term recurrences (numpy.polynomial conventions).
//   P_{n+1} = (A_n x + B_n) P_n - C_n P_{n-1},   P_0 = 1,  P_1 = A_0 x + B_0
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void rec_coef(int family, int n, double& A, double& B, double& C) {
    switch (family) {
        case FAM_POWER:     A = 1.0; B = 0.0; C = 0.0; break;
        case FAM_HERMITE:   A = 2.0; B = 0.0; C = 2.0 * n; break;
        case FAM_HERMITE_E: A = 1.0; B = 0.0; C = (double)n; break;
        case FAM_CHEBYSHEV: A = (n == 0) ? 1.0 : 2.0; B = 0.0; C = 1.0; break;
        case FAM_LAGUERRE:  A = -1.0 / (n + 1); B = (2.0 * n + 1.0) / (n + 1); C = (double)n / (n + 1); break;
        default:            A = (2.0 * n + 1.0) / (n + 1); B = 0.0; C = (double)n / (n + 1); break;  // Legendre
    }
}

// value (and derivative) of P_order(x) for the given family
template <bool DERIV>
__device__ __forceinline__ void poly_eval(int family, int order, double x, double& p, double& dp) {
    double pm = 0.0, pc = 1.0, dm = 0.0, dc = 0.0;
    for (int n = 0; n < order; ++n) {
        double A, B, C;
        rec_coef(family, n, A, B, C);
        const double lin = fma(A, x, B);
        const double pn = fma(lin, pc, -C * pm);
        if (DERIV) {
            const double dn = fma(A, pc, fma(lin, dc, -C * dm));
            dm = dc; dc = dn;
        }
        pm = pc; pc = pn;
    }
    p = pc;
    dp = dc;
}


// 32-byte read-only load (two 16-byte LDG)
__device__ __forceinline__ double4 ldg_d4(const double4* p) {
    const double2 a = __ldg(reinterpret_cast<const double2*>(p));
    const double2 b = __ldg(reinterpret_cast<const double2*>(p) + 1);
    return make_double4(a.x, a.y, b.x, b.y);
}

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// Table root finder of vectorized_root_search_alternate (transport_map.py:4047-4076) for one target t: tab =
// [sorted values | abscissae in the same order], ntab entries each.  truncate clamps t to the values' range (:4074-4076),
// then numpy.searchsorted(side='left'), clip(1, ntab - 1) and scipy's interp1d._call_linear formula, every operation
// correctly rounded as numpy does it.  Callers pass their shared-memory copy of the table.
__device__ __forceinline__ double interp_sorted_table(const double* __restrict__ tab, int ntab, int truncate,
                                                      double t) {
    if (truncate) {
        const double tmin = tab[0], tmax = tab[ntab - 1];
        if (t < tmin) t = tmin;
        if (t > tmax) t = tmax;
    }
    int lo = 0, hi = ntab;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (tab[mid] < t) lo = mid + 1; else hi = mid;
    }
    const int k = lo < 1 ? 1 : (lo > ntab - 1 ? ntab - 1 : lo);
    const double xl = tab[k - 1], xh = tab[k], yl = tab[ntab + k - 1], yh = tab[ntab + k];
    const double den = __dsub_rn(xh, xl);
    return __dadd_rn(__dmul_rn(__ddiv_rn(__dsub_rn(t, xl), den), yh), __dmul_rn(__ddiv_rn(__dsub_rn(xh, t), den), yl));
}

// FP64 tensor-core MMA C += A B (A 8x4, B 4x8, C 8x8): each lane holds one element of A and of B and two of C
__device__ __forceinline__ void dmma_m8n8k4(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

#define TTM_INV_SQRT2 0.70710678118654752440
#define TTM_SQRT_2PI 2.50662827463100050242
#define TTM_SQRT_2_OVER_PI 0.79788456080286535588

// One factor value. fi = {var, kind, order, -}, fd = {scale, scale2, mu, sigma}
// (deliberately not inlined: it is a large switch with erf/exp bodies and is only used off the hot loops)
static __device__ __noinline__ double eval_factor(int kind, int order, double scale, double scale2, double mu,
                                           double sg, int family, double x) {
    double p, dp;
    switch (kind) {
        case F_POLY:
            poly_eval<false>(family, order, x, p, dp);
            return scale * p;
        case F_POLY_HF:
            poly_eval<false>(family, order, x, p, dp);
            return scale * p * exp(-0.25 * x * x);
        case F_DPOLY:
            poly_eval<true>(family, order, x, p, dp);
            return scale * dp;
        case F_DPOLY_HF:
            poly_eval<true>(family, order, x, p, dp);
            return -0.5 * exp(-0.25 * x * x) * (x * (scale * p) - 2.0 * (scale2 * dp));
        case F_RBF: {
            const double z = (x - mu) / sg;
            return exp(-0.5 * z * z) / (sg * TTM_SQRT_2PI);
        }
        case F_IRBF:
            return 0.5 * (1.0 + erf((x - mu) / sg * TTM_INV_SQRT2));
        case F_LET: {
            const double u = (x - mu) / sg * TTM_INV_SQRT2;
            return 0.5 * ((x - mu) * (1.0 - erf(u)) - sg * TTM_SQRT_2_OVER_PI * exp(-u * u));
        }
        case F_RET: {
            const double u = (x - mu) / sg * TTM_INV_SQRT2;
            return 0.5 * ((x - mu) * (1.0 + erf(u)) + sg * TTM_SQRT_2_OVER_PI * exp(-u * u));
        }
        case F_DRBF: {
            const double z = (x - mu) / sg;
            return -(x - mu) / (TTM_SQRT_2PI * sg * sg * sg) * exp(-0.5 * z * z);
        }
        case F_DIRBF: {
            const double z = (x - mu) / sg;
            return exp(-0.5 * z * z) / (TTM_SQRT_2PI * sg);
        }
        case F_DLET:
            return 0.5 * (1.0 - erf((x - mu) / sg * TTM_INV_SQRT2));
        case F_DRET:
            return 0.5 * (1.0 + erf((x - mu) / sg * TTM_INV_SQRT2));
        case F_ONE:
            return 1.0;
        default:
            return 0.0;
    }
}

// factor `f` of the plan evaluated on sample i (columns of the transposed sample matrix Xt)
__device__ __forceinline__ double plan_factor(const PlanView& P, int f, const double* __restrict__ Xt, int64_t ld,
                                              int64_t i) {
    const int4 fi = __ldg(reinterpret_cast<const int4*>(P.ib + P.o_fac_i) + f);
    const double4 fd = ldg_d4(reinterpret_cast<const double4*>(P.db + P.o_d_fac) + f);
    const double x = (fi.y == F_ONE || fi.y == F_ZERO) ? 0.0 : Xt[(int64_t)fi.x * ld + i];
    return eval_factor(fi.y, fi.z, fd.x, fd.y, fd.z, fd.w, P.family, x);
}

// same, but column `ovr_col` is replaced by the value `ovr_x` (root finding / quadrature probes)
__device__ __forceinline__ double plan_factor_ovr(const PlanView& P, int f, const double* __restrict__ Xt,
                                                  int64_t ld, int64_t i, int ovr_col, double ovr_x) {
    const int4 fi = __ldg(reinterpret_cast<const int4*>(P.ib + P.o_fac_i) + f);
    const double4 fd = ldg_d4(reinterpret_cast<const double4*>(P.db + P.o_d_fac) + f);
    double x = 0.0;
    if (fi.y != F_ONE && fi.y != F_ZERO) x = (fi.x == ovr_col) ? ovr_x : Xt[(int64_t)fi.x * ld + i];
    return eval_factor(fi.y, fi.z, fd.x, fd.y, fd.z, fd.w, P.family, x);
}

// product term `j` of a CSR list
__device__ __forceinline__ double plan_term(const PlanView& P, int o_ptr, int o_fac, int j,
                                            const double* __restrict__ Xt, int64_t ld, int64_t i) {
    const int b = __ldg(P.ib + o_ptr + j), e = __ldg(P.ib + o_ptr + j + 1);
    double v = 1.0;
    for (int q = b; q < e; ++q) {
        const double f = plan_factor(P, __ldg(P.ib + o_fac + q), Xt, ld, i);
        v = (q == b) ? f : v * f;
    }
    return v;
}

__device__ __forceinline__ double plan_term_ovr(const PlanView& P, int o_ptr, int o_fac, int j,
                                                const double* __restrict__ Xt, int64_t ld, int64_t i, int ovr_col,
                                                double ovr_x) {
    const int b = __ldg(P.ib + o_ptr + j), e = __ldg(P.ib + o_ptr + j + 1);
    double v = 1.0;
    for (int q = b; q < e; ++q) {
        const double f = plan_factor_ovr(P, __ldg(P.ib + o_fac + q), Xt, ld, i, ovr_col, ovr_x);
        v = (q == b) ? f : v * f;
    }
    return v;
}

// ---------------------------------------------------------------------------------------
// reductions
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---------------------------------------------------------------------------------------
// rectifier g, its coefficient-derivative factor and log(g + delta)  (transport_map.py:4981-5213)
// ---------------------------------------------------------------------------------------
#define TTM_LN2 0.69314718055994530942

__device__ __forceinline__ double rect_eval(int rect, double r) {
    switch (rect) {
        case RECT_EXP: return exp(r);
        case RECT_EXPNEG: return exp(-r);
        case RECT_SOFTPLUS: {
            const double ar = TTM_LN2 * r;
            return log(1.0 + exp(-fabs(ar))) + fmax(ar, 0.0);
        }
        case RECT_SQUARED: return r * r;
        default: return (r < 0.0) ? exp(r) : r + 1.0;
    }
}

// factor multiplying dfdc in rectifier.evaluate_dfdc (NB softplus omits ln2, transport_map.py:5152-5153)
__device__ __forceinline__ double rect_dfac(int rect, double r, double g) {
    switch (rect) {
        case RECT_EXP: return g;
        case RECT_EXPNEG: return -g;
        case RECT_SOFTPLUS: return 1.0 / (1.0 + exp(-TTM_LN2 * r));
        default: return 0.0;  // squared / explinearunit: the reference raises "Not implemented yet."
    }
}

__device__ __forceinline__ double rect_log(int rect, double r, double g, double delta) {
    switch (rect) {
        case RECT_EXP: return (delta == 0.0) ? r : log(g + delta);
        case RECT_EXPNEG: return -r;
        case RECT_SOFTPLUS: return log(g + delta);
        case RECT_SQUARED: return log(r * r);
        default: return log(g);
    }
}
