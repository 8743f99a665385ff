// exp(x) for the FP64-bound kernels (tile K-objgrad, fused inverse): branch-free, interleavable, and cheap on
// SHARED MEMORY as well as on the FP64 pipe.
//
//   exp(x) = 2^n * 2^(j/E) * e^r,   E x / ln 2 = E n + j + f,   r = x - (E n + j) ln2/E,  |r| <= ln2/(2E),   E = 64
//
//   * degree-4 weighted minimax polynomial of e^r on the reduced range (p(0) = 1, p'(0) = 1 imposed; Remez in 60-digit
//     arithmetic): maximum relative error 5.1e-15.  The path's tolerance is 1e-10 (objective / gradient against the
//     reference) and the error averages over samples and nodes: the measured parity of the C4 objective and gradient
//     against the oracle is 4.9e-15 with this polynomial, 4.8e-15 with the 1-ulp variants below;
//   * E-entry table of correctly rounded 2^(j/E), pre-scaled by 2^-1021 and split into low/high 32-bit words
//     (ttm_exp_tab64.h): a look-up is two 32-bit LDS, entries j and j + 32 share a bank (<= 2 wavefronts).  ncu showed
//     that a 64-bit table with more than 16 entries costs ~6 shared-memory wavefronts per look-up (random 8-byte words,
//     2.9-way conflicts per half warp), which made a 1024-entry/degree-3 variant shared-memory bound;
//   * ONE fused reduction step: r carries the representation error of ln2/E, i.e. the result is exp of an argument
//     perturbed by a relative <= 2^-53 (an error of |x| 1.1e-16 in the result; the arguments here are O(10));
//   * the rounding constant carries the offset 1021*E, so the low word of t is E (n + 1021) + j, non-negative in
//     range: one clamp (VIMNMX[.RELU]), one shift and one IMAD insert the binary exponent.
// 8 FP64 + 7 other instructions.  History of the polynomial (each step measured on the C4 bench, same parity):
// 32 entries + degree-6 Taylor (10 FP64, 3.5e-18 truncation: far below its own rounding) 2952 evals/s;
// 32 entries + degree-5 minimax (9 FP64, 1.09e-16; TTM_EXP_VARIANT=32) 3020; 64 entries + degree-4 minimax 3159.
// Domain: |x| < 2.3e7 (the rounded multiple must fit 31 bits); results saturate at 2^-1021 / 2^1023 instead of
// underflowing / overflowing (the objective is inf or the integrand below 4.5e-308 long before); NaN in -> NaN out.
#pragma once

#include <cuda_runtime.h>

#ifndef TTM_EXP_VARIANT
#define TTM_EXP_VARIANT 64
#endif
#if TTM_EXP_VARIANT == 64
#include "ttm_exp_tab64.h"
#else
#include "ttm_exp_tab32.h"
#endif

namespace ttm_exp32 {

#if TTM_EXP_VARIANT == 64
// 64-entry table, |r| <= ln2/128, degree-4 minimax (5.1e-15 relative): 8 FP64 per exp
#define TTM_E32_K 92.33248261689366
#define TTM_E32_C 0.010830424696249145
#define TTM_E32_OFF 65344                                   /* 1021 * 64 */
#define TTM_E32_MAGIC (6755399441055744.0 + 65344.0)
#define TTM_E32_TOP (2044 * 64 + 63)
#define TTM_E32_SHIFT 6
#define TTM_E32_MASK 63
#define TTM_E32_DEG 4
#define TTM_E32_Q0 0.5000000000031141430417529
#define TTM_E32_Q1 0.1666668790482994370921845
#define TTM_E32_Q2 0.04166656921007259929347011
constexpr int TAB_ENTRIES = 64;
#define TTM_E32_TAB_LO g_ttm_exp2_tab64_lo
#define TTM_E32_TAB_HI g_ttm_exp2_tab64_hi
#else
// 32-entry table, |r| <= ln2/64, degree-5 minimax (1.09e-16 relative): 9 FP64 per exp
#define TTM_E32_K 46.16624130844683
#define TTM_E32_C 0.02166084939249829
#define TTM_E32_OFF 32672                                   /* 1021 * 32 */
#define TTM_E32_MAGIC (6755399441055744.0 + 32672.0)
#define TTM_E32_TOP (2044 * 32 + 31)
#define TTM_E32_SHIFT 5
#define TTM_E32_MASK 31
#define TTM_E32_DEG 5
// e^r = 1 + r + r^2 (Q0 + Q1 r + Q2 r^2 + Q3 r^3) on |r| <= ln2/64: weighted minimax (Remez in 60-digit arithmetic,
// p(0) = 1 and p'(0) = 1 imposed), maximum relative error 1.09e-16
#define TTM_E32_Q0 0.4999999999904452171653481
#define TTM_E32_Q1 0.1666666666653016986433126
#define TTM_E32_Q2 0.04166691103830363355853435
#define TTM_E32_Q3 0.008333368243548227860252323
constexpr int TAB_ENTRIES = 32;
#define TTM_E32_TAB_LO g_ttm_exp2_tab32_lo
#define TTM_E32_TAB_HI g_ttm_exp2_tab32_hi
#endif
constexpr int TAB_DOUBLES = TAB_ENTRIES;                    // shared-memory footprint: 2 * TAB_ENTRIES words

// shared-memory copy of the table: [0..E) low words, [E..2E) high words
__device__ __forceinline__ void stage_table(unsigned int* s_tab, int tid, int nthreads) {
    for (int j = tid; j < 2 * TAB_ENTRIES; j += nthreads)
        s_tab[j] = (j < TAB_ENTRIES) ? TTM_E32_TAB_LO[j] : TTM_E32_TAB_HI[j - TAB_ENTRIES];
}

// ---------------------------------------------------------------------------------------------------------------------
// exp of a product, exp(a b), for the tile kernel's hot loops, given bK = b * K (K = E / ln2) instead of a b:
//
//   t = fma(a, bK, MAGIC),  nf = t - MAGIC = E n + j,  u = fma(a, bK, -nf)   (|u| <= 1/2, one rounding)
//   exp(a b) ~ 2^(j/E) 2^n * P(u),   P(u) = 1 + u (C + u (C^2 Q0 + u (C^3 Q1 + u C^4 Q2)))  = p(C u), C = ln2/E
//
// i.e. the same polynomial in the unscaled variable u: 7 FP64 and the final DMUL against the scaled table word, where
// exp(y) of a formed product y = a b takes 1 + 8.  The argument carries one rounding of b K (and of K) instead of one
// rounding of a b and the representation error of C: exp of an argument perturbed by a relative <= 2^-52, the class of
// the fused reduction above.  Maximum relative error of the 64-entry form on |a b| <= 40: 9.8e-15 measured, bound
// 1.5e-14 (polynomial 5.1e-15 plus 40 * 2^-52 from the argument; tests/test_exp_product_form.py).
//
// Exponent insertion before the DMUL, in one IMAD: the "folded" high words hi'[j] = hi[j] - (j << 14) are staged
// behind the table, so that for c = E (n + 1021) + j (E = 64; 2^15 and j << 15 for E = 32)
//   hi(tb[j] 2^(n + 1021)) = hi[j] + (n + 1021) 2^20 = c 2^14 + hi'[j].
// Scaling the table word instead of the product is exact (every intermediate stays normal and finite: c is clamped to
// [0, TOP], or proven in range), so the result equals the scaled product bit for bit.  Without the clamp c is not
// bounded: CLAMP_NONE is only for arguments the caller has proven to lie in [-700, 700].
// ---------------------------------------------------------------------------------------------------------------------
constexpr int TAB_FOLDED_WORDS = 3 * TAB_ENTRIES;           // [0..E) low | [E..2E) high | [2E..3E) folded high words
constexpr int TAB_FOLD = 20 - TTM_E32_SHIFT;                // 14 for E = 64: c 2^14 = (n + 1021) 2^20 + j 2^14
constexpr double PK_C1 = TTM_E32_C;
constexpr double PK_C2 = TTM_E32_C * TTM_E32_C * TTM_E32_Q0;
constexpr double PK_C3 = TTM_E32_C * TTM_E32_C * TTM_E32_C * TTM_E32_Q1;
constexpr double PK_C4 = TTM_E32_C * TTM_E32_C * TTM_E32_C * TTM_E32_C * TTM_E32_Q2;
#if TTM_E32_DEG == 5
constexpr double PK_C5 = TTM_E32_C * TTM_E32_C * TTM_E32_C * TTM_E32_C * TTM_E32_C * TTM_E32_Q3;
#endif

enum { CLAMP_NONE = 0, CLAMP_NEG = 1, CLAMP_GEN = 2 };      // argument proven in range / <= 0 / any

// stage_table's layout followed by the folded high words (TAB_FOLDED_WORDS words)
__device__ __forceinline__ void stage_table_folded(unsigned int* s_tab, int tid, int nthreads) {
    for (int j = tid; j < TAB_FOLDED_WORDS; j += nthreads)
        s_tab[j] = (j < TAB_ENTRIES)       ? TTM_E32_TAB_LO[j]
                 : (j < 2 * TAB_ENTRIES)   ? TTM_E32_TAB_HI[j - TAB_ENTRIES]
                                           : TTM_E32_TAB_HI[j - 2 * TAB_ENTRIES] - ((unsigned)(j - 2 * TAB_ENTRIES) << TAB_FOLD);
}

template <int L, int CLAMP>
__device__ __forceinline__ void exp_prod_v(const double (&a)[L], const double (&bK)[L], double (&out)[L],
                                           const unsigned int* __restrict__ tab) {
    double t[L], u[L], p[L];
    int c[L];
#pragma unroll
    for (int l = 0; l < L; ++l) t[l] = fma(a[l], bK[l], TTM_E32_MAGIC);
#pragma unroll
    for (int l = 0; l < L; ++l) {
        const int m = __double2loint(t[l]);
        c[l] = (CLAMP == CLAMP_NEG) ? max(m, 0) : (CLAMP == CLAMP_GEN) ? __vimin_s32_relu(m, TTM_E32_TOP) : m;
        u[l] = fma(a[l], bK[l], -(t[l] - TTM_E32_MAGIC));
    }
#if TTM_E32_DEG == 5
#pragma unroll
    for (int l = 0; l < L; ++l) p[l] = fma(u[l], PK_C5, PK_C4);
#pragma unroll
    for (int l = 0; l < L; ++l) p[l] = fma(p[l], u[l], PK_C3);
#else
#pragma unroll
    for (int l = 0; l < L; ++l) p[l] = fma(u[l], PK_C4, PK_C3);
#endif
#pragma unroll
    for (int l = 0; l < L; ++l) p[l] = fma(p[l], u[l], PK_C2);
#pragma unroll
    for (int l = 0; l < L; ++l) p[l] = fma(p[l], u[l], PK_C1);
#pragma unroll
    for (int l = 0; l < L; ++l) p[l] = fma(p[l], u[l], 1.0);
#pragma unroll
    for (int l = 0; l < L; ++l) {
        const int j = c[l] & TTM_E32_MASK;
        const unsigned hi = (unsigned)c[l] * (1u << TAB_FOLD) + tab[2 * TAB_ENTRIES + j];
        out[l] = p[l] * __hiloint2double((int)hi, (int)tab[j]);
    }
}

// hi + (c >> SHIFT) * 2^20 as SHF + IMAD (the compiler's own strength reduction takes three instructions)
__device__ __forceinline__ int insert_exponent(int hi, int c) {
    int n, out;
    asm("shr.s32 %0, %1, %2;" : "=r"(n) : "r"(c), "n"(TTM_E32_SHIFT));
    asm("mad.lo.s32 %0, %1, 1048576, %2;" : "=r"(out) : "r"(n), "r"(hi));
    return out;
}

// p = 2^(j/32 - 1021) e^r, m = 32 (n + 1021) + j   (written over L independent arguments so that the dependent
// FP64 chains are interleaved at source level)
template <int L>
__device__ __forceinline__ void core_v(const double (&x)[L], double (&p)[L], int (&m)[L],
                                       const unsigned int* __restrict__ tab) {
    double t[L], nf[L], r[L], tb[L];
#pragma unroll
    for (int l = 0; l < L; ++l) t[l] = fma(x[l], TTM_E32_K, TTM_E32_MAGIC);
#pragma unroll
    for (int l = 0; l < L; ++l) {
        m[l] = __double2loint(t[l]);
        nf[l] = t[l] - TTM_E32_MAGIC;
    }
#pragma unroll
    for (int l = 0; l < L; ++l)
        tb[l] = __hiloint2double((int)tab[TAB_ENTRIES + (m[l] & TTM_E32_MASK)], (int)tab[m[l] & TTM_E32_MASK]);
#pragma unroll
    for (int l = 0; l < L; ++l) r[l] = fma(nf[l], -TTM_E32_C, x[l]);
#if TTM_E32_DEG == 5
#pragma unroll
    for (int l = 0; l < L; ++l) p[l] = fma(r[l], TTM_E32_Q3, TTM_E32_Q2);
#pragma unroll
    for (int l = 0; l < L; ++l) p[l] = fma(p[l], r[l], TTM_E32_Q1);
#else
#pragma unroll
    for (int l = 0; l < L; ++l) p[l] = fma(r[l], TTM_E32_Q2, TTM_E32_Q1);
#endif
#pragma unroll
    for (int l = 0; l < L; ++l) p[l] = fma(p[l], r[l], TTM_E32_Q0);
#pragma unroll
    for (int l = 0; l < L; ++l) p[l] = fma(p[l], r[l], 1.0);
#pragma unroll
    for (int l = 0; l < L; ++l) p[l] = fma(p[l], r[l], 1.0);
#pragma unroll
    for (int l = 0; l < L; ++l) p[l] *= tb[l];
}

// argument <= 0 (Gaussian weight e^{-x^2/4})
template <int L>
__device__ __forceinline__ void exp_neg_v(const double (&x)[L], double (&out)[L], const unsigned int* __restrict__ tab) {
    double p[L];
    int m[L];
    core_v<L>(x, p, m, tab);
#pragma unroll
    for (int l = 0; l < L; ++l)
        out[l] = __hiloint2double(insert_exponent(__double2hiint(p[l]), max(m[l], 0)), __double2loint(p[l]));
}

// general argument (rectifier)
template <int L>
__device__ __forceinline__ void exp_gen_v(const double (&x)[L], double (&out)[L], const unsigned int* __restrict__ tab) {
    double p[L];
    int m[L];
    core_v<L>(x, p, m, tab);
#pragma unroll
    for (int l = 0; l < L; ++l)
        out[l] = __hiloint2double(insert_exponent(__double2hiint(p[l]), __vimin_s32_relu(m[l], TTM_E32_TOP)),
                                  __double2loint(p[l]));
}

__device__ __forceinline__ double exp_neg_1(double x, const unsigned int* __restrict__ tab) {
    double a[1] = {x}, o[1];
    exp_neg_v<1>(a, o, tab);
    return o[0];
}
__device__ __forceinline__ double exp_gen_1(double x, const unsigned int* __restrict__ tab) {
    double a[1] = {x}, o[1];
    exp_gen_v<1>(a, o, tab);
    return o[0];
}

}  // namespace ttm_exp32
