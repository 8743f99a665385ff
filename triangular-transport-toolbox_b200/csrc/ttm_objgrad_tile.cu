// K-objgrad / K-S, tile form: the hot instantiation of the fused integrated-rectifier objective + gradient
// (order <= 3 Hermite-function map components with the exponential rectifier, i.e. BASELINE config C4).
//
// Replaces, in ONE launch (like ttm_objgrad_impl.cuh, which stays the general kernel):
//   objective_function            transport_map.py:3300-3433
//   objective_function_jacobian   transport_map.py:3435-3635
//   s (integrated-rectifier arm)  transport_map.py:2439-2547
//   GaussQuadrature vector branch transport_map.py:4202-4278
//   rectifier (exponential)       transport_map.py:4956-5213
//
// A block of 256 threads walks tiles of 256 samples.  Per tile:
//   phase 1  (thread <-> sample)   Gauss-Legendre node loop of the monotone part: M_i = int_0^{x_c} g(r(t)) dt and
//                                  the slot integrals int g' He_o(t) e^{-t^2/4} dt, NQ nodes in flight per thread.
//                                  r(t) is evaluated in Horner form in the NODE variable tau = 1 + xi_q (coefficients
//                                  rescaled per sample) and the integrals are accumulated as monomial moments in tau
//                                  with node-only weights w tau^i; the node constants are KERNEL PARAMETERS
//                                  (constant-bank operands indexed by the uniform loop counter), the exp table is
//                                  shared memory read without bank conflicts (ttm_exp.cuh): the loop touches
//                                  shared memory with 4 wavefronts per node and warp.  25 FP64 instructions per node;
//                                  warps whose exp arguments are proven in range skip the exps' clamps.
//   phase 2  (warp <-> columns)    ONE sweep over the columns x_<c: every warp owns the dense groups g = warp (mod 8)
//                                  and walks the tile's 8 rows of 32 samples for them: S_non partial sums per sample
//                                  (value) and, in the same pass, h_j = sum_i w_i psi_ij (gradient) accumulated
//                                  per lane in shared memory -- no shuffles, no second exp(-x^2/4) per (i, j).
//                                  Weights w_i = M_i in Gram mode (dJ/da = G a + h, G = Psi^T Psi / N precomputed
//                                  once per ensemble by K-gram); without G the value sweep is followed by a second,
//                                  gradient-only sweep with w_i = S_i.
//   phase 3  (thread <-> sample)   S_i = S_non + M_i, J, monotone gradient into per-thread registers.
// Block partials -> [grid][1+m] buffer -> the last block reduces in fixed block order (bit-reproducible).
//
// Bound: FP64 pipe.  Algorithmic bytes 8 N (c+1): every needed column is read exactly once per evaluation in
// Gram mode (ncu: dram__bytes_read = 1.00 x algorithmic, writes ~ 0).
#include <cuda_runtime.h>

#include "ttm_common.cuh"
#include "ttm_exp.cuh"
#include "ttm_kernels.h"

namespace ttm_tile {

using namespace ttm_exp32;

constexpr int TB = 256;          // threads per block = samples per tile
constexpr int NWARP = TB / 32;
constexpr int ROWS = TB / 32;    // rows of 32 samples per tile
constexpr int MAXMON = TTM_TILE_MAXMON;
constexpr int NPARK = 8;         // L, ratio, hx*I_1..3, base_1..3
constexpr int MAXQ = TTM_TILE_MAXQ;

// node constants {tau, tau^2 K, w, w tau, w tau^2, w tau^3}, tau = 1 + xi_q, K = E / ln2 (the factor of exp_prod_v),
// passed as a kernel parameter
struct NodeTab {
    double v[6 * MAXQ];
};

// outer (x_<c) product of monotone term j on sample i (generic evaluator; a handful of terms per component)
static __device__ __noinline__ double tile_outer_product(const PlanView& P, int j, const double* __restrict__ Xt,
                                                         int64_t ld, int64_t i) {
    const int b = __ldg(P.ib + P.o_out_ptr + j), e = __ldg(P.ib + P.o_out_ptr + j + 1);
    double v = 1.0;
    for (int q = b; q < e; ++q) v *= plan_factor(P, __ldg(P.ib + P.o_out_fac + q), Xt, ld, i);
    return v;
}

// ---------------------------------------------------------------------------------------------------------
// shared-memory layout (offsets in doubles), computed by the launcher and passed in ObjArgs::lay
// ---------------------------------------------------------------------------------------------------------
struct Layout {
    int o_tab, o_coef, o_prod, o_col, o_mon, o_M, o_park, o_u, o_Spart, o_hacc, o_red, o_out, total;
};
static_assert(sizeof(Layout) <= sizeof(((ObjArgs*)nullptr)->lay), "ObjArgs::lay too small");

inline Layout make_layout(int m, int ndense, int ns, int nout, bool grad) {
    Layout L;
    int o = 0;
    L.o_tab = o;   o += (ttm_exp32::TAB_FOLDED_WORDS + 1) / 2;   // exp table: low | high | folded high words
    L.o_coef = o;  o += (m + 2) & ~1;
    L.o_prod = o;  o += 8 * ndense;                   // coefficient * scale, slot 2*order+hf
    L.o_col = o;   o += (ndense + 2) / 2;             // ints
    L.o_mon = o;   o += 4 + MAXMON;                   // scale_1..3, Sconst | ints: order[MAXMON], outer index[MAXMON]
    L.o_M = o;     o += TB;
    L.o_park = o;  o += grad ? NPARK * TB : 0;
    L.o_u = o;     o += grad ? nout * TB : 0;
    L.o_Spart = o; o += NWARP * TB;
    L.o_hacc = o;  o += grad ? ndense * ns * 32 : 0;
    L.o_red = o;   o += grad ? NWARP * (2 + MAXMON) : 0;
    L.o_out = o;   o += grad ? ((m + 2) & ~1) : 0;
    L.total = o;
    return L;
}

__host__ __device__ constexpr int popc8(int v) {
    int n = 0;
    for (int b = 0; b < 8; ++b) n += (v >> b) & 1;
    return n;
}

template <int MASK>
struct Slots {
    __host__ __device__ static constexpr bool has(int o, int hf) { return (MASK >> (2 * o + hf)) & 1; }
    __host__ __device__ static constexpr int idx(int o, int hf) { return popc8(MASK & ((1 << (2 * o + hf)) - 1)); }
    static constexpr int NS = popc8(MASK);
    static constexpr bool ANY_HF = (MASK & 0xAA) != 0;
    static constexpr bool NEED_P2 = has(2, 0) || has(2, 1);
    static constexpr bool NEED_P3 = has(3, 0) || has(3, 1);
};

// ---------------------------------------------------------------------------------------------------------
// phase 2: sweep over the dense groups owned by this warp.  VAL: S_non partial sums -> s_Spart[warp][sample];
// GRD: per-lane gradient sums, weights from s_W[sample].  FULL: the whole tile lies below N (no predicates).
// ---------------------------------------------------------------------------------------------------------
template <int MASK, bool VAL, bool GRD, bool FULL>
__device__ __forceinline__ void sweep_tile(const double* __restrict__ Xt, int64_t ld, int64_t base, int64_t N,
                                           int ndense, const int* __restrict__ s_col,
                                           const double* __restrict__ s_prod, const double* __restrict__ s_W,
                                           double* __restrict__ s_Spart, double* __restrict__ s_hacc,
                                           const unsigned int* __restrict__ s_tab, int warp, int lane) {
    using SL = Slots<MASK>;
    const int64_t i0 = base + lane;
    int nv = ROWS, nvmax = ROWS;                                // rows of this lane / of lane 0 that hold a sample
    if (!FULL) {
        const int64_t left = (N - i0 + 31) / 32, left0 = (N - base + 31) / 32;
        nv = (int)(left < 0 ? 0 : (left > ROWS ? ROWS : left));
        nvmax = (int)(left0 < 0 ? 0 : (left0 > ROWS ? ROWS : left0));
    }
    double Sp[ROWS];
#pragma unroll
    for (int r = 0; r < ROWS; ++r) Sp[r] = 0.0;
    double xn[ROWS];
    int g = warp;
    if (g < ndense) {
        const double* p = Xt + (int64_t)s_col[g] * ld + i0;
#pragma unroll
        for (int r = 0; r < ROWS; ++r) xn[r] = (FULL || r < nv) ? __ldcs(p + 32 * r) : 0.0;
    }
#pragma unroll 1
    for (; g < ndense; g += NWARP) {
        double x[ROWS];
#pragma unroll
        for (int r = 0; r < ROWS; ++r) x[r] = xn[r];
        if (g + NWARP < ndense) {                               // next group of this warp in flight
            const double* p = Xt + (int64_t)s_col[g + NWARP] * ld + i0;
#pragma unroll
            for (int r = 0; r < ROWS; ++r) xn[r] = (FULL || r < nv) ? __ldcs(p + 32 * r) : 0.0;
        }
        const double* c = s_prod + 8 * g;
        double cf[8];
        if (VAL) {
            const double2 c1 = *reinterpret_cast<const double2*>(c + 2), c2 = *reinterpret_cast<const double2*>(c + 4),
                          c3 = *reinterpret_cast<const double2*>(c + 6);
            cf[2] = c1.x; cf[3] = c1.y; cf[4] = c2.x; cf[5] = c2.y; cf[6] = c3.x; cf[7] = c3.y;
        }
        double h[SL::NS > 0 ? SL::NS : 1];
#pragma unroll
        for (int s = 0; s < SL::NS; ++s) h[s] = 0.0;
        // two half-tiles of 4 rows: 4 independent exp chains each (a half without samples is skipped: partial tiles)
#pragma unroll
        for (int r0 = 0; r0 < ROWS; r0 += 4) {
            if (!FULL && r0 >= nvmax) break;
            double xx[4], ga[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) xx[r] = x[r0 + r] * x[r0 + r];
            if (SL::ANY_HF) {                                   // e^{-x^2/4} = exp_prod(x^2, -K/4): no -x^2/4 formed
                const double bK[4] = {-0.25 * TTM_E32_K, -0.25 * TTM_E32_K, -0.25 * TTM_E32_K, -0.25 * TTM_E32_K};
                exp_prod_v<4, CLAMP_NEG>(xx, bK, ga, s_tab);
            }
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const double xv = x[r0 + r];
                const double P2 = SL::NEED_P2 ? xx[r] - 1.0 : 0.0;
                const double P3 = SL::NEED_P3 ? xv * (xx[r] - 3.0) : 0.0;
                const double Pv[4] = {1.0, xv, P2, P3};
                if (VAL) {
                    double acc = Sp[r0 + r];
#pragma unroll
                    for (int o = 1; o <= 3; ++o)
                        if (SL::has(o, 0)) acc = fma(cf[2 * o], Pv[o], acc);
                    if (SL::ANY_HF) {
                        double uh = 0.0;
                        bool first = true;
#pragma unroll
                        for (int o = 1; o <= 3; ++o)
                            if (SL::has(o, 1)) {
                                uh = first ? cf[2 * o + 1] * Pv[o] : fma(cf[2 * o + 1], Pv[o], uh);
                                first = false;
                            }
                        acc = fma(ga[r], uh, acc);
                    }
                    Sp[r0 + r] = acc;
                }
                if (GRD) {
                    const double wr = s_W[32 * (r0 + r) + lane];
                    const double wg = SL::ANY_HF ? wr * ga[r] : 0.0;
#pragma unroll
                    for (int o = 1; o <= 3; ++o) {
                        if (SL::has(o, 0)) h[SL::idx(o, 0)] = fma(wr, Pv[o], h[SL::idx(o, 0)]);
                        if (SL::has(o, 1)) h[SL::idx(o, 1)] = fma(wg, Pv[o], h[SL::idx(o, 1)]);
                    }
                }
            }
        }
        if (GRD) {
            double* hp = s_hacc + (g * SL::NS) * 32 + lane;
#pragma unroll
            for (int s = 0; s < SL::NS; ++s) hp[32 * s] += h[s];
        }
    }
    if (VAL) {
#pragma unroll
        for (int r = 0; r < ROWS; ++r) s_Spart[warp * TB + 32 * r + lane] = Sp[r];
    }
}

// ---------------------------------------------------------------------------------------------------------
// phase 1: the Gauss-Legendre node loop of one sample, NQ nodes in flight.  e^{ya tau^2} = exp_prod(ya, tau^2 K) and
// g = exp_prod(ga, P_K(tau)) with the rectifier polynomial's coefficients EK pre-multiplied by K; Qp (a multiple of NQ)
// nodes, constants loaded through the uniform loop counter.  The loop stays rolled: fully unrolled for Q = 100 (every
// node constant at a fixed constant-bank address, 62 KB of code per instance) the C4 step measured 4.3 % slower, and
// unrolled by 20 nodes 9.4 % slower (profiles/objgrad_tile_r4.json).  FAST: the caller has proven both exp arguments
// to lie in [-700, 700] for every lane of the warp, so the exps skip their clamps (same bits in range).
// ---------------------------------------------------------------------------------------------------------
template <bool GRAD, int NQ, bool FAST>
__device__ __forceinline__ void node_loop(const double* __restrict__ ntv, int Qp, double ya, const double (&EK)[4],
                                          const unsigned int* __restrict__ s_tab, double& Sacc, double& m0, double& m1,
                                          double& m2, double& m3) {
#pragma unroll 1
    for (int q = 0; q < Qp; q += NQ) {
        double yk[NQ], yv[NQ], ga[NQ], r[NQ], g[NQ];
        const double* nd = ntv + 6 * q;                                  // constant bank, uniform index
#pragma unroll
        for (int l = 0; l < NQ; ++l) { yv[l] = ya; yk[l] = nd[6 * l + 1]; }
        exp_prod_v<NQ, FAST ? CLAMP_NONE : CLAMP_NEG>(yv, yk, ga, s_tab);
#pragma unroll
        for (int l = 0; l < NQ; ++l) {
            const double tau = nd[6 * l];
            r[l] = fma(fma(fma(EK[3], tau, EK[2]), tau, EK[1]), tau, EK[0]);
        }
        exp_prod_v<NQ, FAST ? CLAMP_NONE : CLAMP_GEN>(ga, r, g, s_tab);
#pragma unroll
        for (int l = 0; l < NQ; ++l) {
            Sacc = fma(nd[6 * l + 2], g[l], Sacc);
            if (GRAD) {
                const double gg = g[l] * ga[l];
                m0 = fma(nd[6 * l + 2], gg, m0);
                m1 = fma(nd[6 * l + 3], gg, m1);
                m2 = fma(nd[6 * l + 4], gg, m2);
                m3 = fma(nd[6 * l + 5], gg, m3);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------------------------------------
template <int MASK, bool GRAD, bool MERGED, int NQ>
__global__ void __launch_bounds__(TB, 2) objgrad_tile_kernel(const __grid_constant__ ObjArgs a,
                                                             const __grid_constant__ NodeTab nt) {
    extern __shared__ double smem[];
    using SL = Slots<MASK>;
    const PlanView& P = a.P;
    const int m = P.m_non + P.m_mon;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int Qp = (a.Q + NQ - 1) / NQ * NQ;
    const int ndense = P.ndense;
    const Layout& LY = *reinterpret_cast<const Layout*>(a.lay);
    unsigned int* s_tab = reinterpret_cast<unsigned int*>(smem + LY.o_tab);
    double* s_coef = smem + LY.o_coef;
    double* s_prod = smem + LY.o_prod;
    int* s_col = reinterpret_cast<int*>(smem + LY.o_col);
    double* s_mond = smem + LY.o_mon;                          // [0..2] slot scales of orders 1..3, [3] Sconst
    int* s_tord = reinterpret_cast<int*>(smem + LY.o_mon + 4);  // [MAXMON] order of term j's slot
    int* s_tout = s_tord + MAXMON;                              // [MAXMON] index among the terms with outer factors, or -1
    double* s_M = smem + LY.o_M;
    double* s_park = smem + LY.o_park;
    double* s_u = smem + LY.o_u;
    double* s_Spart = smem + LY.o_Spart;
    double* s_hacc = smem + LY.o_hacc;
    double* s_red = smem + LY.o_red;
    double* s_outv = smem + LY.o_out;

    // ---- stage tables
    stage_table_folded(s_tab, tid, TB);
    for (int j = tid; j < m; j += TB) s_coef[j] = a.coeffs[j];
    const int dstride = 2 * (P.dense_maxord + 1);
    for (int e = tid; e < 8 * ndense; e += TB) {
        const int g = e >> 3, s = e & 7;
        int j = -1;
        double sc = 0.0;
        if (s < dstride) {
            j = P.ib[P.o_dense_idx + g * dstride + s];
            sc = P.db[P.o_d_dense_scale + g * dstride + s];
        }
        s_prod[e] = (j >= 0) ? a.coeffs[j] * sc : 0.0;
    }
    for (int g = tid; g < ndense; g += TB) s_col[g] = P.ib[P.o_dense_var + 4 * g];
    if (tid < MAXMON) { s_tord[tid] = 0; s_tout[tid] = -1; }
    __syncthreads();
    if (tid == 0) {
        // monotone terms: slot 2*o+1 (Hermite function of order o of x_c) and optional outer product over x_<c
        int no = 0;
        for (int o = 1; o <= 3; ++o) {
            const int s = 2 * o + 1;
            s_mond[o - 1] = (s < 2 * (P.maxord + 1)) ? P.db[P.o_d_slot_scale + s] : 0.0;
            if (s >= 2 * (P.maxord + 1)) continue;
            for (int jj = P.ib[P.o_slot_ptr + s]; jj < P.ib[P.o_slot_ptr + s + 1]; ++jj) s_tord[P.ib[P.o_slot_term + jj]] = o;
        }
        for (int j = 0; j < P.m_mon; ++j)
            if (P.ib[P.o_out_ptr + j] != P.ib[P.o_out_ptr + j + 1]) s_tout[j] = no++;
        double sc = 0.0;
        for (int q = 0; q < P.nconst; ++q) sc += a.coeffs[P.ib[P.o_const_idx + q]];
        s_mond[3] = sc;
    }
    if (GRAD)
        for (int e = tid; e < ndense * SL::NS * 32; e += TB) s_hacc[e] = 0.0;
    __syncthreads();

    const double* __restrict__ Xt = a.Xt;
    const int64_t ld = a.ld, N = a.N;
    const double* xc_col = Xt + (int64_t)P.c * ld;
    const double* bcoef = s_coef + P.m_non;
    const double sc1 = s_mond[0], sc2 = s_mond[1], sc3 = s_mond[2], Sconst = s_mond[3];
    const int m_mon = P.m_mon;

    double Jacc = 0.0, gconst = 0.0;
    double gm[MAXMON];
#pragma unroll
    for (int j = 0; j < MAXMON; ++j) gm[j] = 0.0;

    // block ranges in units of 32 samples (one warp row), NOT of tiles: every block gets N/grid samples within 32, so
    // the blocks finish together; the last tile of a block is partial and its empty warps skip the node loop
    // (tile-granular ranges cost 14 tiles where the average is 13.2 at N = 1M: 6 % of the kernel)
    const int64_t units = (N + 31) / 32;
    const int64_t s_lo = units * blockIdx.x / gridDim.x * 32;
    const int64_t s_end = units * (blockIdx.x + 1) / gridDim.x * 32;
    const int64_t s_hi = s_end < N ? s_end : N;
#pragma unroll 1
    for (int64_t base = s_lo; base < s_hi; base += TB) {
        const int64_t i = base + tid;
        const bool valid = i < s_hi;
        const bool warp_has_samples = base + 32 * warp < s_hi;
        // ---------------- phase 1: node loop ----------------
        if (!warp_has_samples) {                             // partial tile: nothing to integrate for this warp
            s_M[tid] = 0.0;
            if (GRAD) {                                      // the epilogue multiplies these by 0: keep them finite
#pragma unroll
                for (int q = 0; q < NPARK; ++q) s_park[q * TB + tid] = 0.0;
                for (int q = 0; q < a.n_out_terms; ++q) s_u[q * TB + tid] = 0.0;
            }
        } else {
            const double xc = valid ? xc_col[i] : 0.0;
            const double hx = 0.5 * xc;
            double C1 = 0.0, C2 = 0.0, C3 = 0.0;
#pragma unroll 1
            for (int j = 0; j < m_mon; ++j) {
                const int o = s_tord[j], uo = s_tout[j];
                double u = 1.0;
                if (uo >= 0) {
                    u = valid ? tile_outer_product(P, j, Xt, ld, i) : 0.0;
                    if (GRAD) s_u[uo * TB + tid] = u;
                }
                const double bu = bcoef[j] * u;
                C1 += (o == 1) ? bu : 0.0;
                C2 += (o == 2) ? bu : 0.0;
                C3 += (o == 3) ? bu : 0.0;
            }
            C1 *= sc1; C2 *= sc2; C3 *= sc3;
            // r(t) = e^{-t^2/4} (C1 He1 + C2 He2 + C3 He3)(t) at t = hx tau:  e^{ya tau^2} (((E3 tau + E2) tau + E1) tau + E0)
            const double hx2 = hx * hx;
            const double ya = -0.25 * hx2;
            const double E3 = C3 * (hx2 * hx), E2 = C2 * hx2, E1 = fma(-3.0, C3, C1) * hx, E0 = -C2;
            const double EK[4] = {E0 * TTM_E32_K, E1 * TTM_E32_K, E2 * TTM_E32_K, E3 * TTM_E32_K};
            double Sacc = 0.0, m0 = 0.0, m1 = 0.0, m2 = 0.0, m3 = 0.0;   // moments of w g' e^{-t^2/4} in tau
            // both exp arguments in [-700, 700] on every node (tau <= 2, e^{ya tau^2} <= 1; fails on NaN): no clamps
            const double rbound = fabs(E0) + 2.0 * fabs(E1) + 4.0 * fabs(E2) + 8.0 * fabs(E3);
            if (__all_sync(0xffffffffu, ya >= -175.0 && rbound < 700.0))
                node_loop<GRAD, NQ, true>(nt.v, Qp, ya, EK, s_tab, Sacc, m0, m1, m2, m3);
            else
                node_loop<GRAD, NQ, false>(nt.v, Qp, ya, EK, s_tab, Sacc, m0, m1, m2, m3);
            // back to t = hx tau:  sum w g' e^{-t^2/4} t^i = hx^i m_i
            m1 *= hx; m2 *= hx2; m3 *= hx2 * hx;
            const double M = valid ? hx * fma(a.delta, a.wsum, Sacc) : 0.0;   // sum_q hx w_q (g_q + delta)
            s_M[tid] = M;
            if (GRAD) {
                // values at x_c: log-derivative term of the objective and its coefficient gradient
                const double xx = xc * xc;
                const double P2 = xx - 1.0, P3 = xc * (xx - 3.0);
                const double gax = exp_neg_1(-0.25 * xx, s_tab);
                const double rc = gax * fma(C3, P3, fma(C2, P2, C1 * xc));
                const double gc = exp_gen_1(rc, s_tab);
                const double Lg = (a.delta == 0.0) ? rc : log(gc + a.delta);
                const double ratio = gc / (gc + a.delta);
                double* pk = s_park + tid;
                pk[0 * TB] = Lg;
                pk[1 * TB] = ratio;
                pk[2 * TB] = hx * m1;                      // hx * int g' He1 e^{-t^2/4}
                pk[3 * TB] = hx * (m2 - m0);               // He2 = t^2 - 1
                pk[4 * TB] = hx * fma(-3.0, m1, m3);       // He3 = t^3 - 3t
                pk[5 * TB] = xc * gax;
                pk[6 * TB] = P2 * gax;
                pk[7 * TB] = P3 * gax;
            }
        }
        __syncthreads();
        // ---------------- phase 2: sweep over x_<c ----------------
        const bool full = base + TB <= s_hi;
        if (full)
            sweep_tile<MASK, true, GRAD && MERGED, true>(Xt, ld, base, s_hi, ndense, s_col, s_prod, s_M, s_Spart, s_hacc, s_tab, warp, lane);
        else
            sweep_tile<MASK, true, GRAD && MERGED, false>(Xt, ld, base, s_hi, ndense, s_col, s_prod, s_M, s_Spart, s_hacc, s_tab, warp, lane);
        __syncthreads();
        // ---------------- phase 3: per-sample epilogue ----------------
        {
            const double M = s_M[tid];
            double S = Sconst;
#pragma unroll
            for (int w = 0; w < NWARP; ++w) S += s_Spart[w * TB + tid];
            S += M;
            if (!GRAD) {
                if (valid) a.S_out[i] = S;
            } else {
                const double* pk = s_park + tid;
                const double vf = valid ? 1.0 : 0.0;
                Jacc += vf * (0.5 * S * S - pk[0 * TB]);
                gconst += vf * (MERGED ? M : S);
                const double ratio = pk[1 * TB];
                const double W1 = vf * sc1 * (S * pk[2 * TB] - ratio * pk[5 * TB]);
                const double W2 = vf * sc2 * (S * pk[3 * TB] - ratio * pk[6 * TB]);
                const double W3 = vf * sc3 * (S * pk[4 * TB] - ratio * pk[7 * TB]);
#pragma unroll
                for (int j = 0; j < MAXMON; ++j) {
                    if (j < m_mon) {
                        const int o = s_tord[j], uo = s_tout[j];
                        const double W = (o == 1) ? W1 : ((o == 2) ? W2 : W3);
                        const double u = (uo >= 0) ? s_u[uo * TB + tid] : 1.0;
                        gm[j] = fma(u, W, gm[j]);
                    }
                }
                if (!MERGED) s_M[tid] = vf * S;            // weights of the gradient sweep (s_M[tid] is only read by tid)
            }
        }
        if (GRAD && !MERGED) {
            __syncthreads();
            if (full)
                sweep_tile<MASK, false, true, true>(Xt, ld, base, s_hi, ndense, s_col, s_prod, s_M, s_Spart, s_hacc, s_tab, warp, lane);
            else
                sweep_tile<MASK, false, true, false>(Xt, ld, base, s_hi, ndense, s_col, s_prod, s_M, s_Spart, s_hacc, s_tab, warp, lane);
            __syncthreads();                               // s_M is rewritten by the next tile's phase 1
        }
    }
    if (!GRAD) return;

    // ---- block partial
    __syncthreads();
    {
        double v0 = warp_sum(Jacc), v1 = warp_sum(gconst);
        if (lane == 0) { s_red[warp * (2 + MAXMON)] = v0; s_red[warp * (2 + MAXMON) + 1] = v1; }
#pragma unroll
        for (int j = 0; j < MAXMON; ++j) {
            const double v = warp_sum(gm[j]);
            if (lane == 0) s_red[warp * (2 + MAXMON) + 2 + j] = v;
        }
    }
    for (int j = tid; j < 1 + m; j += TB) s_outv[j] = 0.0;
    __syncthreads();
    if (tid < 2 + MAXMON) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < NWARP; ++w) v += s_red[w * (2 + MAXMON) + tid];
        if (tid == 0) s_outv[0] = v;
        else if (tid == 1) {
            for (int q = 0; q < P.nconst; ++q) s_outv[1 + P.ib[P.o_const_idx + q]] = v;
        } else if (tid - 2 < m_mon) s_outv[1 + P.m_non + tid - 2] = v;
    }
    for (int e = tid; e < ndense * SL::NS; e += TB) {
        const int g = e / SL::NS, si = e - g * SL::NS;
        int slot = 0, cnt = -1;                            // si-th set bit of MASK
#pragma unroll
        for (int b = 0; b < 8; ++b)
            if ((MASK >> b) & 1) { ++cnt; if (cnt == si) slot = b; }
        const int j = (slot < dstride) ? P.ib[P.o_dense_idx + g * dstride + slot] : -1;
        if (j >= 0) {
            const double* hp = s_hacc + e * 32;
            double v = 0.0;
            for (int l = 0; l < 32; ++l) v += hp[(l + tid) & 31];
            s_outv[1 + j] = v * P.db[P.o_d_dense_scale + g * dstride + slot];
        }
    }
    __syncthreads();
    double* part = a.partials + (int64_t)blockIdx.x * (1 + m);
    for (int j = tid; j < 1 + m; j += TB) part[j] = s_outv[j];
    __threadfence();
    __shared__ unsigned int s_last;
    __syncthreads();
    if (tid == 0) s_last = (atomicAdd(a.counter, 1u) == gridDim.x - 1) ? 1u : 0u;
    __syncthreads();
    if (s_last) {
        __threadfence();
        const double invN = 1.0 / (double)N;
        for (int j = tid; j < 1 + m; j += TB) {
            double v = 0.0;
            for (unsigned int b = 0; b < gridDim.x; ++b) v += __ldcg(a.partials + (int64_t)b * (1 + m) + j);
            a.out[j] = v * invN;
            if (a.out_host) a.out_host[j] = v * invN;
        }
        if (a.out_host) {                       // result visible in host memory before the sequence number is
            __threadfence_system();
            __syncthreads();
            if (tid == 0) *reinterpret_cast<volatile unsigned long long*>(a.flag_host) = a.seq;
        }
        if (tid == 0) *a.counter = 0u;
    }
}

template <int MASK, bool GRAD, bool MERGED, int NQ>
cudaError_t launch_one(const ObjArgs& a, const NodeTab& nt, int grid, size_t smem, cudaStream_t st) {
    auto k = objgrad_tile_kernel<MASK, GRAD, MERGED, NQ>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k<<<grid, TB, smem, st>>>(a, nt);
    return cudaGetLastError();
}

constexpr int MASK_C4 = (1 << 2) | (1 << 5) | (1 << 7);   // {He1, He2 e^{-x^2/4}, He3 e^{-x^2/4}} per variable
constexpr int MASK_ALL = 0xFC;

template <int MASK, int NQ>
cudaError_t launch_mask(const ObjArgs& a_in, bool grad, int sm_count, cudaStream_t st) {
    ObjArgs a = a_in;
    const PlanView& P = a.P;
    const int m = P.m_non + P.m_mon;
    const Layout LY = make_layout(m, P.ndense, Slots<MASK>::NS, a.n_out_terms, grad);
    const size_t smem = sizeof(double) * (size_t)LY.total;
    const int Qp = (a.Q + NQ - 1) / NQ * NQ;
    if (smem > 227 * 1024 || Qp > MAXQ || !a.h_xis || !a.h_ws) return cudaErrorInvalidValue;
    *reinterpret_cast<Layout*>(a.lay) = LY;
    NodeTab nt;
    for (int q = 0; q < Qp; ++q) {                            // padding nodes: tau = 0, zero weight
        const double tau = (q < a.Q) ? 1.0 + a.h_xis[q] : 0.0, w = (q < a.Q) ? a.h_ws[q] : 0.0;
        const double t2 = tau * tau;
        double* v = nt.v + 6 * q;
        v[0] = tau; v[1] = t2 * TTM_E32_K; v[2] = w; v[3] = w * tau; v[4] = w * t2; v[5] = w * (t2 * tau);
    }
    const int64_t tiles = (a.N + TB - 1) / TB;
    const int bps = a.blocks_per_sm > 0 ? (a.blocks_per_sm > 2 ? 2 : a.blocks_per_sm) : 2;
    int64_t g = (int64_t)sm_count * bps;
    if (g > tiles) g = tiles;
    if (g > a.max_grid) g = a.max_grid;
    const int grid = (int)(g < 1 ? 1 : g);
    if (!grad) return launch_one<MASK, false, false, NQ>(a, nt, grid, smem, st);
    if (a.gram_mode) return launch_one<MASK, true, true, NQ>(a, nt, grid, smem, st);
    return launch_one<MASK, true, false, NQ>(a, nt, grid, smem, st);
}

}  // namespace ttm_tile

// cudaErrorNotSupported: the plan is outside the tile kernel's class (the caller falls back to the general kernel)
cudaError_t ttm_launch_objgrad_tile(const ObjArgs& a, bool grad, int sm_count, cudaStream_t st) {
    if (!a.tile_ok || a.rect != RECT_EXP) return cudaErrorNotSupported;
    cudaError_t e;
    // nodes in flight per thread: 4, or 5 when that divides the rule (Q = 25: no padding nodes; 6 and 8 measured no faster)
    const bool nq5 = (a.Q % 4 != 0) && (a.Q % 5 == 0);
    if ((a.dense_mask & ~ttm_tile::MASK_C4) == 0)
        e = nq5 ? ttm_tile::launch_mask<ttm_tile::MASK_C4, 5>(a, grad, sm_count, st)
                : ttm_tile::launch_mask<ttm_tile::MASK_C4, 4>(a, grad, sm_count, st);
    else e = ttm_tile::launch_mask<ttm_tile::MASK_ALL, 4>(a, grad, sm_count, st);
    return (e == cudaErrorInvalidValue) ? cudaErrorNotSupported : e;
}
