// K-objgrad / K-S (integrated rectifier): fused objective + gradient of one map component.
//
// Replaces, in ONE launch, the reference's three quadrature sweeps per optimizer callback pair:
//   objective_function            transport_map.py:3300-3433
//   objective_function_jacobian   transport_map.py:3435-3635
//   s (integrated-rectifier arm)  transport_map.py:2439-2547
//   GaussQuadrature vector branch transport_map.py:4202-4278
//   rectifier                     transport_map.py:4956-5213
//
// Work decomposition per thread block (T threads) over a contiguous range of sample rows:
//   phase A  S_non[r]  = sum_j a_j psi^non_j(x_<c)      -- variable-major sweep, R samples/thread
//   phase B  node loop: M = int_0^{x_c} g(sum_j b_j psi^mon_j) dt, I_s = int g' phi_s dt per *slot*
//            (slot = distinct univariate factor of x_c; outer factors u_j(x_<c) are folded into the
//            slot coefficients C_s = sum_j b_j u_j, so the loop body is independent of m_mon)
//   phase C  dJ/da_j   = sum_i S_i psi^non_j(x_i)        -- same sweep as A, warp-reduced per term
// Block partials go to a [grid][1+m] buffer; the last block to finish reduces them in fixed
// block order (bit-reproducible), divides by N and writes (J, grad) to `out`.
//
// Bound: FP64 pipe (two exp per quadrature node), not HBM: algorithmic bytes 8*N*(c+1).
//
// This header is included by one translation unit per instantiation (ttm_objgrad_cfg*.cu) so the
// variants compile in parallel.
#pragma once

#include "ttm_common.cuh"
#include "ttm_kernels.h"
#include "ttm_sweep.cuh"

namespace ttm_obj {

constexpr int T_OBJ = 128;   // threads per block
constexpr int CH_ROWS = 16;  // rows per chunk between two dense phase-C passes (multiple of R_OBJ and RC_SWEEP)
constexpr int RC_SWEEP = 4;  // rows per thread in flight in the dense sweeps (8 independent exp chains)

// ---- polynomial ladder on the inner variable: fills P[0..MAXORD] ----
template <int MAXORD, bool HERME>
__device__ __forceinline__ void ladder(double t, const double* __restrict__ rec, double (&P)[MAXORD + 1]) {
    P[0] = 1.0;
    if (HERME) {
        if (MAXORD >= 1) P[1] = t;
#pragma unroll
        for (int n = 1; n < MAXORD; ++n) P[n + 1] = fma(t, P[n], -(double)n * P[n - 1]);
    } else {
        if (MAXORD >= 1) P[1] = fma(rec[0], t, rec[MAXORD + 1]);
#pragma unroll
        for (int n = 1; n < MAXORD; ++n)
            P[n + 1] = fma(fma(rec[n], t, rec[MAXORD + 1 + n]), P[n], -rec[2 * (MAXORD + 1) + n] * P[n - 1]);
    }
}

// Dynamic shared-memory layout of objgrad_kernel (offsets in doubles): the launcher sizes the launch with `total` and
// passes the offsets in ObjArgs::lay, from which the kernel takes its pointers.
struct Layout {
    int o_coef, o_xis, o_ws, o_exptab, o_rec, o_scale, o_gacc;
    int o_dense;                                      // dense-group tables (stage_dense_tables)
    int o_slot_ptr, o_slot_term, o_out_ptr, o_out_fac;  // ints
    int o_S, o_M, o_I, total;
};
static_assert(sizeof(Layout) <= sizeof(((ObjArgs*)nullptr)->lay), "ObjArgs::lay too small");

// maxord, nq: the instantiation's MAXORD and NQ; gram: Gram mode (GRAD only); ch_rows: rows per chunk
inline Layout make_layout(const PlanView& P, int Q, int maxord, int nq, bool grad, bool gram, int ch_rows) {
    const int m = P.m_non + P.m_mon;
    const int nslot = 2 * (P.maxord + 1) + P.nst;
    const int qp = (Q + nq - 1) / nq * nq;            // node count padded to a multiple of NQ
    Layout L;
    int o = 0;
    L.o_coef = o;      o += m;
    L.o_xis = o;       o += qp;
    L.o_ws = o;        o += qp;
    L.o_exptab = o;    o += 32;                       // 2^(j/32), j < 32: the exp table of the node loop
    L.o_rec = o;       o += 3 * (maxord + 1);         // recurrence coefficients A | B | C
    L.o_scale = o;     o += nslot;
    L.o_gacc = o;      o += grad ? (T_OBJ / 32) * (1 + m) : 0;   // per warp: J, gradient
    L.o_dense = o;     o += dense_smem_doubles(P.ndense, P.dense_maxord);
    // monotone slot tables (the per-row-group prologue/epilogue walks them; from L2 they cost ~300 cycles per hop)
    L.o_slot_ptr = o;  o += (nslot + 2) / 2;          // [nslot + 1]
    L.o_slot_term = o; o += (P.m_mon + 1) / 2;        // [m_mon]
    L.o_out_ptr = o;   o += (P.m_mon + 2) / 2;        // [m_mon + 1]
    L.o_out_fac = o;   o += (P.n_outfac + 1) / 2;     // [n_outfac]
    L.o_S = o;         o += ch_rows * T_OBJ;          // [ch_rows][T_OBJ]
    L.o_M = o;         o += gram ? ch_rows * T_OBJ : 0;                // [ch_rows][T_OBJ]
    L.o_I = o;         o += gram ? P.nactive * ch_rows * T_OBJ : 0;    // [nactive][ch_rows][T_OBJ]
    L.total = o;
    return L;
}

// outer (x_<c) product of monotone term j on sample i; 1 if the term has no outer factor
static __device__ __noinline__ double outer_product(const PlanView& P, const int* __restrict__ out_ptr,
                                                    const int* __restrict__ out_fac, int j,
                                                    const double* __restrict__ Xt, int64_t ld, int64_t i) {
    const int b = out_ptr[j], e = out_ptr[j + 1];
    double v = 1.0;
    for (int q = b; q < e; ++q) v *= plan_factor(P, out_fac[q], Xt, ld, i);
    return v;
}

template <int MAXORD, bool HAS_PLAIN, bool HAS_HF, int NST, bool HERME, bool EXPRECT, bool GRAD, int RB, int NQ>
__global__ void __launch_bounds__(T_OBJ) objgrad_kernel(const ObjArgs a) {
    extern __shared__ __align__(16) double smem[];
    const PlanView& P = a.P;
    const int m = P.m_non + P.m_mon;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = T_OBJ / 32;
    constexpr int NSLOT_T = 2 * (MAXORD + 1) + NST;       // slots of this instantiation
    constexpr int NSTA = NST > 0 ? NST : 1;
    const int st_base = 2 * (P.maxord + 1);               // first special-term slot of the plan
    const int nslot_rt = st_base + P.nst;

    const Layout& L = *reinterpret_cast<const Layout*>(a.lay);
    const int Qp = L.o_ws - L.o_xis;                     // node count padded to a multiple of NQ
    double* s_coef = smem + L.o_coef;
    double* s_xis = smem + L.o_xis;
    double* s_ws = smem + L.o_ws;
    double* s_exptab = smem + L.o_exptab;
    double* s_rec = smem + L.o_rec;
    double* s_scale = smem + L.o_scale;
    double* s_gacc = smem + L.o_gacc;
    int* s_slot_ptr = reinterpret_cast<int*>(smem + L.o_slot_ptr);
    int* s_slot_term = reinterpret_cast<int*>(smem + L.o_slot_term);
    int* s_out_ptr = reinterpret_cast<int*>(smem + L.o_out_ptr);
    int* s_out_fac = reinterpret_cast<int*>(smem + L.o_out_fac);
    double* s_S = smem + L.o_S;
    double* s_M = smem + L.o_M;
    double* s_I = smem + L.o_I;

    for (int j = tid; j < m; j += T_OBJ) s_coef[j] = a.coeffs[j];
    for (int q = tid; q < Qp; q += T_OBJ) {              // padding nodes: mid-point, zero weight
        s_xis[q] = (q < a.Q) ? a.xis[q] : 0.0;
        s_ws[q] = (q < a.Q) ? a.ws[q] : 0.0;
    }
    for (int j = tid; j < 32; j += T_OBJ) s_exptab[j] = g_ttm_exp2_tab[j];
    for (int n = tid; n < 3 * (MAXORD + 1); n += T_OBJ) {
        double A, B, C;
        rec_coef(P.family, n % (MAXORD + 1), A, B, C);
        s_rec[n] = (n / (MAXORD + 1) == 0) ? A : ((n / (MAXORD + 1) == 1) ? B : C);
    }
    for (int s = tid; s < nslot_rt; s += T_OBJ) s_scale[s] = P.db[P.o_d_slot_scale + s];
    if (GRAD)
        for (int j = tid; j < NW * (1 + m); j += T_OBJ) s_gacc[j] = 0.0;
    const DenseSmem DS = stage_dense_tables(P, a.coeffs, L.o_dense, tid, T_OBJ);
    for (int e = tid; e <= nslot_rt; e += T_OBJ) s_slot_ptr[e] = P.ib[P.o_slot_ptr + e];
    for (int e = tid; e < P.m_mon; e += T_OBJ) s_slot_term[e] = P.ib[P.o_slot_term + e];
    for (int e = tid; e <= P.m_mon; e += T_OBJ) s_out_ptr[e] = P.ib[P.o_out_ptr + e];
    for (int e = tid; e < P.n_outfac; e += T_OBJ) s_out_fac[e] = P.ib[P.o_out_fac + e];
    __syncthreads();

    const double* acoef = s_coef;
    const double* bcoef = s_coef + P.m_non;
    double* gslot = s_gacc + warp * (1 + m) + 1;  // gradient slots of this warp (slot -1 = J)
    const double* __restrict__ Xt = a.Xt;
    const int64_t ld = a.ld, N = a.N;
    const double* xc_col = Xt + (int64_t)P.c * ld;

    // special-term inner factors (generic instantiation only)
    int4 sti[NSTA];
    double4 std_[NSTA];
    if (NST > 0) {
#pragma unroll
        for (int q = 0; q < NST; ++q) {
            sti[q] = make_int4(0, F_ZERO, 0, 0);
            std_[q] = make_double4(0, 0, 0, 1);
            if (q < P.nst) {
                const int f = __ldg(P.ib + P.o_st_fac + q);
                sti[q] = __ldg(reinterpret_cast<const int4*>(P.ib + P.o_fac_i) + f);
                std_[q] = ldg_d4(reinterpret_cast<const double4*>(P.db + P.o_d_fac) + f);
            }
        }
    }

    double Jacc = 0.0;
    const int64_t rows = (N + T_OBJ - 1) / T_OBJ;
    const int64_t row_lo = rows * blockIdx.x / gridDim.x, row_hi = rows * (blockIdx.x + 1) / gridDim.x;

    // Gram mode (GRAD only): dJ/da = G a + h with G = Psi_non^T Psi_non / N precomputed on the host side of the
    // ABI; the kernel then needs ONE nonmonotone sweep per chunk (value and h together) instead of two:
    //   pass 1  node loops of the chunk            -> M_i and the slot integrals I_{i,s} parked in shared memory
    //   sweep   S_non and h_j = sum_i M_i psi_ij   (dense_merged_chunk_smem)
    //   pass 2  epilogue: S = S_non + M, J, monotone gradient
    // Otherwise (pass 0): phase A sweep, node loop + epilogue, phase C sweep.
    const bool gm = GRAD && a.gram_mode != 0;
    const int ch_rows = a.ch_rows;
    for (int64_t chunk_lo = row_lo; chunk_lo < row_hi; chunk_lo += ch_rows) {
    const int64_t chunk_hi = (chunk_lo + ch_rows < row_hi) ? chunk_lo + ch_rows : row_hi;
    if (!gm) {
        // ---------------- phase A, dense groups: S_non of the whole chunk -> s_S ----------------
        for (int64_t row8 = chunk_lo; row8 < chunk_hi; row8 += RC_SWEEP) {
            bool okr[RC_SWEEP];
            double S8[RC_SWEEP];
#pragma unroll
            for (int r = 0; r < RC_SWEEP; ++r) {
                okr[r] = (row8 + r < chunk_hi) && ((row8 + r) * T_OBJ + tid < N);
                S8[r] = 0.0;
            }
            dense_value_smem<HERME, 3, RC_SWEEP>(P, DS, Xt, ld, row8 * T_OBJ + tid, T_OBJ, okr, S8);
#pragma unroll
            for (int r = 0; r < RC_SWEEP; ++r)
                if (row8 + r < chunk_hi) s_S[(row8 + r - chunk_lo) * T_OBJ + tid] = S8[r];
        }
    }
#pragma unroll 1
    for (int pass = gm ? 1 : 0; pass <= (gm ? 2 : 0); ++pass) {
    if (pass == 2)
        dense_merged_chunk_smem<HERME, RC_SWEEP>(P, DS, Xt, ld, chunk_lo, chunk_hi, N, T_OBJ, tid, s_M, s_S, gslot, lane);
    for (int64_t row0 = chunk_lo; row0 < chunk_hi; row0 += R_OBJ) {
        int64_t idx[R_OBJ];
        double valid[R_OBJ], S[R_OBJ], Mv[R_OBJ];
#pragma unroll
        for (int r = 0; r < R_OBJ; ++r) {
            const int64_t i = (row0 + r) * T_OBJ + tid;
            const bool ok = (row0 + r < chunk_hi) && (i < N);
            valid[r] = ok ? 1.0 : 0.0;
            idx[r] = ok ? i : (N - 1);
            const bool in = row0 + r < chunk_hi;
            S[r] = (in && pass != 1) ? s_S[(row0 + r - chunk_lo) * T_OBJ + tid] : 0.0;
            Mv[r] = (in && pass == 2) ? s_M[(row0 + r - chunk_lo) * T_OBJ + tid] : 0.0;
        }
        // ---------------- phase A (constants, special terms, multivariate terms) ----------------
        if (pass != 1) nonmon_generic_sweep<false, HERME>(P, Xt, ld, idx, acoef, S, gslot, lane);
        if (pass == 2) nonmon_generic_sweep<true, HERME>(P, Xt, ld, idx, acoef, Mv, gslot, lane);  // their h_j

        // ---------------- phase B ----------------
#pragma unroll 1
        for (int r0 = 0; r0 < R_OBJ; r0 += RB) {
            if (row0 + r0 >= chunk_hi) {     // rows past the chunk (uniform over the block)
#pragma unroll
                for (int r = 0; r < R_OBJ; ++r)
                    if (r >= r0) S[r] = 0.0;
                break;
            }
            double hx[RB], xc[RB], Sacc[RB];
            double Cp[MAXORD + 1][RB], Ch[MAXORD + 1][RB], Cs[NSTA][RB];
            double Ip[MAXORD + 1][RB], Ih[MAXORD + 1][RB], Is[NSTA][RB];
            double tmp[RB][NSLOT_T];  // staging between the rolled (per plan slot) and unrolled code
#pragma unroll
            for (int rb = 0; rb < RB; ++rb) {
                xc[rb] = xc_col[idx[r0 + rb]];
                hx[rb] = 0.5 * xc[rb];
                Sacc[rb] = 0.0;
#pragma unroll
                for (int s = 0; s < NSLOT_T; ++s) tmp[rb][s] = 0.0;
            }
            // slot coefficients C_s = scale_s * sum_{j in s} b_j u_j   (rolled over the plan's slots)
#pragma unroll 1
            for (int s = 0; s < nslot_rt; ++s) {
                const int j0 = s_slot_ptr[s], j1 = s_slot_ptr[s + 1];
                if (j0 == j1) continue;
                const int ts = (s < st_base) ? s : 2 * (MAXORD + 1) + (s - st_base);
                double acc[RB];
#pragma unroll
                for (int rb = 0; rb < RB; ++rb) acc[rb] = 0.0;
                for (int jj = j0; jj < j1; ++jj) {
                    const int j = s_slot_term[jj];
                    const double b = bcoef[j];
                    const bool has_outer = s_out_ptr[j] != s_out_ptr[j + 1];
#pragma unroll
                    for (int rb = 0; rb < RB; ++rb)
                        acc[rb] = fma(b, has_outer ? outer_product(P, s_out_ptr, s_out_fac, j, Xt, ld, idx[r0 + rb]) : 1.0, acc[rb]);
                }
                const double sc = s_scale[s];
#pragma unroll
                for (int rb = 0; rb < RB; ++rb) tmp[rb][ts] = acc[rb] * sc;
            }
#pragma unroll
            for (int rb = 0; rb < RB; ++rb) {
#pragma unroll
                for (int o = 0; o <= MAXORD; ++o) {
                    Cp[o][rb] = tmp[rb][2 * o]; Ip[o][rb] = 0.0;
                    Ch[o][rb] = tmp[rb][2 * o + 1]; Ih[o][rb] = 0.0;
                }
#pragma unroll
                for (int q = 0; q < NST; ++q) { Cs[q][rb] = tmp[rb][2 * (MAXORD + 1) + q]; Is[q][rb] = 0.0; }
            }

            // r(t) and the slot basis values at t for sample rb
            auto inner = [&](int rb, double t, double (&Pl)[MAXORD + 1], double& ga, double (&sv)[NSTA]) {
                ladder<MAXORD, HERME>(t, s_rec, Pl);
                double r = 0.0;
                if (HAS_HF) {
                    ga = ttm_exp_neg(-0.25 * t * t);
                    double u = 0.0;
#pragma unroll
                    for (int o = 1; o <= MAXORD; ++o) u = fma(Ch[o][rb], Pl[o], u);
                    r = ga * u;
                }
                if (HAS_PLAIN) {
#pragma unroll
                    for (int o = 0; o <= MAXORD; ++o) r = fma(Cp[o][rb], Pl[o], r);
                }
                if (NST > 0) {
#pragma unroll 1
                    for (int q = 0; q < NST; ++q) {
                        sv[q] = (q < P.nst) ? eval_factor(sti[q].y, sti[q].z, std_[q].x, std_[q].y, std_[q].z, std_[q].w, P.family, t) : 0.0;
                        r = fma(Cs[q][rb], sv[q], r);
                    }
                }
                return r;
            };

            // ---- Gauss-Legendre node loop (transport_map.py:4252-4278) ----
            if (pass != 2) {
            if (NST == 0) {
                // staged ("vector") form: L = NQ x RB node-samples advance through every stage together
                constexpr int L = NQ * RB;
#pragma unroll 1
                for (int q = 0; q < Qp; q += NQ) {
                    double t[L], Pl[L][MAXORD + 1], ga[L], r[L], g[L];
#pragma unroll
                    for (int l = 0; l < L; ++l) t[l] = fma(hx[l % RB], s_xis[q + l / RB], hx[l % RB]);
#pragma unroll
                    for (int l = 0; l < L; ++l) ladder<MAXORD, HERME>(t[l], s_rec, Pl[l]);
                    if (HAS_HF) {
                        double y[L];
#pragma unroll
                        for (int l = 0; l < L; ++l) y[l] = -0.25 * t[l] * t[l];
                        ttm_exp_neg_v<L, true>(y, ga, s_exptab);
#pragma unroll
                        for (int l = 0; l < L; ++l) r[l] = Ch[1][l % RB] * Pl[l][1];
#pragma unroll
                        for (int o = 2; o <= MAXORD; ++o) {
#pragma unroll
                            for (int l = 0; l < L; ++l) r[l] = fma(Ch[o][l % RB], Pl[l][o], r[l]);
                        }
#pragma unroll
                        for (int l = 0; l < L; ++l) r[l] *= ga[l];
                    } else {
#pragma unroll
                        for (int l = 0; l < L; ++l) { r[l] = 0.0; ga[l] = 1.0; }
                    }
                    if (HAS_PLAIN) {
#pragma unroll
                        for (int o = 0; o <= MAXORD; ++o) {
#pragma unroll
                            for (int l = 0; l < L; ++l) r[l] = fma(Cp[o][l % RB], Pl[l][o], r[l]);
                        }
                    }
                    if (EXPRECT) {
                        ttm_exp_v<L, true>(r, g, s_exptab);
                    } else {
#pragma unroll
                        for (int l = 0; l < L; ++l) g[l] = rect_eval(a.rect, r[l]);
                    }
#pragma unroll
                    for (int l = 0; l < L; ++l) {
                        const int rb = l % RB;
                        const double w = s_ws[q + l / RB];
                        Sacc[rb] = fma(w, g[l], Sacc[rb]);
                        if (GRAD) {
                            const double wd = w * (EXPRECT ? g[l] : rect_dfac(a.rect, r[l], g[l]));
                            if (HAS_PLAIN) {
#pragma unroll
                                for (int o = 0; o <= MAXORD; ++o) Ip[o][rb] = fma(wd, Pl[l][o], Ip[o][rb]);
                            }
                            if (HAS_HF) {
                                const double wg = wd * ga[l];
#pragma unroll
                                for (int o = 1; o <= MAXORD; ++o) Ih[o][rb] = fma(wg, Pl[l][o], Ih[o][rb]);
                            }
                        }
                    }
                }
            } else {
#pragma unroll 1
                for (int q = 0; q < Qp; q += NQ) {
#pragma unroll
                    for (int u = 0; u < NQ; ++u) {
                        const double xi = s_xis[q + u], w = s_ws[q + u];
#pragma unroll
                        for (int rb = 0; rb < RB; ++rb) {
                            const double t = fma(hx[rb], xi, hx[rb]);
                            double Pl[MAXORD + 1], ga = 1.0, sv[NSTA];
                            const double r = inner(rb, t, Pl, ga, sv);
                            const double g = EXPRECT ? ttm_exp(r) : rect_eval(a.rect, r);
                            Sacc[rb] = fma(w, g, Sacc[rb]);
                            if (GRAD) {
                                const double wd = w * (EXPRECT ? g : rect_dfac(a.rect, r, g));
                                if (HAS_PLAIN) {
#pragma unroll
                                    for (int o = 0; o <= MAXORD; ++o) Ip[o][rb] = fma(wd, Pl[o], Ip[o][rb]);
                                }
                                if (HAS_HF) {
                                    const double wg = wd * ga;
#pragma unroll
                                    for (int o = 1; o <= MAXORD; ++o) Ih[o][rb] = fma(wg, Pl[o], Ih[o][rb]);
                                }
                                if (NST > 0) {
#pragma unroll
                                    for (int qq = 0; qq < NST; ++qq) Is[qq][rb] = fma(wd, sv[qq], Is[qq][rb]);
                                }
                            }
                        }
                    }
                }
            }
            }

            // slot integrals I_s into the slot-indexed staging array
            if (GRAD && pass != 2) {
#pragma unroll
                for (int rb = 0; rb < RB; ++rb) {
#pragma unroll
                    for (int o = 0; o <= MAXORD; ++o) {
                        tmp[rb][2 * o] = HAS_PLAIN ? Ip[o][rb] : 0.0;
                        tmp[rb][2 * o + 1] = (HAS_HF && o > 0) ? Ih[o][rb] : 0.0;
                    }
#pragma unroll
                    for (int q = 0; q < NST; ++q) tmp[rb][2 * (MAXORD + 1) + q] = Is[q][rb];
                }
            }
            if (pass == 1) {
                // park M_i and the integrals of the non-empty slots; the epilogue runs after the merged sweep
                int ai = 0;
#pragma unroll 1
                for (int s = 0; s < nslot_rt; ++s) {
                    if (s_slot_ptr[s] == s_slot_ptr[s + 1]) continue;
                    const int ts = (s < st_base) ? s : 2 * (MAXORD + 1) + (s - st_base);
#pragma unroll
                    for (int rb = 0; rb < RB; ++rb)
                        if (row0 + r0 + rb < chunk_hi)
                            s_I[(ai * ch_rows + (int)(row0 + r0 + rb - chunk_lo)) * T_OBJ + tid] = tmp[rb][ts];
                    ++ai;
                }
#pragma unroll
                for (int rb = 0; rb < RB; ++rb)
                    if (row0 + r0 + rb < chunk_hi)
                        s_M[(row0 + r0 + rb - chunk_lo) * T_OBJ + tid] =
                            valid[r0 + rb] * hx[rb] * fma(a.delta, a.wsum, Sacc[rb]);
                continue;
            }
            if (pass == 2) {
                int ai = 0;
#pragma unroll 1
                for (int s = 0; s < nslot_rt; ++s) {
                    if (s_slot_ptr[s] == s_slot_ptr[s + 1]) continue;
                    const int ts = (s < st_base) ? s : 2 * (MAXORD + 1) + (s - st_base);
#pragma unroll
                    for (int rb = 0; rb < RB; ++rb)
                        tmp[rb][ts] = (row0 + r0 + rb < chunk_hi)
                                          ? s_I[(ai * ch_rows + (int)(row0 + r0 + rb - chunk_lo)) * T_OBJ + tid] : 0.0;
                    ++ai;
                }
            }

            // ---- per-sample epilogue ----
            double Sfull[RB], ratio[RB];
            double base[RB][NSLOT_T];   // slot basis values at x_c (local memory, indexed by plan slot below)
#pragma unroll
            for (int rb = 0; rb < RB; ++rb) {
                const double M = (pass == 2) ? Mv[r0 + rb]
                                             : hx[rb] * fma(a.delta, a.wsum, Sacc[rb]);  // sum_q hx w_q (g_q + delta)
                Sfull[rb] = S[r0 + rb] + M;
                if (GRAD) {
                    double Plx[MAXORD + 1], gax = 1.0, svx[NSTA];
                    const double rc = inner(rb, xc[rb], Plx, gax, svx);
                    const double gc = EXPRECT ? ttm_exp(rc) : rect_eval(a.rect, rc);
                    const double L = rect_log(a.rect, rc, gc, a.delta);
                    ratio[rb] = (EXPRECT ? gc : rect_dfac(a.rect, rc, gc)) / (gc + a.delta);
                    Jacc += valid[r0 + rb] * (0.5 * Sfull[rb] * Sfull[rb] - L);
                    S[r0 + rb] = valid[r0 + rb] * Sfull[rb];
#pragma unroll
                    for (int o = 0; o <= MAXORD; ++o) {
                        base[rb][2 * o] = Plx[o];
                        base[rb][2 * o + 1] = Plx[o] * gax;
                    }
#pragma unroll
                    for (int q = 0; q < NST; ++q) base[rb][2 * (MAXORD + 1) + q] = svx[q];
                } else {
                    S[r0 + rb] = Sfull[rb];
                }
            }
            if (GRAD) {
                // dJ/db_j = sum_i u_ij [ S_i hx_i I_{i,s} - ratio_i phi_s(x_ic) ],  s = slot of term j
#pragma unroll 1
                for (int s = 0; s < nslot_rt; ++s) {
                    const int j0 = s_slot_ptr[s], j1 = s_slot_ptr[s + 1];
                    if (j0 == j1) continue;
                    const int ts = (s < st_base) ? s : 2 * (MAXORD + 1) + (s - st_base);
                    const double sc = s_scale[s];
                    double W[RB];
#pragma unroll
                    for (int rb = 0; rb < RB; ++rb)
                        W[rb] = valid[r0 + rb] * sc * (Sfull[rb] * hx[rb] * tmp[rb][ts] - ratio[rb] * base[rb][ts]);
                    for (int jj = j0; jj < j1; ++jj) {
                        const int j = s_slot_term[jj];
                        const bool has_outer = s_out_ptr[j] != s_out_ptr[j + 1];
                        double v = 0.0;
#pragma unroll
                        for (int rb = 0; rb < RB; ++rb)
                            v = fma(has_outer ? outer_product(P, s_out_ptr, s_out_fac, j, Xt, ld, idx[r0 + rb]) : 1.0, W[rb], v);
                        v = warp_sum(v);
                        if (lane == 0) gslot[P.m_non + j] += v;
                    }
                }
            }
        }

        if (!GRAD) {
#pragma unroll
            for (int r = 0; r < R_OBJ; ++r)
                if (valid[r] != 0.0) a.S_out[idx[r]] = S[r];
        } else if (pass == 0) {
            // ---------------- phase C ----------------
            // constants / special terms / multivariate terms per row group; dense groups per chunk below
            nonmon_generic_sweep<true, HERME>(P, Xt, ld, idx, acoef, S, gslot, lane);
#pragma unroll
            for (int r = 0; r < R_OBJ; ++r)
                if (row0 + r < chunk_hi) s_S[(row0 + r - chunk_lo) * T_OBJ + tid] = S[r];
        }
    }
    }
    if (GRAD && !gm)
        dense_grad_chunk_smem<HERME, 3, RC_SWEEP>(P, DS, Xt, ld, chunk_lo, chunk_hi, N, T_OBJ, tid, s_S, gslot, lane);
    }

    if (!GRAD) return;

    // ---- block partial -> global; last block reduces over blocks in fixed order ----
    Jacc = warp_sum(Jacc);
    if (lane == 0) gslot[-1] = Jacc;
    __syncthreads();
    double* part = a.partials + (int64_t)blockIdx.x * (1 + m);
    for (int j = tid; j < 1 + m; j += T_OBJ) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < NW; ++w) v += s_gacc[w * (1 + m) + j];
        part[j] = v;
    }
    __threadfence();
    __shared__ unsigned int s_last;
    __syncthreads();
    if (tid == 0) s_last = (atomicAdd(a.counter, 1u) == gridDim.x - 1) ? 1u : 0u;
    __syncthreads();
    if (s_last) {
        __threadfence();
        const double invN = 1.0 / (double)N;
        for (int j = tid; j < 1 + m; j += T_OBJ) {
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

// One compiled instantiation: its template arguments and resident blocks per SM (BPS)
template <int MAXORD_, bool HAS_PLAIN_, bool HAS_HF_, int NST_, bool HERME_, bool EXPRECT_, int RB_, int NQ_, int BPS_>
struct ObjCfg {
    static constexpr int MAXORD = MAXORD_, NST = NST_, RB = RB_, NQ = NQ_, BPS = BPS_;
    static constexpr bool HAS_PLAIN = HAS_PLAIN_, HAS_HF = HAS_HF_, HERME = HERME_, EXPRECT = EXPRECT_;
    // the instantiation can compute the component: within its orders and special terms, and of its family and rectifier
    static bool covers(const PlanView& P, int rect) {
        return P.maxord <= MAXORD && P.nst <= NST && (HAS_PLAIN || !P.has_plain) && (HAS_HF || !P.has_hf) &&
               (!HERME || P.family == FAM_HERMITE_E) && (!EXPRECT || rect == RECT_EXP);
    }
};

//                   MAXORD  PLAIN  HF    NST  HERME  EXPRECT  RB  NQ  BPS
using Cfg1 = ObjCfg<3,       true,  true, 0,   true,  true,    2,  1,  4>;
using Cfg2 = ObjCfg<6,       true,  true, 0,   true,  true,    2,  1,  3>;
using Cfg3 = ObjCfg<12,      true,  true, 0,   true,  true,    1,  1,  3>;
using Cfg4 = ObjCfg<6,       true,  true, 0,   false, false,   2,  1,  3>;
using Cfg5 = ObjCfg<20,      true,  true, 8,   false, false,   1,  1,  2>;
// hot instantiation (RB = 2 samples x NQ = 2 nodes in flight per thread); reached only when the tile kernel does not
// cover the plan (special / multivariate nonmonotone terms, nonmonotone order > 3)
using Cfg6 = ObjCfg<3,       false, true, 0,   true,  true,    2,  2,  4>;

template <class C>
cudaError_t launch_cfg(const ObjArgs& a, bool grad, int sm_count, cudaStream_t st) {
    const int64_t rows = (a.N + T_OBJ - 1) / T_OBJ;
    int64_t grid = (int64_t)sm_count * (a.blocks_per_sm > 0 ? a.blocks_per_sm : C::BPS);
    if (grid > rows) grid = rows;
    if (grid > a.max_grid) grid = a.max_grid;
    if (grid < 1) grid = 1;
    ObjArgs b = a;
    const Layout L = make_layout(a.P, a.Q, C::MAXORD, C::NQ, grad, a.gram_mode != 0, a.ch_rows);
    *reinterpret_cast<Layout*>(b.lay) = L;
    const size_t smem = sizeof(double) * (size_t)L.total;
    auto k = grad ? objgrad_kernel<C::MAXORD, C::HAS_PLAIN, C::HAS_HF, C::NST, C::HERME, C::EXPRECT, true, C::RB, C::NQ>
                  : objgrad_kernel<C::MAXORD, C::HAS_PLAIN, C::HAS_HF, C::NST, C::HERME, C::EXPRECT, false, C::RB, C::NQ>;
    cudaError_t e;
    if (smem > 48 * 1024 && (e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
    k<<<(int)grid, T_OBJ, smem, st>>>(b);
    return cudaGetLastError();
}

// each instantiation is compiled by its own translation unit, ttm_objgrad_cfg<N>.cu
extern template cudaError_t launch_cfg<Cfg1>(const ObjArgs&, bool, int, cudaStream_t);
extern template cudaError_t launch_cfg<Cfg2>(const ObjArgs&, bool, int, cudaStream_t);
extern template cudaError_t launch_cfg<Cfg3>(const ObjArgs&, bool, int, cudaStream_t);
extern template cudaError_t launch_cfg<Cfg4>(const ObjArgs&, bool, int, cudaStream_t);
extern template cudaError_t launch_cfg<Cfg5>(const ObjArgs&, bool, int, cudaStream_t);
extern template cudaError_t launch_cfg<Cfg6>(const ObjArgs&, bool, int, cudaStream_t);

}  // namespace ttm_obj
