// C ABI of libttm (see include/ttm.h).  Thin: argument checks, device selection, workspace
// ownership, kernel launches.  No torch types, no exceptions across the boundary.

#include <cuda_runtime.h>

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/ttm.h"
#include "ttm_kernels.h"

namespace {
thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
int cuda_fail(cudaError_t e, const char* where) {
    g_err = std::string(where) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
    return TTM_ERR_CUDA;
}
#define CK(call)                                                     \
    do {                                                             \
        cudaError_t e_ = (call);                                     \
        if (e_ != cudaSuccess) return cuda_fail(e_, #call);          \
    } while (0)

constexpr int MAX_GRID = 160 * 8;   // rows of the per-plan partials buffer (>= resident blocks of any launch)
}  // namespace

struct ttm_ctx {
    int device = 0;
    int sm_count = 0;         // cudaDeviceProp::multiProcessorCount of `device` (ttm_ctx_create)
    int Q = 0;
    double wsum = 0.0;
    double* d_xis = nullptr;
    double* d_ws = nullptr;
    std::vector<double> h_xis, h_ws;   // host copies (kernel-parameter node table of the tile kernel)
    int rect = RECT_EXP;
    double delta = 1e-8;
    int* d_flags = nullptr;   // [0] iter_max, [1] not_converged
    int blocks_per_sm = 0;    // 0: kernel default
    int force_general = 0;    // 1: K-objgrad always through the general kernel (A/B parity runs)
    FusedComp* d_fused = nullptr;   // component table of ttm_map_fused (device) and its pinned host mirror
    FusedComp* h_fused = nullptr;
    int fused_cap = 0;
    cudaEvent_t ev_fused = nullptr;
    // descriptors of the plans that took part in a batched K-sepobj launch (device array + host registry)
    SepBatchItem* d_items = nullptr;
    int items_cap = 0;
    std::vector<ttm_plan*> items;   // slot -> plan (nullptr: free)
};

struct ttm_plan {
    ttm_ctx* ctx = nullptr;
    PlanView view{};
    int32_t* d_ib = nullptr;
    double* d_db = nullptr;
    int64_t n_int = 0, n_double = 0;
    int m = 0;
    double* d_coeffs = nullptr;    // [m]
    double* d_out = nullptr;       // [1+m]
    double* d_partials = nullptr;  // [MAX_GRID][1+m]
    unsigned int* d_counter = nullptr;
    int batch_slot = -1;           // index in ctx->items / ctx->d_items, -1: not registered
    bool batch_uploaded = false;   // descriptor in ctx->d_items is current
    double* h_pin = nullptr;       // pinned staging [2*(1+m)]
    cudaEvent_t ev_h2d = nullptr;  // recorded after every H2D copy out of h_pin: the buffer is not rewritten before it
    double* h_res = nullptr;       // pinned + mapped [1+m] result mirror written by the kernels' last block, then
    unsigned long long* h_flag = nullptr;   // the launch's sequence number (after a system fence)
    unsigned long long seq = 0;
    int gram_mode = 0;
    int tile_ok = 0, dense_mask = 0, n_out_terms = 0;   // tile-kernel eligibility (parse_view)
};

extern "C" {

const char* ttm_last_error(void) { return g_err.c_str(); }
int ttm_version(void) { return 100; }

int ttm_host_is_pinned(const void* host_ptr, int* host_out) {
    if (!host_ptr || !host_out) return fail(TTM_ERR_ARG, "ttm_host_is_pinned: null argument");
    cudaPointerAttributes at;
    cudaError_t e = cudaPointerGetAttributes(&at, host_ptr);
    if (e != cudaSuccess) { cudaGetLastError(); *host_out = 0; return TTM_OK; }   // ordinary pageable memory
    *host_out = (at.type == cudaMemoryTypeHost) ? 1 : 0;
    return TTM_OK;
}

int ttm_device_sm_count(int device, int* host_sm_count) {
    cudaDeviceProp p;
    CK(cudaGetDeviceProperties(&p, device));
    *host_sm_count = p.multiProcessorCount;
    return TTM_OK;
}

int ttm_ctx_create(int device, ttm_ctx** host_out) {
    if (!host_out) return fail(TTM_ERR_ARG, "ttm_ctx_create: null output");
    CK(cudaSetDevice(device));
    cudaDeviceProp p;
    CK(cudaGetDeviceProperties(&p, device));
    int* d_flags = nullptr;
    CK(cudaMalloc(&d_flags, 2 * sizeof(int)));
    cudaError_t e0 = cudaMemset(d_flags, 0, 2 * sizeof(int));
    if (e0 != cudaSuccess) { cudaFree(d_flags); return cuda_fail(e0, "cudaMemset"); }
    auto* c = new ttm_ctx();
    c->device = device;
    c->sm_count = p.multiProcessorCount;
    c->d_flags = d_flags;
    *host_out = c;
    return TTM_OK;
}

int ttm_ctx_destroy(ttm_ctx* c) {
    if (!c) return TTM_OK;
    cudaSetDevice(c->device);
    cudaFree(c->d_xis);
    cudaFree(c->d_ws);
    cudaFree(c->d_flags);
    cudaFree(c->d_fused);
    if (c->h_fused) cudaFreeHost(c->h_fused);
    if (c->ev_fused) cudaEventDestroy(c->ev_fused);
    cudaFree(c->d_items);
    delete c;
    return TTM_OK;
}

int ttm_ctx_set_quadrature(ttm_ctx* c, const double* host_xis, const double* host_ws, int Q) {
    if (!c || !host_xis || !host_ws || Q <= 0) return fail(TTM_ERR_ARG, "ttm_ctx_set_quadrature: bad arguments");
    CK(cudaSetDevice(c->device));
    cudaFree(c->d_xis);
    cudaFree(c->d_ws);
    CK(cudaMalloc(&c->d_xis, Q * sizeof(double)));
    CK(cudaMalloc(&c->d_ws, Q * sizeof(double)));
    CK(cudaMemcpy(c->d_xis, host_xis, Q * sizeof(double), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(c->d_ws, host_ws, Q * sizeof(double), cudaMemcpyHostToDevice));
    c->Q = Q;
    c->h_xis.assign(host_xis, host_xis + Q);
    c->h_ws.assign(host_ws, host_ws + Q);
    double s = 0.0;
    for (int q = 0; q < Q; ++q) s += host_ws[q];
    c->wsum = s;
    return TTM_OK;
}

int ttm_ctx_set_blocks_per_sm(ttm_ctx* c, int blocks_per_sm) {
    if (!c || blocks_per_sm < 0 || blocks_per_sm > 8) return fail(TTM_ERR_ARG, "ttm_ctx_set_blocks_per_sm: bad arguments");
    c->blocks_per_sm = blocks_per_sm;
    return TTM_OK;
}

int ttm_ctx_set_objgrad_kernel(ttm_ctx* c, int mode) {
    if (!c || mode < 0 || mode > 1) return fail(TTM_ERR_ARG, "ttm_ctx_set_objgrad_kernel: bad arguments");
    c->force_general = mode;
    return TTM_OK;
}

int ttm_ctx_set_rectifier(ttm_ctx* c, int rect, double delta) {
    if (!c || rect < 0 || rect > RECT_ELU) return fail(TTM_ERR_ARG, "ttm_ctx_set_rectifier: bad arguments");
    c->rect = rect;
    c->delta = delta;
    return TTM_OK;
}

static int parse_view(ttm_plan* p, const int32_t* h) {
    if (p->n_int < H_SIZE || h[H_MAGIC] != TTM_PLAN_MAGIC) return fail(TTM_ERR_ARG, "ttm_plan_create: bad plan blob");
    PlanView& v = p->view;
    v.ib = p->d_ib;
    v.db = p->d_db;
    v.dtot = h[H_DTOT]; v.c = h[H_C]; v.family = h[H_FAMILY]; v.nfac = h[H_NFAC];
    v.m_non = h[H_M_NON]; v.m_mon = h[H_M_MON]; v.m_dmon = h[H_M_DMON];
    v.nconst = h[H_NCONST]; v.nvars = h[H_NVARS]; v.nmulti = h[H_NMULTI];
    v.maxord = h[H_MAXORD]; v.has_plain = h[H_HAS_PLAIN]; v.has_hf = h[H_HAS_HF]; v.nst = h[H_NST];
    v.nslot = h[H_NSLOT];
    v.o_fac_i = h[H_FAC_I];
    v.o_non_ptr = h[H_NON_PTR]; v.o_non_fac = h[H_NON_FAC];
    v.o_mon_ptr = h[H_MON_PTR]; v.o_mon_fac = h[H_MON_FAC];
    v.o_dmon_ptr = h[H_DMON_PTR]; v.o_dmon_fac = h[H_DMON_FAC];
    v.o_const_idx = h[H_CONST_IDX]; v.o_var_idx = h[H_VAR_IDX]; v.o_var_ptr = h[H_VAR_PTR];
    v.o_ent_i = h[H_ENT_I]; v.o_multi_idx = h[H_MULTI_IDX];
    v.o_slot_ptr = h[H_SLOT_PTR]; v.o_slot_term = h[H_SLOT_TERM];
    v.o_out_ptr = h[H_OUT_PTR]; v.o_out_fac = h[H_OUT_FAC]; v.o_st_fac = h[H_ST_FAC];
    v.ndense = h[H_NDENSE]; v.dense_maxord = h[H_DENSE_MAXORD]; v.nactive = h[H_NACTIVE]; v.n_outfac = h[H_NOUTFAC];
    v.o_dense_var = h[H_DENSE_VAR]; v.o_dense_idx = h[H_DENSE_IDX]; v.o_d_dense_scale = h[H_D_DENSE_SCALE];
    v.o_d_fac = h[H_D_FAC]; v.o_d_ent = h[H_D_ENT]; v.o_d_slot_scale = h[H_D_SLOT_SCALE]; v.o_d_rec = h[H_D_REC];
    // alignment of the vector-loaded records
    if ((v.o_fac_i & 3) || (v.o_ent_i & 3) || (v.o_var_idx & 1) || (v.o_dense_var & 3) || (v.o_d_fac & 3) || (v.o_d_ent & 3))
        return fail(TTM_ERR_ARG, "ttm_plan_create: misaligned record offsets");
    if (v.nslot != 2 * (v.maxord + 1) + v.nst) return fail(TTM_ERR_ARG, "ttm_plan_create: inconsistent slot count");
    // ---- class of the tile kernel (ttm_objgrad_tile.cu): Hermite-function slots of order 1..3 of x_c, nonmonotone
    // terms = constants + dense per-variable groups of order <= 3
    p->n_out_terms = 0;
    for (int j = 0; j < v.m_mon; ++j) p->n_out_terms += (h[v.o_out_ptr + j] != h[v.o_out_ptr + j + 1]);
    p->dense_mask = 0;
    const int dstride = 2 * (v.dense_maxord + 1);
    for (int e = 0; e < v.ndense * dstride; ++e)
        if (h[v.o_dense_idx + e] >= 0) p->dense_mask |= 1 << ((e % dstride) & 31);
    bool ok = v.family == FAM_HERMITE_E && v.nst == 0 && !v.has_plain && v.has_hf && v.maxord >= 1 && v.maxord <= 3 &&
              v.nvars == 0 && v.nmulti == 0 && v.dense_maxord <= 3 && v.m_mon >= 1 && v.m_mon <= TTM_TILE_MAXMON &&
              p->n_out_terms <= TTM_TILE_MAXOUT && (p->dense_mask & 3) == 0;
    for (int s = 0; ok && s < v.nslot; ++s)
        if (h[v.o_slot_ptr + s] != h[v.o_slot_ptr + s + 1] && !((s & 1) && s >= 3)) ok = false;
    p->tile_ok = ok ? 1 : 0;
    return TTM_OK;
}

int ttm_plan_create(ttm_ctx* c, const int32_t* host_iblob, int64_t n_int, const double* host_dblob, int64_t n_double,
                    ttm_plan** host_out) {
    if (!c || !host_iblob || !host_dblob || !host_out) return fail(TTM_ERR_ARG, "ttm_plan_create: null argument");
    CK(cudaSetDevice(c->device));
    auto* p = new ttm_plan();
    p->ctx = c;
    // from here on a failing CUDA call frees the partially built plan
#undef CK
#define CK(call)                                                     \
    do {                                                             \
        cudaError_t e_ = (call);                                     \
        if (e_ != cudaSuccess) { ttm_plan_destroy(p); return cuda_fail(e_, #call); } \
    } while (0)
    p->n_int = n_int;
    p->n_double = n_double;
    CK(cudaMalloc(&p->d_ib, (n_int + 4) * sizeof(int32_t)));
    CK(cudaMalloc(&p->d_db, (n_double + 4) * sizeof(double)));
    CK(cudaMemcpy(p->d_ib, host_iblob, n_int * sizeof(int32_t), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(p->d_db, host_dblob, n_double * sizeof(double), cudaMemcpyHostToDevice));
    int rc = parse_view(p, host_iblob);
    if (rc != TTM_OK) { ttm_plan_destroy(p); return rc; }
    p->m = p->view.m_non + p->view.m_mon;
    const int m1 = 1 + p->m;
    CK(cudaMalloc(&p->d_coeffs, (p->m + 1) * sizeof(double)));
    CK(cudaMalloc(&p->d_out, m1 * sizeof(double)));
    CK(cudaMalloc(&p->d_partials, (size_t)MAX_GRID * m1 * sizeof(double)));
    CK(cudaMalloc(&p->d_counter, sizeof(unsigned int)));
    CK(cudaMemset(p->d_counter, 0, sizeof(unsigned int)));
    CK(cudaMemset(p->d_coeffs, 0, (p->m + 1) * sizeof(double)));
    CK(cudaMallocHost(&p->h_pin, 2 * m1 * sizeof(double)));
    CK(cudaEventCreateWithFlags(&p->ev_h2d, cudaEventDisableTiming));
    CK(cudaHostAlloc(&p->h_res, (m1 + 2) * sizeof(double), cudaHostAllocMapped | cudaHostAllocPortable));
    p->h_flag = reinterpret_cast<unsigned long long*>(p->h_res + m1 + 1);
    *p->h_flag = 0ull;
    *host_out = p;
    return TTM_OK;
#undef CK
#define CK(call)                                                     \
    do {                                                             \
        cudaError_t e_ = (call);                                     \
        if (e_ != cudaSuccess) return cuda_fail(e_, #call);          \
    } while (0)
}

int ttm_plan_info(ttm_plan* p, int* host_info) {
    if (!p || !host_info) return fail(TTM_ERR_ARG, "ttm_plan_info: null argument");
    host_info[0] = p->tile_ok;
    host_info[1] = p->dense_mask;
    host_info[2] = p->n_out_terms;
    host_info[3] = p->m;
    return TTM_OK;
}

int ttm_plan_update_doubles(ttm_plan* p, const double* host_dblob, int64_t n_double) {
    if (!p || !host_dblob || n_double != p->n_double) return fail(TTM_ERR_ARG, "ttm_plan_update_doubles: size mismatch");
    CK(cudaSetDevice(p->ctx->device));
    CK(cudaMemcpy(p->d_db, host_dblob, n_double * sizeof(double), cudaMemcpyHostToDevice));
    return TTM_OK;
}

int ttm_plan_destroy(ttm_plan* p) {
    if (!p) return TTM_OK;
    cudaSetDevice(p->ctx->device);
    if (p->batch_slot >= 0 && p->batch_slot < (int)p->ctx->items.size()) p->ctx->items[p->batch_slot] = nullptr;
    cudaFree(p->d_ib); cudaFree(p->d_db); cudaFree(p->d_coeffs); cudaFree(p->d_out);
    cudaFree(p->d_partials); cudaFree(p->d_counter);
    if (p->h_pin) cudaFreeHost(p->h_pin);
    if (p->ev_h2d) cudaEventDestroy(p->ev_h2d);
    if (p->h_res) cudaFreeHost(p->h_res);
    delete p;
    return TTM_OK;
}

static bool known_dtype(int dtype) { return dtype == TTM_DTYPE_F64 || dtype == TTM_DTYPE_F32; }

int ttm_colstats_ld(ttm_ctx* c, const void* X, int dtype, int64_t ldx, int64_t N, int D, double* mean, double* sd,
                    double* scratch, void* stream) {
    if (!c || !X || N <= 0 || D <= 0 || ldx < D || !known_dtype(dtype))
        return fail(TTM_ERR_ARG, "ttm_colstats_ld: bad arguments");
    CK(cudaSetDevice(c->device));
    CK(ttm_launch_colstats(X, dtype, ldx, N, D, mean, sd, scratch, c->sm_count, (cudaStream_t)stream));
    return TTM_OK;
}

int ttm_colstats(ttm_ctx* c, const double* X, int64_t N, int D, double* mean, double* sd, double* scratch, void* stream) {
    return ttm_colstats_ld(c, X, TTM_DTYPE_F64, D, N, D, mean, sd, scratch, stream);
}

int ttm_standardize_transpose_ld(ttm_ctx* c, const void* X, int dtype, int64_t ldx, int64_t N, int D, const double* mean,
                                 const double* sd, double* Xt, int64_t ld, void* stream) {
    if (!c || !X || !Xt || N <= 0 || D <= 0 || ld < N || ldx < D || !known_dtype(dtype))
        return fail(TTM_ERR_ARG, "ttm_standardize_transpose_ld: bad arguments");
    CK(cudaSetDevice(c->device));
    CK(ttm_launch_standardize_transpose(X, dtype, ldx, N, D, mean, sd, Xt, ld, (cudaStream_t)stream));
    return TTM_OK;
}

int ttm_standardize_transpose(ttm_ctx* c, const double* X, int64_t N, int D, const double* mean, const double* sd,
                              double* Xt, int64_t ld, void* stream) {
    return ttm_standardize_transpose_ld(c, X, TTM_DTYPE_F64, D, N, D, mean, sd, Xt, ld, stream);
}

int ttm_transpose_back(ttm_ctx* c, const double* Xt, int64_t ld, int64_t N, int D, const double* mean, const double* sd,
                       double* X, int64_t ldx, void* stream) {
    if (!c || !X || !Xt || N <= 0 || D <= 0 || ld < N || ldx < D) return fail(TTM_ERR_ARG, "ttm_transpose_back: bad arguments");
    CK(cudaSetDevice(c->device));
    CK(ttm_launch_transpose_back(Xt, ld, N, D, mean, sd, X, ldx, 0, (cudaStream_t)stream));
    return TTM_OK;
}

int ttm_basis_eval(ttm_plan* p, int which, const double* Xt, int64_t ld, int64_t N, double* Psi, void* stream) {
    if (!p || !Xt || !Psi || which < 0 || which > 2) return fail(TTM_ERR_ARG, "ttm_basis_eval: bad arguments");
    CK(cudaSetDevice(p->ctx->device));
    CK(ttm_launch_basis(p->view, which, Xt, ld, N, Psi, (cudaStream_t)stream));
    return TTM_OK;
}

int ttm_plan_set_gram_mode(ttm_plan* p, int on) {
    if (!p) return fail(TTM_ERR_ARG, "ttm_plan_set_gram_mode: null plan");
    if (on && p->view.dense_maxord > 3)
        return fail(TTM_ERR_LIMIT, "ttm_plan_set_gram_mode: nonmonotone polynomial order > 3 needs the two-sweep kernel");
    p->gram_mode = on ? 1 : 0;
    return TTM_OK;
}

int ttm_plan_set_coeffs(ttm_plan* p, const double* host_coeffs, void* stream) {
    if (!p || !host_coeffs) return fail(TTM_ERR_ARG, "ttm_plan_set_coeffs: null argument");
    if (p->m == 0) return TTM_OK;
    CK(cudaSetDevice(p->ctx->device));
    CK(cudaEventSynchronize(p->ev_h2d));          // the previous copy out of h_pin has been consumed
    std::memcpy(p->h_pin, host_coeffs, p->m * sizeof(double));
    CK(cudaMemcpyAsync(p->d_coeffs, p->h_pin, p->m * sizeof(double), cudaMemcpyHostToDevice, (cudaStream_t)stream));
    CK(cudaEventRecord(p->ev_h2d, (cudaStream_t)stream));
    return TTM_OK;
}

static int fill_obj(ttm_plan* p, const double* Xt, int64_t ld, int64_t N, ObjArgs& a) {
    ttm_ctx* c = p->ctx;
    if (c->Q <= 0) return fail(TTM_ERR_ARG, "quadrature rule not set (ttm_ctx_set_quadrature)");
    if (!Xt || N <= 0 || ld < N) return fail(TTM_ERR_ARG, "bad sample matrix");
    a.P = p->view;
    a.Xt = Xt; a.ld = ld; a.N = N;
    a.coeffs = p->d_coeffs;
    a.xis = c->d_xis; a.ws = c->d_ws; a.Q = c->Q; a.wsum = c->wsum;
    a.rect = c->rect; a.delta = c->delta;
    a.partials = p->d_partials; a.counter = p->d_counter; a.out = p->d_out;
    a.out_host = p->h_res; a.flag_host = p->h_flag; a.seq = ++p->seq;
    a.S_out = nullptr;
    a.max_grid = MAX_GRID;
    a.blocks_per_sm = c->blocks_per_sm;
    a.gram_mode = p->gram_mode;
    a.ch_rows = 0;
    a.h_xis = c->h_xis.data(); a.h_ws = c->h_ws.data();
    a.tile_ok = (p->tile_ok && !c->force_general) ? 1 : 0; a.dense_mask = p->dense_mask; a.n_out_terms = p->n_out_terms;
    return TTM_OK;
}

int ttm_objgrad_ir_launch(ttm_plan* p, const double* Xt, int64_t ld, int64_t N, void* stream) {
    if (!p) return fail(TTM_ERR_ARG, "ttm_objgrad_ir_launch: null plan");
    CK(cudaSetDevice(p->ctx->device));
    ObjArgs a;
    int rc = fill_obj(p, Xt, ld, N, a);
    if (rc) return rc;
    cudaError_t e = ttm_launch_objgrad(a, true, p->ctx->sm_count, (cudaStream_t)stream);
    if (e == cudaErrorInvalidValue) return fail(TTM_ERR_LIMIT, "ttm_objgrad_ir: component exceeds compiled limits (polynomial order <= 20, <= 8 special inner terms)");
    CK(e);
    return TTM_OK;
}

int ttm_plan_get_out(ttm_plan* p, double* host_out, int n, void* stream) {
    if (!p || !host_out || n < 0 || n > 1 + p->m) return fail(TTM_ERR_ARG, "ttm_plan_get_out: bad arguments");
    CK(cudaSetDevice(p->ctx->device));
    double* pin = p->h_pin + (1 + p->m);
    CK(cudaMemcpyAsync(pin, p->d_out, n * sizeof(double), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CK(cudaStreamSynchronize((cudaStream_t)stream));
    std::memcpy(host_out, pin, n * sizeof(double));
    return TTM_OK;
}

// Wait for the launch with sequence number p->seq to publish its result in the mapped host mirror, then copy it out.
// A spinning read of pinned memory replaces cudaMemcpyAsync(D2H) + cudaStreamSynchronize (~15 us per evaluation,
// which matters for the latency-bound small-N fits); errors are picked up by polling the stream every so often.
static int wait_result(ttm_plan* p, double* host_out, int n, cudaStream_t st) {
    volatile unsigned long long* flag = p->h_flag;
    const unsigned long long want = p->seq;
    for (unsigned long long spins = 0; *flag != want; ++spins) {
        if ((spins & 0xffff) == 0xffff) {
            cudaError_t e = cudaStreamQuery(st);
            if (e != cudaSuccess && e != cudaErrorNotReady) return cuda_fail(e, "kernel execution");
            if (e == cudaSuccess && *flag != want) {          // finished without publishing: should not happen
                CK(cudaMemcpy(host_out, p->d_out, n * sizeof(double), cudaMemcpyDeviceToHost));
                return TTM_OK;
            }
        }
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    std::memcpy(host_out, p->h_res, n * sizeof(double));
    return TTM_OK;
}

int ttm_objgrad_ir(ttm_plan* p, const double* Xt, int64_t ld, int64_t N, const double* host_coeffs, double* host_out,
                   void* stream) {
    int rc = ttm_plan_set_coeffs(p, host_coeffs, stream);
    if (rc) return rc;
    rc = ttm_objgrad_ir_launch(p, Xt, ld, N, stream);
    if (rc) return rc;
    return wait_result(p, host_out, 1 + p->m, (cudaStream_t)stream);
}

int ttm_eval_s_ir(ttm_plan* p, const double* Xt, int64_t ld, int64_t N, double* S_out, void* stream) {
    if (!p || !S_out) return fail(TTM_ERR_ARG, "ttm_eval_s_ir: null argument");
    CK(cudaSetDevice(p->ctx->device));
    ObjArgs a;
    int rc = fill_obj(p, Xt, ld, N, a);
    if (rc) return rc;
    a.S_out = S_out;
    cudaError_t e = ttm_launch_objgrad(a, false, p->ctx->sm_count, (cudaStream_t)stream);
    if (e == cudaErrorInvalidValue) return fail(TTM_ERR_LIMIT, "ttm_eval_s_ir: component exceeds compiled limits (polynomial order <= 20, <= 8 special inner terms)");
    CK(e);
    return TTM_OK;
}

int ttm_sep_eval(ttm_plan* p, const double* Xt, int64_t ld, int64_t N, double* S_out, const double* Xd, int64_t ldd,
                 double* dS_out, void* stream) {
    if (!p || N <= 0 || (S_out && (!Xt || ld < N)) || (dS_out && (!Xd || ldd < N)))
        return fail(TTM_ERR_ARG, "ttm_sep_eval: bad arguments");
    CK(cudaSetDevice(p->ctx->device));
    CK(ttm_launch_sep_eval(p->view, Xt, ld, N, p->d_coeffs, S_out, Xd, ldd, dS_out, p->ctx->sm_count, (cudaStream_t)stream));
    return TTM_OK;
}

int ttm_map_rect(ttm_ctx* c, const double* Xt, int64_t ld, int64_t N, int ncomp, int rows, int ns, int first,
                 const double* Rpack, double* base, int64_t ldb, void* stream) {
    if (!c || !Xt || !Rpack || !base || N <= 0 || ld < N || ldb < N || ncomp <= 0 || rows <= 0 || first < 0)
        return fail(TTM_ERR_ARG, "ttm_map_rect: bad arguments");
    if (ns != 3 && ns != 6) return fail(TTM_ERR_ARG, "ttm_map_rect: ns must be 3 or 6");
    CK(cudaSetDevice(c->device));
    InvRectArgs r;
    r.Xw = Xt; r.ld = ld; r.N = N; r.ncomp = ncomp; r.c0 = rows; r.ns = ns; r.Rpack = Rpack; r.base = base; r.ldb = ldb;
    r.tri = first;
    CK(ttm_launch_inverse_rect(r, c->sm_count, (cudaStream_t)stream));
    return TTM_OK;
}

int ttm_sep_eval_base(ttm_plan* p, const double* Xt, int64_t ld, int64_t N, const double* base, double a0, double* S_out,
                      void* stream) {
    if (!p || !Xt || !base || !S_out || N <= 0 || ld < N) return fail(TTM_ERR_ARG, "ttm_sep_eval_base: bad arguments");
    CK(cudaSetDevice(p->ctx->device));
    CK(ttm_launch_sep_eval(p->view, Xt, ld, N, p->d_coeffs, S_out, nullptr, 0, nullptr, p->ctx->sm_count,
                           (cudaStream_t)stream, base, a0));
    return TTM_OK;
}

int ttm_density_accumulate(ttm_ctx* c, double* acc, const double* S, const double* dS, double sigma, int mode,
                           int64_t N, void* stream) {
    if (!c || !acc || !dS || (mode == 0 && !S) || N <= 0) return fail(TTM_ERR_ARG, "ttm_density_accumulate: bad arguments");
    CK(cudaSetDevice(c->device));
    CK(ttm_launch_density_acc(acc, S, dS, sigma, mode, N, (cudaStream_t)stream));
    return TTM_OK;
}

int ttm_ir_logdet_accumulate(ttm_plan* p, const double* Xt, int64_t ld, int64_t N, const double* S, double sigma,
                             int mode, double* acc, void* stream) {
    if (!p || !Xt || !acc || N <= 0 || ld < N || mode < 0 || mode > 1 || (mode == 0 && !S) || !(sigma > 0.0))
        return fail(TTM_ERR_ARG, "ttm_ir_logdet_accumulate: bad arguments");
    ttm_ctx* c = p->ctx;
    CK(cudaSetDevice(c->device));
    cudaError_t e = ttm_launch_ir_logdet(p->view, p->d_coeffs, Xt, ld, N, S, sigma, c->rect, c->delta, mode, acc,
                                         (cudaStream_t)stream);
    if (e == cudaErrorInvalidValue) return fail(TTM_ERR_LIMIT, "ttm_ir_logdet_accumulate: polynomial order > 32 or > 16 special inner terms");
    CK(e);
    return TTM_OK;
}

int ttm_density_finish(ttm_ctx* c, const double* acc, const double* log_target, double* out, int64_t N, void* stream) {
    if (!c || !acc || !out || N <= 0) return fail(TTM_ERR_ARG, "ttm_density_finish: bad arguments");
    CK(cudaSetDevice(c->device));
    CK(ttm_launch_density_finish(acc, log_target, out, N, (cudaStream_t)stream));
    return TTM_OK;
}

int ttm_map_fused_ld(ttm_ctx* c, ttm_plan* const* host_plans, int D, const double* host_sigma, const void* X, int dtype,
                     int64_t ldx, int64_t n, int Dtot, const double* mean, const double* sd, const double* log_target,
                     int mode, double* Z, double* out, void* stream) {
    if (!c || !host_plans || D <= 0 || !X || n <= 0 || Dtot <= 0 || mode < 0 || mode > 4 || (mode != 2 && (!out || !host_sigma)) ||
        (mode == 2 && !Z) || ((mean == nullptr) != (sd == nullptr)) || ldx < Dtot || !known_dtype(dtype))
        return fail(TTM_ERR_ARG, "ttm_map_fused: bad arguments");
    CK(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (D > c->fused_cap) {
        cudaFree(c->d_fused);
        if (c->h_fused) cudaFreeHost(c->h_fused);
        c->d_fused = nullptr; c->h_fused = nullptr; c->fused_cap = 0;
        CK(cudaMalloc(&c->d_fused, D * sizeof(FusedComp)));
        CK(cudaMallocHost(&c->h_fused, D * sizeof(FusedComp)));
        if (!c->ev_fused) CK(cudaEventCreateWithFlags(&c->ev_fused, cudaEventDisableTiming));
        c->fused_cap = D;
    }
    CK(cudaEventSynchronize(c->ev_fused));                       // previous upload out of h_fused consumed
    for (int k = 0; k < D; ++k) {
        if (!host_plans[k] || host_plans[k]->ctx != c) return fail(TTM_ERR_ARG, "ttm_map_fused: plan of another context");
        c->h_fused[k].P = host_plans[k]->view;
        c->h_fused[k].coeffs = host_plans[k]->d_coeffs;
        c->h_fused[k].sigma = host_sigma ? host_sigma[k] : 1.0;
    }
    CK(cudaMemcpyAsync(c->d_fused, c->h_fused, D * sizeof(FusedComp), cudaMemcpyHostToDevice, st));
    CK(cudaEventRecord(c->ev_fused, st));
    FusedMapArgs a;
    a.comps = c->d_fused; a.D = D; a.Dtot = Dtot; a.X = X; a.dtype = dtype; a.ldx = ldx; a.n = n;
    a.mean = mean; a.sd = sd; a.logt = log_target;
    a.mode = mode; a.Z = Z; a.out = out;
    cudaError_t e = ttm_launch_map_fused(a, st);
    if (e == cudaErrorInvalidValue) return fail(TTM_ERR_LIMIT, "ttm_map_fused: too many columns for one shared-memory tile");
    CK(e);
    return TTM_OK;
}

int ttm_map_fused(ttm_ctx* c, ttm_plan* const* host_plans, int D, const double* host_sigma, const double* X, int64_t n,
                  int Dtot, const double* mean, const double* sd, const double* log_target, int mode, double* Z, double* out,
                  void* stream) {
    return ttm_map_fused_ld(c, host_plans, D, host_sigma, X, TTM_DTYPE_F64, Dtot, n, Dtot, mean, sd, log_target, mode, Z,
                            out, stream);
}

int ttm_gram(ttm_plan* p, const double* Xt, int64_t ld, int64_t N, double* G, double* scratch, int64_t scratch_doubles,
             void* stream) {
    return ttm_gram_tail(p, Xt, ld, N, 0, G, scratch, scratch_doubles, stream);
}

int ttm_gram_tail(ttm_plan* p, const double* Xt, int64_t ld, int64_t N, int first_col, double* G, double* scratch,
                  int64_t scratch_doubles, void* stream) {
    if (!p || !Xt || !G || !scratch || N <= 0 || ld < N || first_col < 0 || first_col > p->m)
        return fail(TTM_ERR_ARG, "ttm_gram: bad arguments");
    CK(cudaSetDevice(p->ctx->device));
    cudaError_t e = ttm_launch_gram(p->view, Xt, ld, N, first_col, G, scratch, scratch_doubles, p->ctx->sm_count, (cudaStream_t)stream);
    if (e == cudaErrorInvalidValue) return fail(TTM_ERR_LIMIT, "ttm_gram: scratch too small or too many terms for one shared-memory tile");
    CK(e);
    return TTM_OK;
}

int ttm_sep_objgrad_launch(ttm_plan* p, const double* Xt, int64_t ld, int64_t N, const double* host_b, void* stream) {
    if (!p || !Xt || !host_b || N <= 0 || ld < N) return fail(TTM_ERR_ARG, "ttm_sep_objgrad: bad arguments");
    CK(cudaSetDevice(p->ctx->device));
    const int mm = p->view.m_dmon;
    if (mm > p->m) return fail(TTM_ERR_ARG, "ttm_sep_objgrad: inconsistent plan");
    // the coefficients are read by the kernel straight from pinned (mapped) host memory and the result comes back
    // the same way: one launch, no copies, no stream synchronisation (h_pin is free again once the result arrived;
    // callers of the split form collect every launch with ttm_sep_objgrad_wait before launching on the plan again)
    CK(cudaEventSynchronize(p->ev_h2d));
    std::memcpy(p->h_pin, host_b, mm * sizeof(double));
    double* d_b = p->d_coeffs + p->view.m_non;
    p->seq += 1;
    cudaError_t e = ttm_launch_sepobj(p->view, Xt, ld, N, p->h_pin, d_b, p->ctx->delta, p->d_partials, p->d_counter,
                                      p->d_out, p->h_res, p->h_flag, p->seq, MAX_GRID, p->ctx->sm_count,
                                      (cudaStream_t)stream);
    if (e == cudaErrorInvalidValue) return fail(TTM_ERR_LIMIT, "ttm_sep_objgrad: too many monotone terms for shared memory");
    CK(e);
    return TTM_OK;
}

int ttm_sep_objgrad_wait(ttm_plan* p, double* host_out, void* stream) {
    if (!p || !host_out) return fail(TTM_ERR_ARG, "ttm_sep_objgrad_wait: bad arguments");
    return wait_result(p, host_out, 1 + p->view.m_dmon, (cudaStream_t)stream);
}

int ttm_sep_reduced_batch(int n, ttm_plan* const* plans, const double* Xt, int64_t ld, int64_t N, double n_total,
                          const double* const* host_b, const double* const* host_A, const double* const* host_c,
                          double* const* host_fg, void* stream) {
    if (n < 0 || (n > 0 && (!plans || !host_b || !host_A || !host_c || !host_fg)) || !(n_total > 0.0))
        return fail(TTM_ERR_ARG, "ttm_sep_reduced_batch: bad arguments");
    for (int i = 0; i < n; ++i)
        if (!plans[i] || !host_b[i] || !host_A[i] || !host_c[i] || !host_fg[i])
            return fail(TTM_ERR_ARG, "ttm_sep_reduced_batch: null entry");
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < i; ++j)
            if (plans[i] == plans[j]) return fail(TTM_ERR_ARG, "ttm_sep_reduced_batch: a plan may appear once per call");
    // all launches first: ONE kernel for up to 64 components (blockIdx.y = component).  Descriptors of the plans are
    // registered in a device array on first use; per launch only the sequence numbers and the active list travel.
    ttm_ctx* c = n > 0 ? plans[0]->ctx : nullptr;
    if (n > 0) {
        CK(cudaSetDevice(c->device));
        bool grew = false;
        for (int i = 0; i < n; ++i) {
            ttm_plan* p = plans[i];
            if (p->ctx != c) return fail(TTM_ERR_ARG, "ttm_sep_reduced_batch: plans of different contexts");
            if (p->view.m_dmon > p->m) return fail(TTM_ERR_ARG, "ttm_sep_reduced_batch: inconsistent plan");
            if (p->batch_slot < 0) {
                int slot = -1;
                for (size_t q = 0; q < c->items.size(); ++q) if (!c->items[q]) { slot = (int)q; break; }
                if (slot < 0) { slot = (int)c->items.size(); c->items.push_back(nullptr); }
                c->items[slot] = p;
                p->batch_slot = slot;
                if (slot >= c->items_cap) grew = true;
            }
        }
        if (grew) {                                      // (re)allocate: every live descriptor is uploaded again
            CK(cudaStreamSynchronize((cudaStream_t)stream));
            cudaFree(c->d_items);
            c->d_items = nullptr;
            c->items_cap = (int)c->items.size() * 2 + 16;
            CK(cudaMalloc(&c->d_items, sizeof(SepBatchItem) * c->items_cap));
            for (ttm_plan* q : c->items) if (q) q->batch_uploaded = false;
        }
        for (size_t q = 0; q < c->items.size(); ++q) {
            ttm_plan* p = c->items[q];
            if (!p || p->batch_uploaded) continue;
            SepBatchItem it;
            it.P = p->view; it.b = p->h_pin; it.d_b = p->d_coeffs + p->view.m_non; it.partials = p->d_partials;
            it.counter = p->d_counter; it.out = p->d_out; it.out_host = p->h_res; it.flag_host = p->h_flag;
            CK(cudaMemcpy(c->d_items + q, &it, sizeof(it), cudaMemcpyHostToDevice));
            p->batch_uploaded = true;
        }
    }
    for (int i0 = 0; i0 < n; i0 += TTM_SEP_BATCH_MAX) {
        const int na = (n - i0 < TTM_SEP_BATCH_MAX) ? n - i0 : TTM_SEP_BATCH_MAX;
        SepBatchLaunch L;
        int max_mm = 1;
        for (int a = 0; a < na; ++a) {
            ttm_plan* p = plans[i0 + a];
            const int mm = p->view.m_dmon;
            CK(cudaEventSynchronize(p->ev_h2d));         // h_pin free (an earlier asynchronous coefficient upload)
            std::memcpy(p->h_pin, host_b[i0 + a], mm * sizeof(double));
            p->seq += 1;
            L.seq[a] = p->seq;
            L.item[a] = p->batch_slot;
            if (mm > max_mm) max_mm = mm;
        }
        cudaError_t e = ttm_launch_sepobj_batch(c->d_items, L, na, max_mm, Xt, ld, N, c->delta, MAX_GRID, c->sm_count,
                                                (cudaStream_t)stream);
        if (e == cudaErrorInvalidValue) return fail(TTM_ERR_LIMIT, "ttm_sep_reduced_batch: too many monotone terms for shared memory");
        CK(e);
    }
    for (int i = 0; i < n; ++i) {                       // then collect; the m x m algebra runs while the others finish
        ttm_plan* p = plans[i];
        const int m = p->view.m_dmon;
        double* fg = host_fg[i];
        int rc = wait_result(p, fg, 1 + m, (cudaStream_t)stream);
        if (rc) return rc;
        const double *b = host_b[i], *A = host_A[i], *cv = host_c[i];
        double quad = 0.0, lin = 0.0;
        const double sumlog = fg[0];
        for (int r = 0; r < m; ++r) {
            double ab = 0.0;
            for (int q = 0; q < m; ++q) ab += A[(size_t)r * m + q] * b[q];
            quad += b[r] * ab;
            lin += b[r] * cv[r];
            fg[1 + r] = ab - fg[1 + r] / n_total + cv[r];
        }
        fg[0] = quad / 2 - sumlog / n_total + lin;
    }
    return TTM_OK;
}

int ttm_sep_objgrad(ttm_plan* p, const double* Xt, int64_t ld, int64_t N, const double* host_b, double* host_out,
                    void* stream) {
    if (!host_out) return fail(TTM_ERR_ARG, "ttm_sep_objgrad: bad arguments");
    int rc = ttm_sep_objgrad_launch(p, Xt, ld, N, host_b, stream);
    if (rc) return rc;
    return ttm_sep_objgrad_wait(p, host_out, stream);
}

int ttm_mon_table(ttm_plan* p, int ntab, double* table, void* stream) {
    if (!p || !table || ntab < 2) return fail(TTM_ERR_ARG, "ttm_mon_table: bad arguments");
    CK(cudaSetDevice(p->ctx->device));
    CK(ttm_launch_mon_table(p->view, p->d_coeffs, ntab, table, (cudaStream_t)stream));
    return TTM_OK;
}

static void fill_inv(ttm_plan* p, double* Xt, int64_t ld, int64_t N, const double* z, InvArgs& a) {
    ttm_ctx* c = p->ctx;
    a.P = p->view;
    a.Xt = Xt; a.ld = ld; a.N = N; a.z = z;
    a.coeffs = p->d_coeffs;
    a.xis = c->d_xis; a.ws = c->d_ws; a.Q = c->Q; a.wsum = c->wsum;
    a.rect = c->rect; a.delta = c->delta;
    a.separable = 0;
    a.table = nullptr; a.ntab = 0; a.truncate = 0;
    a.first = 0; a.count = N; a.max_iter = 100;
    a.iter_max = nullptr; a.not_converged = nullptr;
}

int ttm_inverse_table(ttm_plan* p, double* Xt, int64_t ld, int64_t N, const double* z, const double* table, int ntab,
                      int truncate, void* stream) {
    if (!p || !Xt || !z || !table || ntab < 2 || N <= 0 || ld < N) return fail(TTM_ERR_ARG, "ttm_inverse_table: bad arguments");
    CK(cudaSetDevice(p->ctx->device));
    InvArgs a;
    fill_inv(p, Xt, ld, N, z, a);
    a.separable = 1;
    a.table = table; a.ntab = ntab; a.truncate = truncate;
    CK(ttm_launch_inverse_table(a, p->ctx->sm_count, (cudaStream_t)stream));
    return TTM_OK;
}

int ttm_inverse_fused_apack_size(int ncomp, int c0, int ns, int64_t* host_doubles) {
    if (ncomp <= 0 || c0 < 0 || (ns != 3 && ns != 6) || !host_doubles) return fail(TTM_ERR_ARG, "ttm_inverse_fused_apack_size: bad arguments");
    *host_doubles = (int64_t)ttm_inverse_fused_apack_doubles(ncomp, c0, ns);
    return TTM_OK;
}

static const std::string fused_ntab_limit =
    "ntab exceeds TTM_INVERSE_FUSED_MAX_NTAB = " + std::to_string(TTM_INVERSE_FUSED_MAX_NTAB) + " (tables are staged in shared memory)";

int ttm_inverse_fused(ttm_ctx* c, double* Xw, int64_t ld, int64_t N, const double* Zt, int64_t ldz, int ncomp, int c0, int ns,
                      const double* Apack, const double* a0, const double* tables, int ntab, int truncate, void* stream) {
    if (!c || !Xw || !Zt || !Apack || !a0 || !tables || N <= 0 || ld < N || ldz < N || ncomp <= 0 || c0 < 0 || ntab < 2)
        return fail(TTM_ERR_ARG, "ttm_inverse_fused: bad arguments");
    if (ns != 3 && ns != 6) return fail(TTM_ERR_ARG, "ttm_inverse_fused: ns must be 3 or 6");
    if (ntab > TTM_INVERSE_FUSED_MAX_NTAB) return fail(TTM_ERR_LIMIT, "ttm_inverse_fused: " + fused_ntab_limit);
    CK(cudaSetDevice(c->device));
    InvFusedArgs a;
    a.Xw = Xw; a.ld = ld; a.N = N; a.Zt = Zt; a.ldz = ldz; a.ncomp = ncomp; a.c0 = c0; a.ns = ns;
    a.Apack = Apack; a.a0 = a0; a.tables = tables; a.ntab = ntab; a.truncate = truncate;
    a.base = nullptr; a.ldb = 0;
    CK(ttm_launch_inverse_fused(a, c->sm_count, (cudaStream_t)stream));
    return TTM_OK;
}

int ttm_inverse_rect_rpack_size(int ncomp, int c0, int ns, int64_t* host_doubles) {
    if (ncomp <= 0 || c0 < 0 || (ns != 3 && ns != 6) || !host_doubles) return fail(TTM_ERR_ARG, "ttm_inverse_rect_rpack_size: bad arguments");
    *host_doubles = (int64_t)ttm_inverse_rect_rpack_doubles(ncomp, c0, ns);
    return TTM_OK;
}

int ttm_inverse_fused_split(ttm_ctx* c, double* Xw, int64_t ld, int64_t N, const double* Zt, int64_t ldz, int ncomp, int c0,
                            int ns, const double* Apack, const double* Rpack, const double* a0, const double* tables,
                            int ntab, int truncate, double* base, int64_t ldb, void* stream) {
    if (!c || !Xw || !Zt || !Apack || !Rpack || !a0 || !tables || !base || N <= 0 || ld < N || ldz < N || ldb < N ||
        ncomp <= 0 || c0 <= 0 || ntab < 2)
        return fail(TTM_ERR_ARG, "ttm_inverse_fused_split: bad arguments");
    if (ns != 3 && ns != 6) return fail(TTM_ERR_ARG, "ttm_inverse_fused_split: ns must be 3 or 6");
    if (ntab > TTM_INVERSE_FUSED_MAX_NTAB) return fail(TTM_ERR_LIMIT, "ttm_inverse_fused_split: " + fused_ntab_limit);
    if ((ldb & 1) || (reinterpret_cast<uintptr_t>(base) & 15))
        return fail(TTM_ERR_ARG, "ttm_inverse_fused_split: base must be 16-byte aligned with an even leading dimension");
    CK(cudaSetDevice(c->device));
    InvRectArgs r;
    r.Xw = Xw; r.ld = ld; r.N = N; r.ncomp = ncomp; r.c0 = c0; r.ns = ns; r.Rpack = Rpack; r.base = base; r.ldb = ldb;
    r.tri = -1;
    CK(ttm_launch_inverse_rect(r, c->sm_count, (cudaStream_t)stream));
    InvFusedArgs a;
    a.Xw = Xw; a.ld = ld; a.N = N; a.Zt = Zt; a.ldz = ldz; a.ncomp = ncomp; a.c0 = c0; a.ns = ns;
    a.Apack = Apack; a.a0 = a0; a.tables = tables; a.ntab = ntab; a.truncate = truncate;
    a.base = base; a.ldb = ldb;
    CK(ttm_launch_inverse_fused(a, c->sm_count, (cudaStream_t)stream));
    return TTM_OK;
}

int ttm_inverse_bisect(ttm_plan* p, double* Xt, int64_t ld, int64_t N, const double* z, int separable, int max_iter,
                       int* host_not_converged, void* stream) {
    if (!p || !Xt || !z || N <= 0 || ld < N) return fail(TTM_ERR_ARG, "ttm_inverse_bisect: bad arguments");
    ttm_ctx* c = p->ctx;
    if (!separable && c->Q <= 0) return fail(TTM_ERR_ARG, "quadrature rule not set (ttm_ctx_set_quadrature)");
    CK(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    CK(cudaMemsetAsync(c->d_flags, 0, 2 * sizeof(int), st));
    InvArgs a;
    fill_inv(p, Xt, ld, N, z, a);
    a.separable = separable;
    a.max_iter = max_iter;
    a.iter_max = c->d_flags;
    a.not_converged = c->d_flags + 1;
    // samples 1..N-1 first; sample 0 then iterates only as long as any of them did
    // (the reference's loop condition sums the remaining *indices*, tm.py:3952)
    a.first = 1; a.count = N - 1;
    cudaError_t e = ttm_launch_inverse_bisect(a, c->sm_count, st);
    if (e == cudaErrorInvalidValue) return fail(TTM_ERR_LIMIT, "ttm_inverse_bisect: polynomial order > 32 or > 16 special inner terms");
    CK(e);
    a.first = 0; a.count = 1;
    CK(ttm_launch_inverse_bisect(a, c->sm_count, st));
    if (host_not_converged) {
        CK(cudaMemcpyAsync(host_not_converged, c->d_flags + 1, sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    return TTM_OK;
}

int ttm_fp64_peak(ttm_ctx* c, double* host_tflops) {
    if (!c || !host_tflops) return fail(TTM_ERR_ARG, "ttm_fp64_peak: null argument");
    CK(cudaSetDevice(c->device));
    double* sink;
    CK(cudaMalloc(&sink, sizeof(double)));
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    const int block = 256, grid = c->sm_count * 8, iters = 1 << 16;
    CK(ttm_launch_fp64_peak(sink, 1024, grid, block, 0));
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        CK(cudaEventRecord(e0, 0));
        CK(ttm_launch_fp64_peak(sink, iters, grid, block, 0));
        CK(cudaEventRecord(e1, 0));
        CK(cudaEventSynchronize(e1));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        const double tf = 2.0 * 8.0 * (double)iters * (double)grid * block / (ms * 1e-3) / 1e12;
        if (tf > best) best = tf;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    *host_tflops = best;
    return TTM_OK;
}

}  // extern "C"
