// Dispatcher of K-objgrad / K-S: picks the narrowest compiled instantiation that covers the
// component's slot structure (see ttm_objgrad_impl.cuh for the kernel).
#include "ttm_objgrad_impl.cuh"

// Returns cudaErrorInvalidValue if the plan exceeds the compiled limits (order > 20 or > 8
// special-term inner factors).
cudaError_t ttm_launch_objgrad(const ObjArgs& a_in, bool grad, int sm_count, cudaStream_t st) {
    using namespace ttm_obj;
    ObjArgs a = a_in;
    const PlanView& P = a.P;
    if (!grad) a.gram_mode = 0;
    // tile kernel first (ttm_objgrad_tile.cu) when the plan is in its class (a.tile_ok, see ttm_ctx_set_objgrad_kernel)
    {
        const cudaError_t e = ttm_launch_objgrad_tile(a, grad, sm_count, st);
        if (e != cudaErrorNotSupported) return e;
    }
    if (a.gram_mode && P.dense_maxord > 3) return cudaErrorInvalidValue;   // merged sweep handles orders <= 3
    a.ch_rows = a.gram_mode ? 2 * RC_SWEEP : CH_ROWS;
    if (Cfg6::covers(P, a.rect)) return launch_cfg<Cfg6>(a, grad, sm_count, st);
    a.blocks_per_sm = 0;   // the context's blocks-per-SM setting applies to the hot instantiation only
    if (Cfg1::covers(P, a.rect)) return launch_cfg<Cfg1>(a, grad, sm_count, st);
    if (Cfg2::covers(P, a.rect)) return launch_cfg<Cfg2>(a, grad, sm_count, st);
    if (Cfg3::covers(P, a.rect)) return launch_cfg<Cfg3>(a, grad, sm_count, st);
    if (Cfg4::covers(P, a.rect)) return launch_cfg<Cfg4>(a, grad, sm_count, st);
    if (Cfg5::covers(P, a.rect)) return launch_cfg<Cfg5>(a, grad, sm_count, st);
    return cudaErrorInvalidValue;
}
