// instantiation 1 of the K-objgrad kernel template (see ttm_objgrad_impl.cuh)
#include "ttm_objgrad_impl.cuh"

template cudaError_t ttm_obj::launch_cfg<ttm_obj::Cfg1>(const ObjArgs&, bool, int, cudaStream_t);
