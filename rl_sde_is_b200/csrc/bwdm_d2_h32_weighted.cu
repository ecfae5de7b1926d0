// weighted reverse-pass kernels (rlsde_rollout_bwd_weighted) for d = 2, hidden width = 32: the tensor-core
// thread-per-trajectory family and the warp-per-trajectory kernel
#include "rollout_bwd_mma_inst.cuh"
#include "rollout_warp_inst.cuh"
RLSDE_INSTANTIATE_BWD_MMA(2, true, false)
RLSDE_INSTANTIATE_BWD_WARP(2, true, false)
