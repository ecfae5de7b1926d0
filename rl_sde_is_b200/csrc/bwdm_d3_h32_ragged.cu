// weighted reverse pass over the ragged checkpoint store (rlsde_rollout_bwd_ragged) for d = 3, hidden width = 32: the
// tensor-core thread-per-trajectory family and the warp-per-trajectory kernel
#include "rollout_bwd_mma_inst.cuh"
#include "rollout_warp_inst.cuh"
RLSDE_INSTANTIATE_BWD_MMA(3, true, true)
RLSDE_INSTANTIATE_BWD_WARP(3, true, true)
