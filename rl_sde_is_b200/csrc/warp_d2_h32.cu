// warp-per-trajectory (small-batch, latency-oriented) rollout kernels for d = 2, hidden width = 32
#include "rollout_warp_inst.cuh"
RLSDE_INSTANTIATE_FWD_WARP(2, false)
RLSDE_INSTANTIATE_BWD_WARP(2, false, false)
RLSDE_INSTANTIATE_PACK_DEV(2)
