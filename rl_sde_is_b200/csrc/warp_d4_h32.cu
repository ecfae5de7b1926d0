// warp-per-trajectory (small-batch, latency-oriented) rollout kernels for d = 4, hidden width = 32
#include "rollout_warp_inst.cuh"
RLSDE_INSTANTIATE_FWD_WARP(4, false)
RLSDE_INSTANTIATE_BWD_WARP(4, false, false)
RLSDE_INSTANTIATE_PACK_DEV(4)
