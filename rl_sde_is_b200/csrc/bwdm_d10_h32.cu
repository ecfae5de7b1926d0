// tensor-core (mma.sync, float16 x 3 split) reverse-pass kernels for d = 10, hidden width = 32
#include "rollout_bwd_mma_inst.cuh"
RLSDE_INSTANTIATE_BWD_MMA(10, false, false)
