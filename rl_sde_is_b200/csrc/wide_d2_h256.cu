// wide-policy rollout kernels (tile contraction through shared memory) for d = 2, hidden width = 256
#include "rollout_wide_inst.cuh"
RLSDE_INSTANTIATE_FWD_WIDE(2, 256, false)
RLSDE_INSTANTIATE_BWD_WIDE(2, 256, false, false)
