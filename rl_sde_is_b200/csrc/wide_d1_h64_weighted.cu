// weighted reverse-pass kernels (rlsde_rollout_bwd_weighted) for d = 1, hidden width = 64: the wide-policy tile kernel
#include "rollout_wide_inst.cuh"
RLSDE_INSTANTIATE_BWD_WIDE(1, 64, true, false)
