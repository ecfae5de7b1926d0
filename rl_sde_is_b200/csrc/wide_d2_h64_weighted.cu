// weighted reverse-pass kernels (rlsde_rollout_bwd_weighted) for d = 2, hidden width = 64: the wide-policy tile kernel
#include "rollout_wide_inst.cuh"
RLSDE_INSTANTIATE_WIDE_BWD_WEIGHTED(2, 64)
