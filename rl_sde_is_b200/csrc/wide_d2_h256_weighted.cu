// weighted reverse-pass kernels (rlsde_rollout_bwd_weighted) for d = 2, hidden width = 256: the wide-policy tile kernel
// and the tcgen05 producer / consumer kernel
#include "rollout_wide_inst.cuh"
#include "rollout_umma_bwd_inst.cuh"
RLSDE_INSTANTIATE_BWD_WIDE(2, 256, true, false)
RLSDE_INSTANTIATE_UMMA_BWD(2, 256, true, false)
