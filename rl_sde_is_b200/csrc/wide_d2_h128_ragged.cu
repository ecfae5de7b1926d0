// the ragged checkpoint store (rlsde_rollout_fwd_ragged / rlsde_rollout_bwd_ragged) for d = 2, hidden width = 128: the
// CUDA-core tile kernels and the tcgen05 kernels
#include "rollout_wide_inst.cuh"
#include "rollout_umma_inst.cuh"
#include "rollout_umma_bwd_inst.cuh"
RLSDE_INSTANTIATE_FWD_WIDE(2, 128, true)
RLSDE_INSTANTIATE_BWD_WIDE(2, 128, true, true)
RLSDE_INSTANTIATE_UMMA(2, 128, true)
RLSDE_INSTANTIATE_UMMA_BWD(2, 128, true, true)
