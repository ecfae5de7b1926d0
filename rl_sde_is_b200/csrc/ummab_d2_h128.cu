// tcgen05 reverse pass (producer / consumer CTAs, dW2 in tensor memory) for d = 2, hidden width = 128
#include "rollout_umma_bwd_inst.cuh"
RLSDE_INSTANTIATE_UMMA_BWD_SCRATCH(2, 128)
RLSDE_INSTANTIATE_UMMA_BWD(2, 128, false, false)
