// tcgen05 reverse pass (producer / consumer CTAs, dW2 in tensor memory) for d = 1, hidden width = 256
#include "rollout_umma_bwd_inst.cuh"
RLSDE_INSTANTIATE_UMMA_BWD_SCRATCH(1, 256)
RLSDE_INSTANTIATE_UMMA_BWD(1, 256, false, false)
