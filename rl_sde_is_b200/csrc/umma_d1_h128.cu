// tcgen05 forward rollout kernels (tensor-memory accumulator, streamed float16 hi/lo weights) for d = 1, hidden width = 128
#include "rollout_umma_inst.cuh"
RLSDE_INSTANTIATE_UMMA(1, 128, false)
