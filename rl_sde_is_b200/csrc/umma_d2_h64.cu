// tcgen05 forward rollout kernels (tensor-memory accumulator, resident float16 hi/lo weights) for d = 2, hidden width = 64
#include "rollout_umma_inst.cuh"
RLSDE_INSTANTIATE_UMMA(2, 64, false)
