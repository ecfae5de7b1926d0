// tcgen05 forward rollout kernels for d = 1, hidden width = 32 (resident weights)
#include "rollout_umma_inst.cuh"
RLSDE_INSTANTIATE_UMMA(1, 32, false)
