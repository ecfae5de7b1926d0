// tcgen05 forward rollout kernels for d = 2, hidden width = 32 (resident weights)
#include "rollout_umma_inst.cuh"
RLSDE_INSTANTIATE_UMMA(2, 32, false)
