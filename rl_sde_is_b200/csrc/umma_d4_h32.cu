// tcgen05 forward rollout kernels for d = 4, hidden width = 32 (resident weights)
#include "rollout_umma_inst.cuh"
RLSDE_INSTANTIATE_UMMA(4, 32, false)
