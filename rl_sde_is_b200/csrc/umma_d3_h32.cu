// tcgen05 forward rollout kernels for d = 3, hidden width = 32 (resident weights)
#include "rollout_umma_inst.cuh"
RLSDE_INSTANTIATE_UMMA(3, 32, false)
