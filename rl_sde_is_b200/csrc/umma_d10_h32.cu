// tcgen05 forward rollout kernels for d = 10, hidden width = 32 (resident weights)
#include "rollout_umma_inst.cuh"
RLSDE_INSTANTIATE_UMMA(10, 32, false)
