// forward rollout into the ragged checkpoint store (rlsde_rollout_fwd_ragged) for d = 4, hidden width = 32: the
// tcgen05 kernel
#include "rollout_umma_inst.cuh"
RLSDE_INSTANTIATE_UMMA(4, 32, true)
