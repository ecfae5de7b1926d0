// forward rollout kernels for d = 1, hidden width = 32 (all precision / tanh variants)
#include "rollout_fwd_inst.cuh"
RLSDE_INSTANTIATE_FWD(1, 32, false)
