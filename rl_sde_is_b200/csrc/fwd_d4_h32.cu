// forward rollout kernels for d = 4, hidden width = 32 (all precision / tanh variants)
#include "rollout_fwd_inst.cuh"
RLSDE_INSTANTIATE_FWD(4, 32, false)
