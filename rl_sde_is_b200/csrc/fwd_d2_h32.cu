// forward rollout kernels for d = 2, hidden width = 32 (all precision / tanh variants)
#include "rollout_fwd_inst.cuh"
RLSDE_INSTANTIATE_FWD(2, 32, false)
