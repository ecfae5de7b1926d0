// forward rollout kernels for d = 10, hidden width = 32 (all precision / tanh variants)
#include "rollout_fwd_inst.cuh"
RLSDE_INSTANTIATE_FWD(10, 32, false)
