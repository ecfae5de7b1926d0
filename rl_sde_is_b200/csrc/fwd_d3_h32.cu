// forward rollout kernels for d = 3, hidden width = 32 (all precision / tanh variants)
#include "rollout_fwd_inst.cuh"
RLSDE_INSTANTIATE_FWD(3, 32, false)
