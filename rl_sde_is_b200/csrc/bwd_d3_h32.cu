// reverse-pass kernels for d = 3, hidden width = 32 (precise and fast tanh)
#include "rollout_bwd_inst.cuh"
RLSDE_INSTANTIATE_BWD(3, 32, false, false)
