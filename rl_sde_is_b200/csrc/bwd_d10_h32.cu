// reverse-pass kernels for d = 10, hidden width = 32 (precise and fast tanh)
#include "rollout_bwd_inst.cuh"
RLSDE_INSTANTIATE_BWD(10, 32, false, false)
