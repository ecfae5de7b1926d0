// reverse-pass kernels for d = 2, hidden width = 32 (precise and fast tanh)
#include "rollout_bwd_inst.cuh"
RLSDE_INSTANTIATE_BWD(2, 32, false, false)
