// weighted reverse-pass kernels (rlsde_rollout_bwd_weighted) for d = 2, hidden width = 32: the thread-per-trajectory
// CUDA-core family (a translation unit of its own, like every weighted instantiation: the unweighted kernels keep their code)
#include "rollout_bwd_inst.cuh"
RLSDE_INSTANTIATE_BWD(2, 32, true, false)
