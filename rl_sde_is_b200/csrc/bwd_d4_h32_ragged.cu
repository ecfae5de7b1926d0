// weighted reverse pass over the ragged checkpoint store (rlsde_rollout_bwd_ragged) for d = 4, hidden width = 32: the
// thread-per-trajectory CUDA-core family
#include "rollout_bwd_inst.cuh"
RLSDE_INSTANTIATE_BWD(4, 32, true, true)
