// forward rollout into the ragged checkpoint store (rlsde_rollout_fwd_ragged) for d = 3, hidden width = 32: the
// thread-per-trajectory kernel and the warp-per-trajectory kernel, fresh and continuing K1's hand-off (a translation unit
// of its own, like every ragged instantiation: the dense-store kernels keep their code)
#include "rollout_fwd_inst.cuh"
#include "rollout_warp_inst.cuh"
RLSDE_INSTANTIATE_FWD(3, 32, true)
RLSDE_INSTANTIATE_FWD_WARP(3, true)
