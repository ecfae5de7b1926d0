// forward rollout kernels for d = 1, hidden width = 32 with the Brownian-bridge hit test (RLSDE_F_HIT_BRIDGE)
#include "rollout_fwd_inst.cuh"

namespace rlsde {
template <int D, int H>
int launch_rollout_fwd_bridge(const float* params_host, const FwdArgs& args, int sm_count, cudaStream_t stream) {
  return launch_fwd_policy<D, H, true>(params_host, args, sm_count, stream);
}
template int launch_rollout_fwd_bridge<1, 32>(const float*, const FwdArgs&, int, cudaStream_t);
}  // namespace rlsde
