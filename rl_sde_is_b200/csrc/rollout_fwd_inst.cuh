// Launcher + explicit instantiation helper for one policy shape (D, H) of the forward rollout.
#pragma once
#include "rollout_fwd.cuh"

namespace rlsde {

template <int D, int H, bool F64, bool FAST, bool MMA, bool BRIDGE, bool RAGGED = false>
static int launch_fwd_variant(const float* params_host, const FwdArgs& args, int sm_count, cudaStream_t stream) {
  MlpConst<D, H> W;
  if (!FAST && RLSDE_FWD_FOLDED) pack_mlp_const_folded<D, H>(params_host, W);
  else pack_mlp_const<D, H>(params_host, FAST, W);
  typename FwdMmaSel<D, MMA>::type M;
  if constexpr (MMA) pack_mlp_mma<D>(W, M);
  else M.unused = 0;
  FwdArgs a = args;
  auto kern = rollout_fwd_kernel<D, H, F64, FAST, MMA, true, BRIDGE, RAGGED>;
  a.mma_x1_max = -1.0f;
  if constexpr (MMA && !FAST) {
    // leave the clamp of the grouped reciprocal out where it provably cannot bind (same bits, fewer instructions)
    double z2_max, x1_max;
    fwd_mma_clamp_bounds<D, H>(W, z2_max, x1_max);
    a.mma_x1_max = (float)x1_max;
    if (z2_max <= RCP_GROUP_SAFE_Z) kern = rollout_fwd_kernel<D, H, F64, FAST, MMA, false, BRIDGE, RAGGED>;
  }
  int block;
  const long long grid = persistent_grid(kern, args.K, sm_count, 0, args.blocks_per_sm_cap, block);
  // Schedule (rollout_fwd.cuh; chosen by the C ABI layer: args.q_quantum passes per slice, or run to completion with
  // the tail handed over to the warp-per-trajectory kernel at args.q_handoff live trajectories): large batches only, and
  // only if the caller's workspace holds a ring with one record per trajectory plus one per lane.
  const long long lanes = grid * block;
  long long need_cap = 1;
  int cap_log2 = 0;
  while (need_cap < args.K + lanes) { need_cap <<= 1; ++cap_log2; }      // power of two: slot = index & (cap - 1)
  const size_t rec = sizeof(ContRec<D, F64>);
  if (block == 128 && (args.q_quantum > 0 || args.q_handoff > 0) && args.q_ring != nullptr &&
      (size_t)need_cap * rec <= (size_t)args.q_cap) {
    a.q_cap = need_cap;                                  // args.q_cap came in as the BYTES available for the ring
    a.q_cap_log2 = cap_log2;
    if (a.q_quantum > 0) {                               // the FIFO protocol needs all-zero sequence words
      cudaError_t e = cudaMemsetAsync(a.q_ring, 0, (size_t)need_cap * rec, stream);
      if (e != cudaSuccess) return (int)e;
    }
  } else {
    a.q_ring = nullptr; a.q_cap = 0; a.q_cap_log2 = 0; a.q_quantum = 0; a.q_handoff = 0;
  }
  kern<<<(unsigned)grid, block, 0, stream>>>(W, a, M);
  note_kernel_launches(1);
  return (int)cudaGetLastError();
}

// args.policy_mma selects the policy arithmetic; the caller checks fwd_mma_shape(D, H) before it sets it
template <int D, int H, bool BRIDGE, bool RAGGED = false>
static int launch_fwd_policy(const float* params_host, const FwdArgs& args, int sm_count, cudaStream_t stream) {
  return with_flag<fwd_mma_shape(D, H)>(args.policy_mma != 0, [&](auto mma) {
    return with_fwd_state<RAGGED>(args.flags, [&](auto f64, auto fast) {
      return launch_fwd_variant<D, H, f64, fast, mma, BRIDGE, RAGGED>(params_host, args, sm_count, stream);
    });
  });
}

// The kernels with the Brownian-bridge hit test (RLSDE_F_HIT_BRIDGE, d = 1) live in a translation unit of their own
// (fwd_d1_h32_bridge.cu): compiled next to the others, they changed how ptxas allocated an existing kernel's registers.
// So do the ragged-store kernels (fwd_d*_h32_ragged.cu).
template <int D, int H>
int launch_rollout_fwd_bridge(const float* params_host, const FwdArgs& args, int sm_count, cudaStream_t stream);

template <int D, int H, bool RAGGED>
int launch_rollout_fwd(const float* params_host, const FwdArgs& args, int sm_count, cudaStream_t stream) {
  return with_fwd_bridge<D, RAGGED>(args.flags, [&](auto bridge) {
    if constexpr (bridge) return launch_rollout_fwd_bridge<D, H>(params_host, args, sm_count, stream);
    else return launch_fwd_policy<D, H, false, RAGGED>(params_host, args, sm_count, stream);
  });
}

}  // namespace rlsde

#define RLSDE_INSTANTIATE_FWD(D, H, RAGGED) \
  template int rlsde::launch_rollout_fwd<D, H, RAGGED>(const float*, const rlsde::FwdArgs&, int, cudaStream_t);
