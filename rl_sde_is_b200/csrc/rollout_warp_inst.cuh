// Launchers + explicit instantiation helper for the warp-per-trajectory kernels of one state dimension D (H = 32).
#pragma once
#include <cstring>
#include "rollout_bwd.cuh"
#include "rollout_warp.cuh"

namespace rlsde {

// grad[p] (+)= scale * sum_w partial[w][p], warps in index order
static __global__ void bwd_reduce_kernel(const float* __restrict__ partial, int n_warps, int P, float scale, float* __restrict__ grad,
                                         int accumulate) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  double acc = 0.0;
  for (int w = 0; w < n_warps; ++w) acc += (double)partial[(long long)w * P + p];
  const float g = (float)(acc * (double)scale);
  grad[p] = accumulate ? grad[p] + g : g;
}

static inline long long warp_grid(long long K, int sm_count) {
  long long g = (K + 3) / 4;
  const long long cap = (long long)sm_count * 4;     // 16 warps per SM: every warp still has an SM sub-partition mostly to itself
  if (g > cap) g = cap;
  return g < 1 ? 1 : g;
}

// device-side twin of pack_mlp_const (common.cuh): one thread per entry, same double-precision scaling
template <int D>
static __global__ void pack_mlp_const_kernel(const float* __restrict__ p, MlpConst<D, WARP_H>* out, bool fast_tanh) {
  constexpr int H = WARP_H;
  const double s = fast_tanh ? 1.0 : RLSDE_TWO_LOG2E;
  const float* W1 = p;
  const float* b1 = W1 + H * D;
  const float* W2 = b1 + H;
  const float* b2 = W2 + H * H;
  const float* W3 = b2 + H;
  const float* b3 = W3 + D * H;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < H * H; e += gridDim.x * blockDim.x) {
    const int i = e / H, j = e % H;
    out->W2t[i][j] = (float)(s * (double)W2[j * H + i]);
    if (i < D) { out->W1t[i][j] = (float)(s * (double)W1[j * D + i]); out->W3[i][j] = W3[i * H + j]; }
    if (i == 0) { out->b1[j] = (float)(s * (double)b1[j]); out->b2[j] = (float)(s * (double)b2[j]); }
    if (e < ((D + 3) & ~3)) out->b3[e] = e < D ? b3[e] : 0.0f;
  }
}

template <int D>
int launch_pack_mlp_const_dev(const float* theta_dev, void* W_dev, bool fast_tanh, cudaStream_t stream) {
  static_assert(D <= WARP_H, "one pass over the H x H block covers the narrow blocks too");
  pack_mlp_const_kernel<D><<<4, 256, 0, stream>>>(theta_dev, reinterpret_cast<MlpConst<D, WARP_H>*>(W_dev), fast_tanh);
  note_kernel_launches(1);
  return (int)cudaGetLastError();
}

template <int D, bool F64, bool FAST, bool BRIDGE, bool RAGGED>
static int launch_fwd_warp_variant(const float* params_host, const void* W_dev, const FwdArgs& args, int sm_count, cudaStream_t stream) {
  MlpConst<D, WARP_H> W;
  if (params_host != nullptr) pack_mlp_const<D, WARP_H>(params_host, FAST, W);
  else memset(&W, 0, sizeof(W));
  rollout_fwd_warp_kernel<D, F64, FAST, false, false, BRIDGE, RAGGED><<<(unsigned)warp_grid(args.K, sm_count), 128, 0, stream>>>(
      W, params_host != nullptr ? nullptr : reinterpret_cast<const MlpConst<D, WARP_H>*>(W_dev), args, MlpMmaNone{0});
  note_kernel_launches(1);
  return (int)cudaGetLastError();
}

template <int D, bool RAGGED>
int launch_rollout_fwd_warp(const float* params_host, const void* W_dev, const FwdArgs& args, int sm_count, cudaStream_t stream) {
  return with_fwd_variant<D, RAGGED>(args.flags, [&](auto f64, auto fast, auto bridge) {
    return launch_fwd_warp_variant<D, f64, fast, bridge, RAGGED>(params_host, W_dev, args, sm_count, stream);
  });
}

template <int D, bool F64, bool FAST, bool MMA, bool BRIDGE, bool RAGGED>
static int launch_fwd_warp_resume_variant(const float* params_host, const FwdArgs& args, int sm_count, cudaStream_t stream) {
  MlpConst<D, WARP_H> W;
  if (!FAST && RLSDE_FWD_FOLDED) pack_mlp_const_folded<D, WARP_H>(params_host, W);      // the image K1 itself was launched with
  else pack_mlp_const<D, WARP_H>(params_host, FAST, W);
  typename FwdMmaSel<D, MMA>::type M;
  if constexpr (MMA) pack_mlp_mma<D>(W, M);
  else M.unused = 0;
  // the number of records is only known on the device: a full grid (16 warps per SM), warps without a record leave at once
  rollout_fwd_warp_kernel<D, F64, FAST, true, MMA, BRIDGE, RAGGED><<<(unsigned)(sm_count * 4), 128, 0, stream>>>(W, nullptr, args, M);
  note_kernel_launches(1);
  return (int)cudaGetLastError();
}

// continues with the policy arithmetic K1 was launched with (args.policy_mma)
template <int D, bool RAGGED>
int launch_rollout_fwd_warp_resume(const float* params_host, const FwdArgs& args, int sm_count, cudaStream_t stream) {
  return with_flag<fwd_mma_shape(D, WARP_H)>(args.policy_mma != 0, [&](auto mma) {
    return with_fwd_variant<D, RAGGED>(args.flags, [&](auto f64, auto fast, auto bridge) {
      return launch_fwd_warp_resume_variant<D, f64, fast, mma, bridge, RAGGED>(params_host, args, sm_count, stream);
    });
  });
}

template <int D, bool FAST, bool WEIGHTED, bool RAGGED>
static int launch_bwd_warp_variant(const float* params_host, const void* W_dev, const FwdArgs& args, float scale, float* grad,
                                   float* partial, int sm_count, cudaStream_t stream) {
  constexpr int P = D * WARP_H + WARP_H + WARP_H * WARP_H + WARP_H + WARP_H * D + D;
  MlpConst<D, WARP_H> W;
  if (params_host != nullptr) pack_mlp_const<D, WARP_H>(params_host, FAST, W);
  else memset(&W, 0, sizeof(W));
  const long long grid = warp_grid(args.K, sm_count);
  rollout_bwd_warp_kernel<D, FAST, WEIGHTED, RAGGED><<<(unsigned)grid, 128, 0, stream>>>(
      W, params_host != nullptr ? nullptr : reinterpret_cast<const MlpConst<D, WARP_H>*>(W_dev), args, partial);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  bwd_reduce_kernel<<<(P + 127) / 128, 128, 0, stream>>>(partial, (int)(grid * 4), P, scale, grad, args.grad_accumulate);
  note_kernel_launches(2);
  return (int)cudaGetLastError();
}

template <int D, bool WEIGHTED, bool RAGGED>
int launch_rollout_bwd_warp(const float* params_host, const void* W_dev, const FwdArgs& args, float scale, float* grad,
                            float* partial, int sm_count, cudaStream_t stream) {
  return with_flag((args.flags & RLSDE_F_TANH_FAST) != 0, [&](auto fast) {
    return launch_bwd_warp_variant<D, fast, WEIGHTED, RAGGED>(params_host, W_dev, args, scale, grad, partial, sm_count, stream);
  });
}

}  // namespace rlsde

// the forward launchers of the warp-per-trajectory kernel: fresh trajectories and the ones K1 handed over
#define RLSDE_INSTANTIATE_FWD_WARP(D, RAGGED)                                                                              \
  template int rlsde::launch_rollout_fwd_warp<D, RAGGED>(const float*, const void*, const rlsde::FwdArgs&, int, cudaStream_t); \
  template int rlsde::launch_rollout_fwd_warp_resume<D, RAGGED>(const float*, const rlsde::FwdArgs&, int, cudaStream_t);
#define RLSDE_INSTANTIATE_BWD_WARP(D, WEIGHTED, RAGGED)                                                                    \
  template int rlsde::launch_rollout_bwd_warp<D, WEIGHTED, RAGGED>(const float*, const void*, const rlsde::FwdArgs&, float, \
                                                                   float*, float*, int, cudaStream_t);
#define RLSDE_INSTANTIATE_PACK_DEV(D) \
  template int rlsde::launch_pack_mlp_const_dev<D>(const float*, void*, bool, cudaStream_t);
