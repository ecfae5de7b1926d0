// Launcher + explicit instantiation helper for one policy shape (D, H) of the reverse pass.
#pragma once
#include "rollout_bwd.cuh"

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

template <int D, int H, bool FAST, bool WEIGHTED, bool RAGGED>
static int launch_bwd_variant(const float* params_host, const FwdArgs& args, float scale, float* grad, float* partial,
                              int sm_count, cudaStream_t stream) {
  constexpr int P = D * H + H + H * H + H + H * D + D;
  static_assert(P <= BWD_MAX_PARAMS, "raise BWD_MAX_PARAMS");
  if (args.ckpt_every > BWD_MAX_SEG) return (int)cudaErrorInvalidValue;
  MlpConst<D, H> W;
  pack_mlp_const<D, H>(params_host, FAST, W);
  auto kern = rollout_bwd_kernel<D, H, FAST, WEIGHTED, RAGGED>;
  const size_t smem_per_warp = (size_t)(2 * tile_floats<H, bwd_tiles_padded(D)>() + 64 * D) * sizeof(float);
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smem_per_warp * 4));
  int block;
  long long grid = persistent_grid(kern, args.K, sm_count, smem_per_warp * 4, 0, block);
  long long n_warps = grid * (block / 32);
  if (n_warps > BWD_MAX_WARPS) { grid = BWD_MAX_WARPS / (block / 32); n_warps = grid * (block / 32); }
  const size_t smem = smem_per_warp * (block / 32);
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  kern<<<(unsigned)grid, block, smem, stream>>>(W, args, partial);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  bwd_reduce_kernel<<<(P + 127) / 128, 128, 0, stream>>>(partial, (int)n_warps, P, scale, grad, args.grad_accumulate);
  note_kernel_launches(2);
  return (int)cudaGetLastError();
}

template <int D, int H, bool WEIGHTED, bool RAGGED>
int launch_rollout_bwd(const float* params_host, const FwdArgs& args, float scale, float* grad, float* partial,
                       int sm_count, cudaStream_t stream) {
  return with_flag((args.flags & RLSDE_F_TANH_FAST) != 0, [&](auto fast) {
    return launch_bwd_variant<D, H, fast, WEIGHTED, RAGGED>(params_host, args, scale, grad, partial, sm_count, stream);
  });
}

}  // namespace rlsde

#define RLSDE_INSTANTIATE_BWD(D, H, WEIGHTED, RAGGED) \
  template int rlsde::launch_rollout_bwd<D, H, WEIGHTED, RAGGED>(const float*, const rlsde::FwdArgs&, float, float*, float*, int, cudaStream_t);
