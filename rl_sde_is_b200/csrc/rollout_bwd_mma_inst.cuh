// Launcher + explicit instantiation helper for the tensor-core reverse pass of one state dimension D (H = 32).
#pragma once
#include <cmath>
#include <cstring>
#include "rollout_bwd_mma.cuh"

namespace rlsde {

template <int D, bool FAST, bool WEIGHTED, bool RAGGED>
static int launch_bwd_mma_variant(const float* params_host, const FwdArgs& args, float scale, float* grad, void* partial,
                                  int sm_count, cudaStream_t stream, cudaEvent_t join) {
  constexpr int P = D * MMA_H + MMA_H + MMA_H * MMA_H + MMA_H + MMA_H * D + D;
  static_assert((size_t)P * sizeof(double) <= (size_t)BWD_MAX_PARAMS * sizeof(float) , "fp64 partials must fit the reverse-pass workspace");
  if (args.ckpt_every > BWD_MAX_SEG) return (int)cudaErrorInvalidValue;
  MlpConst<D, MMA_H> W;
  pack_mlp_const<D, MMA_H>(params_host, FAST, W);
  BwdMmaWeights F;
  pack_bwd_mma_weights<D>(W, F);
  typename BwdMmaSmallSel<D>::type FS;
  pack_bwd_mma_small<D>(W, FAST, FS);
  auto kern = rollout_bwd_mma_kernel<D, FAST, WEIGHTED, RAGGED>;
  // d > 4: fragment table of the d-sized products + per-warp staging rows; accumulator tiles (rollout_bwd_mma.cuh)
  auto dyn_smem = [](int blk) { return bwd_mma_dyn_smem(D, blk); };
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn_smem(128));
  int block;
  long long grid = persistent_grid(kern, args.K, sm_count, dyn_smem(128), 0, block);
  long long n_warps = grid * (block / 32);
  if (n_warps > BWD_MAX_WARPS) { grid = BWD_MAX_WARPS / (block / 32); n_warps = grid * (block / 32); }
  kern<<<(unsigned)grid, block, dyn_smem(block), stream>>>(W, args, F, FS, reinterpret_cast<double*>(partial));
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  if (join != nullptr && (e = cudaStreamWaitEvent(stream, join, 0)) != cudaSuccess) return (int)e;
  bwd_reduce64_kernel<<<(P + 127) / 128, 128, 0, stream>>>(reinterpret_cast<const double*>(partial), (int)n_warps, P, scale, grad,
                                                           args.grad_accumulate);
  note_kernel_launches(2);
  return (int)cudaGetLastError();
}

template <int D, bool WEIGHTED, bool RAGGED>
int launch_rollout_bwd_mma(const float* params_host, const FwdArgs& args, float scale, float* grad, void* partial,
                           int sm_count, cudaStream_t stream, cudaEvent_t join) {
  return with_flag((args.flags & RLSDE_F_TANH_FAST) != 0, [&](auto fast) {
    return launch_bwd_mma_variant<D, fast, WEIGHTED, RAGGED>(params_host, args, scale, grad, partial, sm_count, stream, join);
  });
}

}  // namespace rlsde

#define RLSDE_INSTANTIATE_BWD_MMA(D, WEIGHTED, RAGGED)                                                                  \
  template int rlsde::launch_rollout_bwd_mma<D, WEIGHTED, RAGGED>(const float*, const rlsde::FwdArgs&, float, float*, void*, int, \
                                                                  cudaStream_t, cudaEvent_t);
