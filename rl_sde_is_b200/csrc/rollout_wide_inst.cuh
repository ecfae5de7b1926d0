// Launchers + explicit instantiation helper for the wide-policy kernels of one shape (D, H), H in {64, 128, 256}.
#pragma once
#include <vector>
#include "rollout_wide.cuh"

namespace rlsde {

// policy parameters: host (state_dict order) -> packed float32 image -> the caller's workspace.  The copy is ordered on
// the stream; cudaMemcpyAsync from pageable memory returns once the source has been staged, so the temporary may go.
template <int D, int H>
static int wide_upload_params(const float* params_host, float* params_dev, bool fast, cudaStream_t stream) {
  std::vector<float> img(WideParams<D, H>::count);
  pack_wide_params<D, H>(params_host, fast, img.data());
  return (int)cudaMemcpyAsync(params_dev, img.data(), img.size() * sizeof(float), cudaMemcpyHostToDevice, stream);
}

// rows per warp: 8 (tiles of 32 trajectories) when the batch fills the GPU with such tiles, else 4 (tiles of 16)
static inline bool wide_small_tiles(long long K, int sm_count) { return K < (long long)sm_count * 32; }

template <int D, int H, int R, bool F64, bool FAST, bool BRIDGE, bool RAGGED = false>
static int launch_fwd_wide_variant(const float* params_dev, const FwdArgs& args, int sm_count, cudaStream_t stream) {
  auto kern = rollout_fwd_wide_kernel<D, H, R, F64, FAST, BRIDGE, RAGGED>;
  const size_t smem = wide_fwd_smem_bytes<H>();
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WIDE_THREADS, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
  long long grid = (long long)sm_count * per_sm;
  const long long need = (args.K + 4 * R - 1) / (4 * R);
  if (grid > need) grid = need;
  if (grid < 1) grid = 1;
  kern<<<(unsigned)grid, WIDE_THREADS, smem, stream>>>(params_dev, args);
  note_kernel_launches(1);
  return (int)cudaGetLastError();
}

template <int D, int H, bool RAGGED>
int launch_rollout_fwd_wide(const float* params_host, float* params_dev, const FwdArgs& args, int sm_count, cudaStream_t stream) {
  int rc = wide_upload_params<D, H>(params_host, params_dev, (args.flags & RLSDE_F_TANH_FAST) != 0, stream);
  if (rc != 0) return rc;
  return with_flag(wide_small_tiles(args.K, sm_count), [&](auto small) {
    return with_fwd_variant<D, RAGGED>(args.flags, [&](auto f64, auto fast, auto bridge) {
      return launch_fwd_wide_variant<D, H, small ? 4 : 8, f64, fast, bridge, RAGGED>(params_dev, args, sm_count, stream);
    });
  });
}

template <int D, int H, int R, bool FAST, bool WEIGHTED, bool RAGGED>
static int launch_bwd_wide_variant(const float* params_dev, const FwdArgs& args, float scale, float* grad, float* partial,
                                   size_t partial_bytes, int sm_count, cudaStream_t stream) {
  constexpr int P = D * H + H + H * H + H + H * D + D;
  auto kern = rollout_bwd_wide_kernel<D, H, R, FAST, WEIGHTED, RAGGED>;
  const size_t smem = wide_bwd_smem_bytes<H>();
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WIDE_THREADS, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
  long long grid = (long long)sm_count * per_sm;
  const long long need = (args.K + 4 * R - 1) / (4 * R);
  if (grid > need) grid = need;
  const long long fit = (long long)(partial_bytes / ((size_t)P * sizeof(float)));
  if (grid > fit) grid = fit;
  if (grid < 1) return (int)cudaErrorInvalidValue;
  kern<<<(unsigned)grid, WIDE_THREADS, smem, stream>>>(params_dev, args, partial);
  e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  wide_reduce_kernel<<<(P + 127) / 128, 128, 0, stream>>>(partial, (int)grid, P, scale, grad, args.grad_accumulate);
  note_kernel_launches(2);
  return (int)cudaGetLastError();
}

template <int D, int H, bool WEIGHTED, bool RAGGED>
int launch_rollout_bwd_wide(const float* params_host, float* params_dev, const FwdArgs& args, float scale, float* grad, float* partial,
                            size_t partial_bytes, int sm_count, cudaStream_t stream) {
  if (args.ckpt_every != 1) return (int)cudaErrorInvalidValue;
  int rc = wide_upload_params<D, H>(params_host, params_dev, (args.flags & RLSDE_F_TANH_FAST) != 0, stream);
  if (rc != 0) return rc;
  return with_flag(wide_small_tiles(args.K, sm_count), [&](auto small) {
    return with_flag((args.flags & RLSDE_F_TANH_FAST) != 0, [&](auto fast) {
      return launch_bwd_wide_variant<D, H, small ? 4 : 8, fast, WEIGHTED, RAGGED>(params_dev, args, scale, grad, partial,
                                                                                 partial_bytes, sm_count, stream);
    });
  });
}

}  // namespace rlsde

#define RLSDE_INSTANTIATE_FWD_WIDE(D, H, RAGGED) \
  template int rlsde::launch_rollout_fwd_wide<D, H, RAGGED>(const float*, float*, const rlsde::FwdArgs&, int, cudaStream_t);
#define RLSDE_INSTANTIATE_BWD_WIDE(D, H, WEIGHTED, RAGGED)                                                                  \
  template int rlsde::launch_rollout_bwd_wide<D, H, WEIGHTED, RAGGED>(const float*, float*, const rlsde::FwdArgs&, float,   \
                                                                      float*, float*, size_t, int, cudaStream_t);
