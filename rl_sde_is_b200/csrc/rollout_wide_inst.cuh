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
  const bool f64 = (args.flags & RLSDE_F_STATE_F64) != 0, fast = (args.flags & RLSDE_F_TANH_FAST) != 0;
  int rc = wide_upload_params<D, H>(params_host, params_dev, fast, stream);
  if (rc != 0) return rc;
  const bool small = wide_small_tiles(args.K, sm_count);
#define RLSDE_WIDE_FWD(R_, B_) \
  (f64 ? (fast ? launch_fwd_wide_variant<D, H, R_, true, true, B_>(params_dev, args, sm_count, stream)    \
               : launch_fwd_wide_variant<D, H, R_, true, false, B_>(params_dev, args, sm_count, stream))  \
       : (fast ? launch_fwd_wide_variant<D, H, R_, false, true, B_>(params_dev, args, sm_count, stream)   \
               : launch_fwd_wide_variant<D, H, R_, false, false, B_>(params_dev, args, sm_count, stream)))
  if constexpr (RAGGED) {      // float32 state, no Brownian-bridge test: the caller refuses both
    if (small) return fast ? launch_fwd_wide_variant<D, H, 4, false, true, false, true>(params_dev, args, sm_count, stream)
                           : launch_fwd_wide_variant<D, H, 4, false, false, false, true>(params_dev, args, sm_count, stream);
    return fast ? launch_fwd_wide_variant<D, H, 8, false, true, false, true>(params_dev, args, sm_count, stream)
                : launch_fwd_wide_variant<D, H, 8, false, false, false, true>(params_dev, args, sm_count, stream);
  } else {
    if constexpr (D == 1) {      // RLSDE_F_HIT_BRIDGE: the caller accepts it at d = 1 only
      if (args.flags & RLSDE_F_HIT_BRIDGE) return small ? RLSDE_WIDE_FWD(4, true) : RLSDE_WIDE_FWD(8, true);
    }
    return small ? RLSDE_WIDE_FWD(4, false) : RLSDE_WIDE_FWD(8, false);
  }
#undef RLSDE_WIDE_FWD
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
  const bool fast = (args.flags & RLSDE_F_TANH_FAST) != 0;
  int rc = wide_upload_params<D, H>(params_host, params_dev, fast, stream);
  if (rc != 0) return rc;
  const bool small = wide_small_tiles(args.K, sm_count);
  if (small) return fast ? launch_bwd_wide_variant<D, H, 4, true, WEIGHTED, RAGGED>(params_dev, args, scale, grad, partial, partial_bytes, sm_count, stream)
                         : launch_bwd_wide_variant<D, H, 4, false, WEIGHTED, RAGGED>(params_dev, args, scale, grad, partial, partial_bytes, sm_count, stream);
  return fast ? launch_bwd_wide_variant<D, H, 8, true, WEIGHTED, RAGGED>(params_dev, args, scale, grad, partial, partial_bytes, sm_count, stream)
              : launch_bwd_wide_variant<D, H, 8, false, WEIGHTED, RAGGED>(params_dev, args, scale, grad, partial, partial_bytes, sm_count, stream);
}

}  // namespace rlsde

#define RLSDE_INSTANTIATE_WIDE(D, H)                                                                                        \
  template int rlsde::launch_rollout_fwd_wide<D, H>(const float*, float*, const rlsde::FwdArgs&, int, cudaStream_t);       \
  template int rlsde::launch_rollout_bwd_wide<D, H>(const float*, float*, const rlsde::FwdArgs&, float, float*, float*,   \
                                                    size_t, int, cudaStream_t);
// the weighted reverse pass (rlsde_rollout_bwd_weighted), in translation units of its own
#define RLSDE_INSTANTIATE_WIDE_BWD_WEIGHTED(D, H)                                                                           \
  template int rlsde::launch_rollout_bwd_wide<D, H, true>(const float*, float*, const rlsde::FwdArgs&, float, float*, float*, \
                                                          size_t, int, cudaStream_t);
// the ragged checkpoint store (rlsde_rollout_fwd_ragged / rlsde_rollout_bwd_ragged), in translation units of its own
#define RLSDE_INSTANTIATE_WIDE_RAGGED(D, H)                                                                                 \
  template int rlsde::launch_rollout_fwd_wide<D, H, true>(const float*, float*, const rlsde::FwdArgs&, int, cudaStream_t); \
  template int rlsde::launch_rollout_bwd_wide<D, H, true, true>(const float*, float*, const rlsde::FwdArgs&, float, float*,  \
                                                                float*, size_t, int, cudaStream_t);
