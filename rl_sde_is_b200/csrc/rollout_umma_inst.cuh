// Launcher + explicit instantiation helper for the tcgen05 forward rollout of one shape (D, H), H in {128, 256}.
#pragma once
#include <vector>
#include "rollout_umma.cuh"

namespace rlsde {

template <int D, int H, bool F64, bool FAST, bool BRIDGE, bool RAGGED = false>
static int launch_fwd_umma_variant(const float* params_dev, const uint8_t* image_dev, const FwdArgs& args, int sm_count, cudaStream_t stream) {
  auto kern = rollout_fwd_umma_kernel<D, H, F64, FAST, BRIDGE, RAGGED>;
  const size_t smem = umma_smem_bytes<D, H>();
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  // two CTAs per SM when shared memory and tensor memory allow (100 KB, H <= 256 columns each): one reads its accumulator
  // back while the other's MMAs run
  // (the occupancy query answers 1 under the default carveout, so the carveout is requested and the count derived here)
  cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
  constexpr int THREADS = umma_threads<H>();
  cudaFuncAttributes fa;
  if ((e = cudaFuncGetAttributes(&fa, kern)) != cudaSuccess) return (int)e;
  int per_sm = (int)(((size_t)227 * 1024) / (smem + 2048));
  const int by_regs = 65536 / (THREADS * (fa.numRegs > 0 ? ((fa.numRegs + 7) & ~7) : 128));
  if (per_sm > by_regs) per_sm = by_regs;
  if (per_sm > 512 / umma_tmem_cols<H>()) per_sm = 512 / umma_tmem_cols<H>();     // tensor memory: 512 columns per SM
  if (per_sm > 8) per_sm = 8;
  if (per_sm < 1) per_sm = 1;
  long long grid = (long long)sm_count * per_sm;
  const long long need = (args.K + UMMA_M - 1) / UMMA_M;
  if (grid > need) grid = need;
  if (grid < 1) grid = 1;
  kern<<<(unsigned)grid, THREADS, smem, stream>>>(params_dev, image_dev, args);
  note_kernel_launches(1);
  return (int)cudaGetLastError();
}

template <int D, int H, bool RAGGED>
int launch_rollout_fwd_umma(const float* params_host, float* params_dev, uint8_t* image_dev, const FwdArgs& args, int sm_count,
                            cudaStream_t stream) {
  const bool fast = (args.flags & RLSDE_F_TANH_FAST) != 0;
  std::vector<float> img(WideParams<D, H>::count);
  pack_wide_params<D, H>(params_host, fast, img.data());
  std::vector<uint16_t> wimg(umma_image_bytes<H>() / 2);
  pack_umma_weights<H>(img.data() + WideParams<D, H>::o_W2, wimg.data());
  cudaError_t e = cudaMemcpyAsync(params_dev, img.data(), img.size() * sizeof(float), cudaMemcpyHostToDevice, stream);
  if (e != cudaSuccess) return (int)e;
  e = cudaMemcpyAsync(image_dev, wimg.data(), umma_image_bytes<H>(), cudaMemcpyHostToDevice, stream);
  if (e != cudaSuccess) return (int)e;
  return with_fwd_variant<D, RAGGED>(args.flags, [&](auto f64, auto fast, auto bridge) {
    return launch_fwd_umma_variant<D, H, f64, fast, bridge, RAGGED>(params_dev, image_dev, args, sm_count, stream);
  });
}

}  // namespace rlsde

#define RLSDE_INSTANTIATE_UMMA(D, H, RAGGED) \
  template int rlsde::launch_rollout_fwd_umma<D, H, RAGGED>(const float*, float*, uint8_t*, const rlsde::FwdArgs&, int, cudaStream_t);
