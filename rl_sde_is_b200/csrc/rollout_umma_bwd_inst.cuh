// Launcher + explicit instantiation helper for the tcgen05 reverse pass of one shape (D, H), H in {128, 256}.
#pragma once
#include <cmath>
#include <cstdio>
#include <vector>
#include "rollout_umma_bwd.cuh"

namespace rlsde {

// producers and consumers for a batch: every producer needs a tile, every consumer serves at most UB_PPC producers, and
// the whole grid must be resident (one CTA per SM)
static inline void ub_grid(long long K, int sm_count, int& n_prod, int& n_cons) {
  const long long tiles = (K + UMMA_M - 1) / UMMA_M;
  long long np = (long long)sm_count * UB_PPC / (UB_PPC + 1);
  if (np > tiles) np = tiles;
  if (np < 1) np = 1;
  n_prod = (int)np;
  n_cons = (n_prod + UB_PPC - 1) / UB_PPC;
}

template <int D, int H>
struct UbScratch {
  static constexpr size_t o_ctl = 0;
  static constexpr size_t o_img2 = 512 * UB_CTL_WORDS * sizeof(unsigned);            // control words of up to 512 producers
  static constexpr size_t o_partial = o_img2 + umma_image_bytes<H>();
  static size_t partial_bytes(int n_prod, int n_cons) {
    return (((size_t)n_cons * H * H + (size_t)n_prod * ub_small_count<D, H>()) * sizeof(double) + 255) & ~(size_t)255;
  }
  static size_t o_xbuf(int n_prod, int n_cons) { return o_partial + partial_bytes(n_prod, n_cons); }
  static size_t total(int n_prod, int n_cons) { return o_xbuf(n_prod, n_cons) + (size_t)n_prod * UB_RING * ub_pass_bytes<H>(); }
};

template <int D, int H>
size_t bwd_umma_scratch_bytes(int sm_count) {
  int n_prod, n_cons;
  ub_grid((long long)1 << 40, sm_count, n_prod, n_cons);
  return UbScratch<D, H>::total(n_prod, n_cons);
}

template <int D, int H, bool FAST, bool WEIGHTED, bool RAGGED>
static int launch_bwd_umma_variant(const float* params_dev, const uint8_t* img1, const FwdArgs& args, float scale, float* grad,
                                   uint8_t* scratch, int n_prod, int n_cons, float w3max, cudaStream_t stream) {
  typedef UbScratch<D, H> S;
  constexpr int P = D * H + H + H * H + H + H * D + D;
  auto kern = rollout_bwd_umma_kernel<D, H, FAST, WEIGHTED, RAGGED>;
  const size_t smem = ub_smem_bytes<D, H>();
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
  double* partial = reinterpret_cast<double*>(scratch + S::o_partial);
  // producers and consumers wait for each other: a cooperative launch makes the runtime guarantee that the whole grid is
  // resident at once (it fails with cudaErrorCooperativeLaunchTooLarge instead of deadlocking if it cannot be)
  const uint8_t* img2 = scratch + S::o_img2;
  uint8_t* xbuf = scratch + S::o_xbuf(n_prod, n_cons);
  unsigned* ctl = reinterpret_cast<unsigned*>(scratch + S::o_ctl);
  FwdArgs a = args;
  void* kargs[] = {(void*)&params_dev, (void*)&img1, (void*)&img2, (void*)&a, (void*)&xbuf, (void*)&ctl, (void*)&partial,
                   (void*)&n_prod, (void*)&n_cons};
  if constexpr (WEIGHTED)
    ub_scale_weighted_kernel<<<1, 1024, 0, stream>>>((const float*)args.S, (const float*)args.G, args.T, args.K, w3max, sqrtf(args.dt_f),
                                                     D, n_prod, ctl);
  else
    ub_scale_kernel<<<1, 1024, 0, stream>>>((const float*)args.G, args.T, args.K, w3max, sqrtf(args.dt_f), D, n_prod, ctl);
  e = cudaLaunchCooperativeKernel((const void*)kern, dim3((unsigned)(n_prod + n_cons)), dim3(UB_THREADS), kargs, smem, stream);
  if (e != cudaSuccess) return (int)e;
  ub_reduce_kernel<D, H><<<(P + 127) / 128, 128, 0, stream>>>(partial, n_prod, n_cons, scale, ctl, grad, args.grad_accumulate);
#ifdef UB_PROFILE
  {
    std::vector<unsigned> h((size_t)n_prod * UB_CTL_WORDS);
    cudaStreamSynchronize(stream);
    cudaMemcpy(h.data(), scratch + S::o_ctl, h.size() * sizeof(unsigned), cudaMemcpyDeviceToHost);
    const char* names[8] = {"slot_wait", "layer1", "wait_accZ", "sweep1", "a+sweep2", "publish", "wait_accG", "sweep3+adjoint"};
    for (int pi = 0; pi < n_prod; pi += (n_prod > 8 ? n_prod / 4 : 1)) {
      fprintf(stderr, "[ub profile] producer %d: passes %u;", pi, h[(size_t)pi * UB_CTL_WORDS]);
      for (int i = 0; i < 8; ++i) fprintf(stderr, " %s %.2f us/pass;", names[i], 256.0 * h[(size_t)pi * UB_CTL_WORDS + 4 + i] / 1.965e3 / (h[(size_t)pi * UB_CTL_WORDS] ? h[(size_t)pi * UB_CTL_WORDS] : 1));
      fprintf(stderr, "\n");
    }
  }
#endif
  note_kernel_launches(3);
  return (int)cudaGetLastError();
}

template <int D, int H, bool WEIGHTED, bool RAGGED>
int launch_rollout_bwd_umma(const float* params_host, float* params_dev, uint8_t* image_dev, const FwdArgs& args, float scale,
                            float* grad, uint8_t* scratch, size_t scratch_bytes, int sm_count, cudaStream_t stream) {
  typedef UbScratch<D, H> S;
  if (args.ckpt_every != 1) return (int)cudaErrorInvalidValue;
  const bool fast = (args.flags & RLSDE_F_TANH_FAST) != 0;
  int n_prod, n_cons;
  ub_grid(args.K, sm_count, n_prod, n_cons);
  if (n_prod > 512 || scratch_bytes < S::total(n_prod, n_cons)) return (int)cudaErrorInvalidValue;
  std::vector<float> img(WideParams<D, H>::count);
  pack_wide_params<D, H>(params_host, fast, img.data());
  std::vector<uint16_t> w1(umma_image_bytes<H>() / 2), w2(umma_image_bytes<H>() / 2);
  pack_umma_weights<H>(img.data() + WideParams<D, H>::o_W2, w1.data());      // B[n = out][k = in]   (Z2 = H1 W2^T)
  pack_umma_weights<H>(img.data() + WideParams<D, H>::o_W2t, w2.data());     // B[n = in][k = out]   (dH1 = dZ2 W2)
  // largest head weight: the device picks the launch's scale exponent from it and from max |G| (ub_scale_kernel) or the
  // coefficients (ub_scale_weighted_kernel)
  double w3max = 0.0;
  for (int c = 0; c < H; ++c)
    for (int i = 0; i < D; ++i) w3max = fmax(w3max, fabs((double)img[WideParams<D, H>::o_W3 + (size_t)i * H + c]));
  cudaError_t e = cudaMemcpyAsync(params_dev, img.data(), img.size() * sizeof(float), cudaMemcpyHostToDevice, stream);
  if (e != cudaSuccess) return (int)e;
  if ((e = cudaMemcpyAsync(image_dev, w1.data(), umma_image_bytes<H>(), cudaMemcpyHostToDevice, stream)) != cudaSuccess) return (int)e;
  if ((e = cudaMemcpyAsync(scratch + S::o_img2, w2.data(), umma_image_bytes<H>(), cudaMemcpyHostToDevice, stream)) != cudaSuccess) return (int)e;
  if ((e = cudaMemsetAsync(scratch + S::o_ctl, 0, S::o_img2, stream)) != cudaSuccess) return (int)e;
  if ((e = cudaMemsetAsync(scratch + S::o_partial, 0, S::partial_bytes(n_prod, n_cons), stream)) != cudaSuccess) return (int)e;
  return with_flag(fast, [&](auto fast_c) {
    return launch_bwd_umma_variant<D, H, fast_c, WEIGHTED, RAGGED>(params_dev, image_dev, args, scale, grad, scratch, n_prod, n_cons,
                                                                   (float)w3max, stream);
  });
}

}  // namespace rlsde

#define RLSDE_INSTANTIATE_UMMA_BWD(D, H, WEIGHTED, RAGGED)                                                                  \
  template int rlsde::launch_rollout_bwd_umma<D, H, WEIGHTED, RAGGED>(const float*, float*, uint8_t*, const rlsde::FwdArgs&, float, \
                                                                      float*, uint8_t*, size_t, int, cudaStream_t);
#define RLSDE_INSTANTIATE_UMMA_BWD_SCRATCH(D, H) template size_t rlsde::bwd_umma_scratch_bytes<D, H>(int);
