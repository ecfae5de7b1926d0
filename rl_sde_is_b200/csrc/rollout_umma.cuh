// K1u: forward rollout for wide policies (hidden width 128 / 256) with the hidden-hidden layer on the 5th-generation
// tensor cores (tcgen05.mma, accumulator in tensor memory) -- the case BASELINE.json's north_star reserves tcgen05 for:
// at H = 256 a pass of a 128-trajectory tile is a real dense contraction, 128 x 256 x 256.
//
// Same semantics, Philox stream and outputs as K1 / K1x (rollout_fwd.cuh, rollout_wide.cuh).  One CTA of 192 threads per
// SM advances a tile of 128 trajectories in lock step:
//   warps 0-3  one THREAD per trajectory (= one TMEM lane).  Per pass the thread evaluates layer 1 for its own state
//              (H FMAs + H tanh) sixteen units at a time, splits the activations into float16 hi + lo and writes its row
//              of that k-step's A operand into a ring of shared-memory slots in the K-major core-matrix layout tcgen05
//              reads (8 rows x 16 bytes, no swizzle) -- the MMAs of a k-step start as soon as its slot is full, so layer 1
//              overlaps the tensor pipe; after the MMAs it reads its row of the accumulator back (tcgen05.ld 32x32b: 32
//              columns per instruction), applies bias + tanh and sums the head in registers -- no cross-thread reduction
//              anywhere -- and runs the environment pass with K1's arithmetic (traj_owner.cuh).  Finished trajectories
//              are replaced from the global work counter (lane refill), so the tile stays full until the batch runs out.
//   warp 4     lane 0 issues the MMAs: per 16-wide k-step D += A_hi B_hi + A_lo B_hi + A_hi B_lo (M = 128, N = H, K = 16,
//              kind::f16, fp32 accumulate): float16 hi + lo carry 22 significand bits per operand, the dropped lo x lo
//              term is ~2^-22 -- fp32-level accuracy (rollout_bwd_mma.cuh has the error budget).  tcgen05.commit hands
//              each weight stage back to the producer and finally signals the accumulator.
//   warp 5     lane 0 streams the weights: W2 (pre-scaled, split into float16 hi / lo and laid out per k-step as the
//              shared-memory image of the B operand by the host) does not fit beside A at H = 256 (2 x 128 KB), so every
//              pass it travels L2 -> shared memory again, one cp.async.bulk of H x 64 bytes per k-step through a ring of
//              four mbarrier-guarded stages.  128 trajectories share each byte.
// Synchronisation is mbarriers only (a_full: 128 arrivals per slot, a_empty / empty / acc_ready: tcgen05.commit; full:
// the bulk copy's transaction count) plus one __syncthreads_or per pass for the "any trajectory left?" vote.  A CTA needs
// 100 KB of shared memory and H tensor-memory columns, so TWO CTAs share an SM: while one is in its accumulator-readback
// phase (MUFU-bound) the other's MMAs keep the tensor pipe busy.
#pragma once
#include <cuda_fp16.h>
#include "rollout_bwd_mma.cuh"     // f32 <-> f16 host helpers, split_pair
#include "rollout_wide.cuh"        // WideParams (device image of the small layers)
#include "traj_owner.cuh"

namespace rlsde {

constexpr int UMMA_M = 128;                 // trajectories per tile = TMEM lanes
constexpr int UMMA_STAGES = 4;                // weight stages (one k-step of B, hi + lo, each) when the weights are streamed
constexpr uint32_t UMMA_ACHUNK = UMMA_M * 16 * 2 * 2;   // bytes of one A slot: 128 rows x 16 halfs, hi + lo
// Hidden widths up to 64 keep the whole float16 hi / lo image of W2 in shared memory (4 KB at H = 32): no producer warp,
// 160 threads, four or more CTAs per SM.  Above, the image is streamed every pass (192 threads, two CTAs per SM).
template <int H> __host__ __device__ constexpr bool umma_streams() { return H > 64; }
template <int H> __host__ __device__ constexpr int umma_threads() { return umma_streams<H>() ? 192 : 160; }
template <int H> __host__ __device__ constexpr int umma_aslots() { return H / 16 < 4 ? H / 16 : 4; }   // activation slots (one k-step of A each)
template <int H> __host__ __device__ constexpr int umma_tmem_cols() { return H < 32 ? 32 : H; }

template <int H> __host__ __device__ constexpr size_t umma_chunk_bytes() { return (size_t)H * 64; }        // hi + lo of one k-step
template <int H> __host__ __device__ constexpr size_t umma_image_bytes() { return umma_chunk_bytes<H>() * (H / 16); }
template <int D, int H>
__host__ __device__ constexpr size_t umma_smem_bytes() {
  // the A ring, the weight ring (or the whole image), the small layers (W1t [D][H], b1, b2, W3 [D][H])
  return (size_t)umma_aslots<H>() * UMMA_ACHUNK + (umma_streams<H>() ? UMMA_STAGES * umma_chunk_bytes<H>() : umma_image_bytes<H>()) +
         (size_t)(2 * D + 2) * H * sizeof(float);
}

// host: W2 (pre-scaled like MlpConst / WideParams: w2s[out * H + in]) -> the B-operand image streamed by the kernel.
// Chunk ks (k = 16 ks .. 16 ks + 15): [hi | lo], each N = H rows x 16 halfs as 8 x 8 core matrices,
// core(kc, ng) at (kc * H/8 + ng) * 128 bytes, row n % 8 at +16 bytes, 8 halfs along k.
template <int H>
inline void pack_umma_weights(const float* w2s, uint16_t* img) {
  for (int ks = 0; ks < H / 16; ++ks)
    for (int n = 0; n < H; ++n)
      for (int kc = 0; kc < 2; ++kc)
        for (int e = 0; e < 8; ++e) {
          const float w = w2s[(size_t)n * H + 16 * ks + 8 * kc + e];
          const uint16_t hi = f32_to_f16_bits(w);
          const uint16_t lo = f32_to_f16_bits(w - f16_bits_to_f32(hi));
          const size_t base = (size_t)ks * (umma_chunk_bytes<H>() / 2) + ((size_t)(kc * (H / 8) + (n >> 3)) * 64) + (size_t)(n & 7) * 8 + e;
          img[base] = hi;
          img[base + (size_t)H * 16] = lo;
        }
}

namespace umma {
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// K-major, SWIZZLE_NONE shared-memory matrix descriptor (cute/arch/mma_sm100_desc.hpp SmemDescriptor): start >> 4 at
// [0,14), leading-dimension byte offset >> 4 at [16,30) (between the two core matrices of a k-step), stride byte offset
// >> 4 at [32,46) (between 8-row groups), version 1 at [46,48)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((saddr >> 4) & 0x3fff) | ((uint64_t)((lbo >> 4) & 0x3fff) << 16) | ((uint64_t)((sbo >> 4) & 0x3fff) << 32) |
         ((uint64_t)1 << 46);
}
// kind::f16 instruction descriptor: D f32 (bit 4), A / B f16 K-major, N >> 3 at [17,23), M >> 4 at [24,29)
__host__ __device__ constexpr uint32_t make_idesc(int m, int n) { return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24); }
__device__ __forceinline__ void mma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
        "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]),
        "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
}  // namespace umma

// BRIDGE: the Brownian-bridge hit test between passes (TrajOwner::pass; d = 1 only)
// RAGGED: checkpoints go to the ragged store (TrajOwner::pass)
template <int D, int H, bool F64, bool FAST, bool BRIDGE = false, bool RAGGED = false>
__global__ void __launch_bounds__(umma_threads<H>(), umma_streams<H>() ? 2 : 4) rollout_fwd_umma_kernel(const float* __restrict__ Wp, const uint8_t* __restrict__ Bimg,
                                                                           const __grid_constant__ FwdArgs A) {
  using namespace umma;
  typedef WideParams<D, H> L;
  constexpr int KSTEPS = H / 16;
  constexpr bool STREAM = umma_streams<H>();
  constexpr int UMMA_ASLOTS = umma_aslots<H>();
  constexpr uint32_t CHUNK = (uint32_t)umma_chunk_bytes<H>();
  extern __shared__ __align__(128) uint8_t umma_smem[];
  uint8_t* const smem = umma_smem;
  uint8_t* sA = smem;                                           // UMMA_ASLOTS x [hi 4 KB | lo 4 KB]
  uint8_t* sB = smem + UMMA_ASLOTS * UMMA_ACHUNK;
  float* sW1 = reinterpret_cast<float*>(sB + (STREAM ? UMMA_STAGES * CHUNK : (uint32_t)umma_image_bytes<H>()));     // [D][H]
  float* sb1 = sW1 + D * H;
  float* sb2 = sb1 + H;
  float* sW3 = sb2 + H;                                                // [D][H]
  __shared__ __align__(8) uint64_t full[UMMA_STAGES], empty[UMMA_STAGES], a_full[UMMA_ASLOTS], a_empty[UMMA_ASLOTS], acc_ready;
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool inject = (A.flags & RLSDE_F_NOISE_INJECTED) != 0;
  const long long lim = inject ? (A.noise_steps < A.n_steps_lim ? A.noise_steps : A.n_steps_lim) : A.n_steps_lim;

  if constexpr (!STREAM) {          // resident weights: the whole image, once
    for (int i = tid; i < (int)(umma_image_bytes<H>() / 16); i += blockDim.x)
      reinterpret_cast<uint4*>(sB)[i] = __ldg(reinterpret_cast<const uint4*>(Bimg) + i);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  for (int i = tid; i < H; i += blockDim.x) {
    sb1[i] = __ldg(Wp + L::o_b1 + i);
    sb2[i] = __ldg(Wp + L::o_b2 + i);
#pragma unroll
    for (int k = 0; k < D; ++k) { sW1[k * H + i] = __ldg(Wp + L::o_W1t + (size_t)k * H + i); sW3[k * H + i] = __ldg(Wp + L::o_W3 + (size_t)k * H + i); }
  }
  if (tid == 0) {
    for (int s = 0; s < UMMA_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int s = 0; s < UMMA_ASLOTS; ++s) { mbar_init(&a_full[s], UMMA_M); mbar_init(&a_empty[s], 1); }
    mbar_init(&acc_ready, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 4) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(umma_tmem_cols<H>()) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = tmem_base_s;

  TrajOwner<D, F64, BRIDGE, RAGGED> T;
  T.init(A);
  const bool owner = warp < 4;
  float b3[D];
#pragma unroll
  for (int k = 0; k < D; ++k) b3[k] = __ldg(Wp + L::o_b3 + k);

  for (unsigned pass = 0;; ++pass) {
    // ---- lane refill (trajectory threads), then the block-wide vote
    if (owner) {
      const unsigned need = __ballot_sync(0xffffffffu, !T.alive && !T.exhausted);
      if (need) {
        unsigned long long base = 0;
        const int leader = __ffs(need) - 1;
        if (lane == leader) base = atomicAdd(A.counter, (unsigned long long)__popc(need));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (!T.alive && !T.exhausted) {
          const long long idx = (long long)base + __popc(need & ((1u << lane) - 1u));
          if (idx < A.K) T.start(A, idx);
          else T.exhausted = true;
        }
      }
    }
    if (!__syncthreads_or(owner && T.alive)) break;
    const uint32_t par = pass & 1u;

    if (owner) {
      // ---- layer 1 for this thread's trajectory -> its row of A (hi / lo), one k-step (16 units = two 16-byte core-matrix
      // rows) per ring slot; the issuer starts the k-step's MMAs as soon as all 128 rows of the slot are in
      float xf[D];
#pragma unroll
      for (int k = 0; k < D; ++k) xf[k] = (float)T.x[k];
      const uint32_t row_off = (uint32_t)((tid >> 3) * 128 + (tid & 7) * 16);
#pragma unroll 1
      for (int ks = 0; ks < KSTEPS; ++ks) {
        const unsigned c = pass * KSTEPS + ks;                    // running k-step index
        const int slot = c % UMMA_ASLOTS;
        if (c >= UMMA_ASLOTS) mbar_wait(&a_empty[slot], ((c / UMMA_ASLOTS) - 1u) & 1u);   // the MMAs that read it have completed
        uint8_t* dst = sA + (size_t)slot * UMMA_ACHUNK + row_off;
#pragma unroll
        for (int kc2 = 0; kc2 < 2; ++kc2) {
          const int kc = 2 * ks + kc2;
          float h[8];
#pragma unroll
          for (int q4 = 0; q4 < 2; ++q4) {
            const float4 bb = *reinterpret_cast<const float4*>(sb1 + 8 * kc + 4 * q4);
            float zz[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
            for (int k = 0; k < D; ++k) {
              const float4 ww = *reinterpret_cast<const float4*>(sW1 + k * H + 8 * kc + 4 * q4);
              zz[0] = fmaf(xf[k], ww.x, zz[0]); zz[1] = fmaf(xf[k], ww.y, zz[1]);
              zz[2] = fmaf(xf[k], ww.z, zz[2]); zz[3] = fmaf(xf[k], ww.w, zz[3]);
            }
            tanh_pair<FAST>(pack2(zz[0], zz[1]), h[4 * q4], h[4 * q4 + 1]);
            tanh_pair<FAST>(pack2(zz[2], zz[3]), h[4 * q4 + 2], h[4 * q4 + 3]);
          }
          uint4 hi, lo;
          split_pair(h[0], h[1], hi.x, lo.x);
          split_pair(h[2], h[3], hi.y, lo.y);
          split_pair(h[4], h[5], hi.z, lo.z);
          split_pair(h[6], h[7], hi.w, lo.w);
          const uint32_t off = (uint32_t)kc2 * (UMMA_M / 8) * 128;
          *reinterpret_cast<uint4*>(dst + off) = hi;
          *reinterpret_cast<uint4*>(dst + UMMA_ACHUNK / 2 + off) = lo;
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");    // generic-proxy writes -> visible to the tensor core
        mbar_arrive(&a_full[slot]);
      }

      // ---- accumulator row -> h2 = tanh(z2 + b2) -> head, all in this thread's registers
      mbar_wait(&acc_ready, par);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      float u[D];
#pragma unroll
      for (int k = 0; k < D; ++k) u[k] = 0.f;
#pragma unroll 1
      for (int cb = 0; cb < H / 32; ++cb) {
        uint32_t r[32];
        ld32(tmem_base + ((uint32_t)(32 * warp) << 16) + (uint32_t)(32 * cb), r);
#pragma unroll
        for (int c4 = 0; c4 < 8; ++c4) {
          const float4 bb = *reinterpret_cast<const float4*>(sb2 + 32 * cb + 4 * c4);
          float h2[4];
          tanh_pair<FAST>(pack2(__uint_as_float(r[4 * c4]) + bb.x, __uint_as_float(r[4 * c4 + 1]) + bb.y), h2[0], h2[1]);
          tanh_pair<FAST>(pack2(__uint_as_float(r[4 * c4 + 2]) + bb.z, __uint_as_float(r[4 * c4 + 3]) + bb.w), h2[2], h2[3]);
#pragma unroll
          for (int k = 0; k < D; ++k) {
            const float4 w3 = *reinterpret_cast<const float4*>(sW3 + k * H + 32 * cb + 4 * c4);
            u[k] = fmaf(w3.x, h2[0], u[k]); u[k] = fmaf(w3.y, h2[1], u[k]);
            u[k] = fmaf(w3.z, h2[2], u[k]); u[k] = fmaf(w3.w, h2[3], u[k]);
          }
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");  // the next pass's MMAs overwrite the accumulator
#pragma unroll
      for (int k = 0; k < D; ++k) u[k] += b3[k];
      if (T.alive) T.pass(A, u, lim);
    } else if (warp == 4) {
      if (lane == 0) {
        constexpr uint32_t idesc = make_idesc(UMMA_M, H);
#pragma unroll 1
        for (int ks = 0; ks < KSTEPS; ++ks) {
          const unsigned c = pass * KSTEPS + ks;                  // running k-step index
          const int s = STREAM ? c % UMMA_STAGES : ks, slot = c % UMMA_ASLOTS;
          mbar_wait(&a_full[slot], (c / UMMA_ASLOTS) & 1u);       // (also orders the previous pass's accumulator reads first)
          if constexpr (STREAM) mbar_wait(&full[s], (c / UMMA_STAGES) & 1u);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t a_base = smem_u32(sA) + (uint32_t)slot * UMMA_ACHUNK;
          const uint64_t ah = make_desc(a_base, (UMMA_M / 8) * 128, 128);
          const uint64_t al = make_desc(a_base + UMMA_ACHUNK / 2, (UMMA_M / 8) * 128, 128);
          const uint64_t bh = make_desc(smem_u32(sB) + (uint32_t)s * CHUNK, (H / 8) * 128, 128);
          const uint64_t bl = make_desc(smem_u32(sB) + (uint32_t)s * CHUNK + CHUNK / 2, (H / 8) * 128, 128);
          mma_f16(tmem_base, ah, bh, idesc, ks > 0 ? 1u : 0u);
          mma_f16(tmem_base, al, bh, idesc, 1u);
          mma_f16(tmem_base, ah, bl, idesc, 1u);
          commit(&a_empty[slot]);                                 // both rings get their slot back once these MMAs have read it
          if constexpr (STREAM) commit(&empty[s]);
        }
        commit(&acc_ready);
      }
    } else if constexpr (STREAM) {
      if (lane == 0) {
#pragma unroll 1
        for (int ks = 0; ks < KSTEPS; ++ks) {
          const unsigned c = pass * KSTEPS + ks;
          const int s = c % UMMA_STAGES;
          if (c >= UMMA_STAGES) mbar_wait(&empty[s], ((c / UMMA_STAGES) - 1u) & 1u);
          mbar_expect_tx(&full[s], CHUNK);
          bulk_g2s(sB + (size_t)s * CHUNK, Bimg + (size_t)ks * CHUNK, CHUNK, &full[s]);
        }
      }
    }
  }
  __syncthreads();
  if (warp == 4) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(umma_tmem_cols<H>()) : "memory");
}

// params_dev: WideParams<D, H> image; image_dev: umma_image_bytes<H>() bytes (both in the caller's workspace).
// RAGGED: the ragged checkpoint store (float32 state only, no Brownian-bridge test: the caller refuses both)
template <int D, int H, bool RAGGED = false>
int launch_rollout_fwd_umma(const float* params_host, float* params_dev, uint8_t* image_dev, const FwdArgs& args, int sm_count,
                            cudaStream_t stream);

}  // namespace rlsde
