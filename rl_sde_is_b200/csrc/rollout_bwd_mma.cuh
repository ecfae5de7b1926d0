// K2m: reverse (adjoint) pass of the REINFORCE surrogate loss with the three 32 x 32 x 32 products of a warp-pass on the
// tensor cores (hidden width 32).
//
// The recursion is rollout_bwd.cuh's (SURVEY.md Appendix C; replaces eff_loss.backward(), reinforce_deterministic_core.py:240).
// Work assignment: one trajectory per lane, processed segment by segment from the last checkpoint backwards.  A round =
// phase A (recompute the segment's states X_j from its checkpoint, identical arithmetic to K1) + phase B (walk the segment
// in reverse: recompute the activations, backpropagate).  All lanes of a warp are in the same phase at the same time, so
// the 32 trajectories stay in lock step although their lengths differ.  dB is regenerated from Philox, never stored.
// Trajectories go to lanes statically, round robin over the length-sorted order, so the gradients are deterministic.
//
// The CUDA-core kernel this one replaced (K2, DESIGN.md) had the same assignment and staged (delta, activation) tiles in
// shared memory for an FFMA2 outer product: 3 717 instructions per warp-pass, 1 564 of them FFMA2, at 62 % issue
// utilisation (profiles/r01/ncu_rollout_bwd_v4.txt).  Here the activations of the 32 trajectories are held in mma.sync FRAGMENT layout across the warp (row = trajectory,
// column = hidden unit), so that
//     Z2  = H1  W2^T      (recomputed forward, layer 2)        M = trajectory, K = in,  N = out
//     dH1 = dZ2 W2                                              M = trajectory, K = out, N = in
//     dW2 += dZ2^T H1     (sum over the warp's trajectories)    M = out,        K = trajectory, N = in
// are 3 x 48 `mma.sync.m16n8k16` instructions (SASS HMMA.16816.F32) and the accumulator layout of one product is the
// A-operand layout of the next (no shared-memory staging; the K = trajectory product takes its operands through
// `movmatrix` transposes).  The scalar per-trajectory work (state, adjoint, Philox increments, a_j) stays with the
// "owner" lane (lane t owns row t) and moves in and out of fragment space with shuffles.
//
// Precision.  B200's legacy warp-level tensor path issues 0.5 HMMA per clock per SM whatever the type
// (profiles/r02/microbench_mma.jsonl): TF32 m16n8k8 = 512 MAC/clk/SM, f16/bf16 m16n8k16 = 1 024 -- against 128 for
// FFMA.  Operands are split x = hi + lo in float16 and each product is hi.hi + hi.lo + lo.hi with fp32 accumulation:
// 22 significand bits per operand while the value stays in float16's normal range, an absolute floor of 2^-25 below
// it.  Activations (|h| <= 1) and weights (O(1)) are split as they are -- the floor is fp32's own rounding of an O(1)
// sum; the deltas dz2, whose magnitude is anybody's guess, are multiplied by a warp-uniform power of two first, taken
// from a bound on max |dz2| (max |a| x max |W3|) and changed only when that bound leaves a window of eight binades;
// the running dW2 sum lives in the same scaled units and is rescaled exactly when the scale moves.  Emulated on the
// reference's gradient fixtures the split costs 1.75e-7 of max |g| against 2.7e-7 for plain fp32 and 1.1e-5 for a
// bfloat16 split (DESIGN.md).  Gradient partials are kept in fp32 over a window of passes and flushed to fp64
// per-warp partials in global memory (the sums cancel heavily: ~1e4 G dB terms); a second kernel adds the warps in
// index order (deterministic, as before).
//
// A pass is run as two half-passes of 16 trajectories (one m16 tile of rows each): all three products separate over
// the row blocks, and the live fragment set halves -- which is what lets three or four blocks share an SM.
#pragma once
#include <cuda_fp16.h>
#include <type_traits>
#include "rollout_bwd.cuh"

namespace rlsde {

constexpr int MMA_H = 32;
constexpr int MMA_FLUSH_EVERY = 64;        // micro-steps between flushes of the fp32 window sums into the fp64 partials

// B operands of products 1 and 2 in fragment order, float16 hi / lo of W2 (pre-scaled like MlpConst::W2t):
//   frag[p][hl][kk][jp][lane] = uint4 {b0, b1 of n-tile 2 jp, b0, b1 of n-tile 2 jp + 1}   for k-chunk kk
//   p = 0: B[k = in][n = out] = W2[out][in]      p = 1: B[k = out][n = in] = W2[out][in]
struct alignas(16) BwdMmaWeights {
  uint32_t frag[2][2][2][2][32][4];
  float w3_max;         // max |W3| (bound for the scale of the deltas)
  float pad[3];
};

template <int D>
inline void pack_bwd_mma_weights(const MlpConst<D, MMA_H>& W, BwdMmaWeights& out) {
  constexpr int H = MMA_H;
  float wmax = 0.f, w3max = 0.f;
  for (int i = 0; i < H; ++i)
    for (int j = 0; j < H; ++j) wmax = fmaxf(wmax, fabsf(W.W2t[i][j]));
  for (int k = 0; k < D; ++k)
    for (int j = 0; j < H; ++j) w3max = fmaxf(w3max, fabsf(W.W3[k][j]));
  (void)wmax;
  out.w3_max = w3max > 0.f ? w3max : 1.0f;
  out.pad[0] = out.pad[1] = out.pad[2] = 0.f;
  pack_w2_frags<D, H>(W, 2, out.frag);
}

// d > 4: the d-sized products run on the tensor cores too, with d padded to one k-chunk / two n-tiles of 16:
//   q = 0: Z1  = X   W1^T    B[k = d][n = hidden] = W1[n][k]  (tanh pre-scale included)   frag[0][hl][jp][lane]
//   q = 1: U   = H2  W3^T    B[k = hidden][n = d] = W3[n][k]                              frag[1][hl][kk][lane]
//   q = 2: dH2 = A   W3      B[k = d][n = hidden] = W3[k][n]                              frag[2][hl][jp][lane]
//   q = 3: dX  = dZ1 W1      B[k = hidden][n = d] = W1[k][n]  (pre-scaled)                frag[3][hl][kk][lane]
// (uint4 = {b0, b1 of the first n-tile, b0, b1 of the second}; rows / columns >= d are zero)
constexpr int MMA_DP = 16;
struct alignas(16) BwdMmaSmall {
  uint32_t frag[4][2][2][32][4];
  int sh1;              // dz1 enters the tensor cores as dz1 2^(dsh - sh1): 2^sh1 >= max_in sum_out |W2[out][in]|
  float a_mul;          // max(1, max |W3|): bound on max(|a|, |dz2|) from sum_k |a_k|
  int pad[2];
};
struct BwdMmaSmallNone { int unused; };
constexpr bool bwd_mma_small(int D) { return D > 4; }
template <int D> struct BwdMmaSmallSel { typedef typename std::conditional<bwd_mma_small(D), BwdMmaSmall, BwdMmaSmallNone>::type type; };

template <int D>
inline void pack_bwd_mma_small(const MlpConst<D, MMA_H>& W, bool fast, BwdMmaSmallNone& out) { (void)W; (void)fast; out.unused = 0; }
template <int D>
inline void pack_bwd_mma_small(const MlpConst<D, MMA_H>& W, bool fast, BwdMmaSmall& out) {
  constexpr int H = MMA_H;
  static_assert(D <= MMA_DP, "state dimension beyond one padded tile");
  // element (k, n) of the B operand of product q
  auto elem = [&](int q, int k, int n) -> float {
    switch (q) {
      case 0: return k < D ? W.W1t[k][n] : 0.f;
      case 1: return n < D ? W.W3[n][k] : 0.f;
      case 2: return k < D ? W.W3[k][n] : 0.f;
      default: return n < D ? W.W1t[n][k] : 0.f;
    }
  };
  for (int q = 0; q < 4; ++q)
    for (int c = 0; c < 2; ++c)             // jp (q = 0, 2: pair of n-tiles, one k-chunk) or kk (q = 1, 3: k-chunk, two n-tiles)
      for (int lane = 0; lane < 32; ++lane) {
        const int g = lane >> 2, t = lane & 3;
        for (int jj = 0; jj < 2; ++jj)
          for (int b = 0; b < 2; ++b) {
            const bool k_small = (q == 0 || q == 2);
            const int n = k_small ? 8 * (2 * c + jj) + g : 8 * jj + g;
            const int k = (k_small ? 0 : 16 * c) + 2 * t + 8 * b;
            uint32_t hi, lo;
            split_pair_host(elem(q, k, n), elem(q, k + 1, n), hi, lo);
            out.frag[q][0][c][lane][2 * jj + b] = hi;
            out.frag[q][1][c][lane][2 * jj + b] = lo;
          }
      }
  const float inv_s = fast ? 1.0f : (float)(1.0 / RLSDE_TWO_LOG2E);
  float cs = 1.0f, w3max = 1.0f;
  for (int i = 0; i < H; ++i) {
    float c = 0.f;
    for (int o = 0; o < H; ++o) c += fabsf(W.W2t[i][o]) * inv_s;
    cs = fmaxf(cs, c);
  }
  for (int k = 0; k < D; ++k)
    for (int j = 0; j < H; ++j) w3max = fmaxf(w3max, fabsf(W.W3[k][j]));
  int sh1 = 0;
  while (sh1 < 20 && ldexpf(1.0f, sh1) < cs) ++sh1;
  out.sh1 = sh1;
  out.a_mul = w3max;
  out.pad[0] = out.pad[1] = 0;
}

// ------------------------------------------------------------------ device helpers
__device__ __forceinline__ uint32_t movm_trans(uint32_t a) {
  uint32_t d;
  asm volatile("movmatrix.sync.aligned.m8n8.trans.b16 %0, %1;" : "=r"(d) : "r"(a));
  return d;
}
// One m16 row tile in accumulator layout v[j][r] (row = g + 8 (r >> 1), column = 8 j + 2 q + (r & 1)), times `scale`,
// as the A operand (hi / lo) of a product whose K dimension is the column index: a[kk][4]
template <bool SCALED>
__device__ __forceinline__ void acc_to_a_frags(const float (&v)[4][4], float scale, uint32_t (&ah)[2][4], uint32_t (&al)[2][4]) {
#pragma unroll
  for (int kk = 0; kk < 2; ++kk)
#pragma unroll
    for (int r4 = 0; r4 < 4; ++r4) {
      const int j = 2 * kk + (r4 >> 1), r = 2 * (r4 & 1);
      if constexpr (SCALED) split_pair(v[j][r] * scale, v[j][r + 1] * scale, ah[kk][r4], al[kk][r4]);
      else split_pair(v[j][r], v[j][r + 1], ah[kk][r4], al[kk][r4]);
    }
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void* smem_ptr) {
  const unsigned addr = (unsigned)__cvta_generic_to_shared(smem_ptr);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
// staging of per-trajectory d-vectors between the owner lanes and fragment space (d > 4): float16 rows of MMA_DP
// entries, hi plane then lo plane, 48-byte pitch (conflict-free for ldmatrix), 32 rows per warp
constexpr int MMA_ROW_PITCH = 48;                              // bytes
constexpr int MMA_PLANE = 32 * MMA_ROW_PITCH;                  // bytes
constexpr int MMA_TILE_PITCH = 24;                             // floats: 16 x 16 result tile going back to the owners
constexpr int MMA_STAGE_BYTES = 2 * MMA_PLANE + 16 * MMA_TILE_PITCH * 4;    // per warp
template <int D>
__device__ __forceinline__ void stage_row(unsigned char* stage, int row, const float (&v)[D], float scale) {
  uint32_t hi[8], lo[8];
#pragma unroll
  for (int p = 0; p < 8; ++p) {
    if (2 * p < D) split_pair(v[2 * p] * scale, (2 * p + 1 < D) ? v[(2 * p + 1 < D) ? 2 * p + 1 : 0] * scale : 0.f, hi[p], lo[p]);
    else { hi[p] = 0u; lo[p] = 0u; }
  }
  uint4* h = reinterpret_cast<uint4*>(stage + row * MMA_ROW_PITCH);
  uint4* l = reinterpret_cast<uint4*>(stage + MMA_PLANE + row * MMA_ROW_PITCH);
  h[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]); h[1] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
  l[0] = make_uint4(lo[0], lo[1], lo[2], lo[3]); l[1] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
}
// rows 16 mt .. 16 mt + 15 of the staged vectors as the A operand (m = trajectory, k = d)
__device__ __forceinline__ void load_staged(const unsigned char* stage, int mt, int lane, uint32_t (&ah)[4], uint32_t (&al)[4]) {
  const int m = lane >> 3, r = lane & 7;
  const unsigned char* a = stage + (16 * mt + r + 8 * (m & 1)) * MMA_ROW_PITCH + 16 * (m >> 1);
  ldmatrix_x4(ah, a);
  ldmatrix_x4(al, a + MMA_PLANE);
}
// acc[0..3] (four n-tiles) += A (one k-chunk, hi + lo) x B (product q of the small-block table: two uint4 per hi / lo)
__device__ __forceinline__ void mma_small_k16(float (&acc)[4][4], const uint32_t (&ah)[4], const uint32_t (&al)[4],
                                              const uint4* __restrict__ sfrag, int q, int lane) {
  const uint4 bh0 = sfrag[((q * 2 + 0) * 2 + 0) * 32 + lane], bh1 = sfrag[((q * 2 + 0) * 2 + 1) * 32 + lane];
  const uint4 bl0 = sfrag[((q * 2 + 1) * 2 + 0) * 32 + lane], bl1 = sfrag[((q * 2 + 1) * 2 + 1) * 32 + lane];
  mma16816(acc[0], ah, bh0.x, bh0.y); mma16816(acc[1], ah, bh0.z, bh0.w);
  mma16816(acc[2], ah, bh1.x, bh1.y); mma16816(acc[3], ah, bh1.z, bh1.w);
  mma16816(acc[0], al, bh0.x, bh0.y); mma16816(acc[1], al, bh0.z, bh0.w);
  mma16816(acc[2], al, bh1.x, bh1.y); mma16816(acc[3], al, bh1.z, bh1.w);
  mma16816(acc[0], ah, bl0.x, bl0.y); mma16816(acc[1], ah, bl0.z, bl0.w);
  mma16816(acc[2], ah, bl1.x, bl1.y); mma16816(acc[3], ah, bl1.z, bl1.w);
}
// acc[0..1] (two n-tiles = the padded d columns) += A (two k-chunks over the hidden units) x B (product q)
__device__ __forceinline__ void mma_small_k32(float (&acc)[2][4], const uint32_t (&ah)[2][4], const uint32_t (&al)[2][4],
                                              const uint4* __restrict__ sfrag, int q, int lane) {
#pragma unroll
  for (int kk = 0; kk < 2; ++kk) {
    const uint4 bh = sfrag[((q * 2 + 0) * 2 + kk) * 32 + lane], bl = sfrag[((q * 2 + 1) * 2 + kk) * 32 + lane];
    mma16816(acc[0], ah[kk], bh.x, bh.y); mma16816(acc[1], ah[kk], bh.z, bh.w);
    mma16816(acc[0], al[kk], bh.x, bh.y); mma16816(acc[1], al[kk], bh.z, bh.w);
    mma16816(acc[0], ah[kk], bl.x, bl.y); mma16816(acc[1], ah[kk], bl.z, bl.w);
  }
}
// the 16 x 16 result tile (two n-tiles in accumulator layout) to shared memory; afterwards row r is read by its owner
__device__ __forceinline__ void store_tile(float* tile, const float (&acc)[2][4], int g, int q) {
#pragma unroll
  for (int nt = 0; nt < 2; ++nt) {
    *reinterpret_cast<float2*>(tile + g * MMA_TILE_PITCH + 8 * nt + 2 * q) = make_float2(acc[nt][0], acc[nt][1]);
    *reinterpret_cast<float2*>(tile + (g + 8) * MMA_TILE_PITCH + 8 * nt + 2 * q) = make_float2(acc[nt][2], acc[nt][3]);
  }
}

#ifndef RLSDE_BWD_MMA_MIN_BLOCKS
#define RLSDE_BWD_MMA_MIN_BLOCKS(D) ((D) <= 2 ? 3 : 2)
#endif
// accumulator fragments of the weight gradients in shared memory ([tile][thread] float4, loaded around the MMAs that add
// to them) instead of registers: 64 registers per thread at d > 4
#ifndef RLSDE_BWD_MMA_SACC
#define RLSDE_BWD_MMA_SACC(D) ((D) > 4)
#endif
constexpr bool bwd_mma_sacc(int D) { return RLSDE_BWD_MMA_SACC(D); }
constexpr int bwd_mma_sacc_tiles(int D) { return !bwd_mma_sacc(D) ? 0 : (bwd_mma_small(D) ? 16 : 8); }
constexpr size_t bwd_mma_dyn_smem(int D, int block) {
  return (bwd_mma_small(D) ? (size_t)(4 * 2 * 2 * 32 * 16 + (block / 32) * MMA_STAGE_BYTES) : (size_t)0) +
         (size_t)bwd_mma_sacc_tiles(D) * block * 16;
}

// Per-warp partial gradient layout = state_dict order (W1 (H,D), b1, W2 (H,H), b2, W3 (D,H), b3), doubles.
// WEIGHTED: per-trajectory coefficients (rollout_bwd.cuh, the comment above em_step_f32); the per-pass scale window below adapts
// to their magnitude as it does to G's
// RAGGED: the checkpoints come from the ragged store (ckpt_slot, rollout_fwd.cuh)
template <int D, bool FAST, bool WEIGHTED = false, bool RAGGED = false>
__global__ void __launch_bounds__(128, RLSDE_BWD_MMA_MIN_BLOCKS(D)) rollout_bwd_mma_kernel(const __grid_constant__ MlpConst<D, MMA_H> W,
                                                                  const __grid_constant__ FwdArgs A,
                                                                  const __grid_constant__ BwdMmaWeights F,
                                                                  const __grid_constant__ typename BwdMmaSmallSel<D>::type FS,
                                                                  double* __restrict__ partial) {
  constexpr int H = MMA_H;
  constexpr unsigned FULL = 0xffffffffu;
  constexpr int P = D * H + H + H * H + H + H * D + D;
  __shared__ uint4 s_wfrag[2 * 2 * 2 * 2 * 32];
  constexpr int DS = bwd_mma_small(D) ? 1 : D;       // (the d-sized weight blocks are MMA fragments at d > 4)
  __shared__ __align__(16) float s_W1[DS][H], s_b1[H], s_b2[H], s_W3[DS][H];
  for (int i = threadIdx.x; i < 2 * 2 * 2 * 2 * 32; i += blockDim.x) s_wfrag[i] = reinterpret_cast<const uint4*>(&F.frag[0][0][0][0][0][0])[i];
  for (int i = threadIdx.x; i < H; i += blockDim.x) {
    s_b1[i] = W.b1[i];
    s_b2[i] = W.b2[i];
#pragma unroll
    for (int k = 0; k < DS; ++k) { s_W1[k][i] = W.W1t[k][i]; s_W3[k][i] = W.W3[k][i]; }
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int g = lane >> 2, q = lane & 3;
  const int warp_in_block = threadIdx.x >> 5;
  const int warps_per_block = blockDim.x >> 5;
  const bool inject = (A.flags & RLSDE_F_NOISE_INJECTED) != 0;
  const bool s_exact = (A.flags & RLSDE_F_STOCH_INT_EXACT) != 0;
  const int C = A.ckpt_every;
  const float inv_s = FAST ? 1.0f : (float)(1.0 / RLSDE_TWO_LOG2E);
  const long long n_lanes = (long long)gridDim.x * blockDim.x;
  const long long gl = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  // row `lane` of a half-pass is held by quad (lane & 7); its member ((lane >> 3) & 1) hands the row's value over
  const int src_lane = ((lane & 7) << 2) | ((lane >> 3) & 1);

  // fp32 window sums (flushed to the fp64 partials every MMA_FLUSH_EVERY micro-steps)
  constexpr bool SACC = bwd_mma_sacc(D);
  constexpr int NTILES = bwd_mma_sacc_tiles(D);   // tile 4 mt + j: dW2; 8 + j: dW3 (DMMA); 12 + 2 mt + nt: dW1 (DMMA)
  float wW2[SACC ? 1 : 2][4][4];               // 2^dsh x dW2[out = 16 mt + g + 8 (r >> 1)][in = 8 j + 2 q + (r & 1)]
  // small blocks, d <= 4: column 8 j + 2 q + e, partial over this thread's rows (16 d floats per thread)
  // d > 4 (DMMA): the d-sized products run on the tensor cores as well (d padded to 16); their gradient blocks are
  // accumulator fragments like dW2
  constexpr bool DMMA = bwd_mma_small(D);
  constexpr int NREG_ACC = DMMA ? 1 : D;
  extern __shared__ __align__(16) unsigned char bwdm_smem[];
  const uint4* const s_sfrag = reinterpret_cast<const uint4*>(bwdm_smem);                    // [4][2][2][32]
  unsigned char* const stage = bwdm_smem + 4 * 2 * 2 * 32 * 16 + warp_in_block * MMA_STAGE_BYTES;
  float* const tile = reinterpret_cast<float*>(stage + 2 * MMA_PLANE);
  float4* const sacc = reinterpret_cast<float4*>(bwdm_smem + (DMMA ? 4 * 2 * 2 * 32 * 16 + warps_per_block * MMA_STAGE_BYTES : 0)) + threadIdx.x;
  auto acc_load = [&](int i, float (&c)[4]) { const float4 t = sacc[(size_t)i * blockDim.x]; c[0] = t.x; c[1] = t.y; c[2] = t.z; c[3] = t.w; };
  auto acc_store = [&](int i, const float (&c)[4]) { sacc[(size_t)i * blockDim.x] = make_float4(c[0], c[1], c[2], c[3]); };
  if constexpr (DMMA) {
    for (int i = threadIdx.x; i < 4 * 2 * 2 * 32; i += blockDim.x)
      reinterpret_cast<uint4*>(bwdm_smem)[i] = reinterpret_cast<const uint4*>(&FS.frag[0][0][0][0][0])[i];
    __syncthreads();
  }
  float wb1[4][2], wb2[4][2], wW1[4][2][NREG_ACC], wW3[4][2][NREG_ACC], wb3[D];
  float wW1a[SACC ? 1 : 2][2][4];   // DMMA: 2^(dsh - sh1) x dW1[hidden = 16 mt + g + 8 (r >> 1)][d = 8 nt + 2 q + (r & 1)]
  float wW3a[SACC ? 1 : 4][4];      // DMMA: 2^dsh x dW3[d = g + 8 (r >> 1)][hidden = 8 j + 2 q + (r & 1)]
  int dsh = 0;                                 // the deltas enter the tensor cores as dz2 2^dsh (warp-uniform)
  if constexpr (SACC) {
    const float zero4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < NTILES; ++i) acc_store(i, zero4);
  } else {
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int r = 0; r < 4; ++r) wW2[mt][j][r] = 0.f;
  }
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      wb1[j][e] = 0.f; wb2[j][e] = 0.f;
#pragma unroll
      for (int k = 0; k < NREG_ACC; ++k) { wW1[j][e][k] = 0.f; wW3[j][e][k] = 0.f; }
    }
  if constexpr (!SACC) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int r = 0; r < 4; ++r) { wW3a[j][r] = 0.f; wW1a[j >> 1][j & 1][r] = 0.f; }
  }
#pragma unroll
  for (int k = 0; k < D; ++k) wb3[k] = 0.f;
  bool flushed_once = false;
  int since_flush = 0;

  const long long gw = (long long)blockIdx.x * warps_per_block + warp_in_block;
  double* const out = partial + gw * P;
  double* const oW1 = out;
  double* const ob1 = oW1 + H * D;
  double* const oW2 = ob1 + H;
  double* const ob2 = oW2 + H * H;
  double* const oW3 = ob2 + H;
  double* const ob3 = oW3 + D * H;

  auto flush = [&]() {
    // dW2: every element is owned by exactly one thread of the warp
    const double un = (double)__uint_as_float((unsigned)(127 - dsh) << 23);
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int j = 0; j < 4; ++j)
      {
        float c[4];
        if constexpr (SACC) {
          const float zero4[4] = {0.f, 0.f, 0.f, 0.f};
          acc_load(4 * mt + j, c);
          acc_store(4 * mt + j, zero4);
        } else {
#pragma unroll
          for (int r = 0; r < 4; ++r) { c[r] = wW2[mt][j][r]; wW2[mt][j][r] = 0.f; }
        }
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
          double* dst = oW2 + (16 * mt + g + 8 * rr) * H + 8 * j + 2 * q;     // (P may be odd: no 16-byte accesses)
          dst[0] = (flushed_once ? dst[0] : 0.0) + un * (double)c[2 * rr];
          dst[1] = (flushed_once ? dst[1] : 0.0) + un * (double)c[2 * rr + 1];
        }
      }
    // the small blocks: sum over the 8 row groups (g), then the g == 0 lanes add their 8 columns
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        float v1 = wb1[j][e], v2 = wb2[j][e];
#pragma unroll
        for (int o = 4; o < 32; o <<= 1) { v1 += __shfl_xor_sync(FULL, v1, o); v2 += __shfl_xor_sync(FULL, v2, o); }
        const int col = 8 * j + 2 * q + e;
        if (g == 0) {
          ob1[col] = (flushed_once ? ob1[col] : 0.0) + (double)v1;
          ob2[col] = (flushed_once ? ob2[col] : 0.0) + (double)v2;
        }
        wb1[j][e] = 0.f; wb2[j][e] = 0.f;
        if constexpr (!DMMA) {
#pragma unroll
          for (int k = 0; k < D; ++k) {
            float a1 = wW1[j][e][k], a3 = wW3[j][e][k];
            wW1[j][e][k] = 0.f; wW3[j][e][k] = 0.f;
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) { a1 += __shfl_xor_sync(FULL, a1, o); a3 += __shfl_xor_sync(FULL, a3, o); }
            if (g == 0) {
              oW1[col * D + k] = (flushed_once ? oW1[col * D + k] : 0.0) + (double)a1;
              oW3[k * H + col] = (flushed_once ? oW3[k * H + col] : 0.0) + (double)a3;
            }
          }
        }
      }
    if constexpr (DMMA) {
      // every element of the fragment accumulators is owned by exactly one thread of the warp (padding rows / columns dropped)
      const double un1 = (double)__uint_as_float((unsigned)(127 - dsh + FS.sh1) << 23);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int mt1 = j >> 1, nt1 = j & 1;
        float c3v[4], c1v[4];
        if constexpr (SACC) {
          const float zero4[4] = {0.f, 0.f, 0.f, 0.f};
          acc_load(8 + j, c3v); acc_load(12 + j, c1v);
          acc_store(8 + j, zero4); acc_store(12 + j, zero4);
        } else {
#pragma unroll
          for (int r = 0; r < 4; ++r) { c3v[r] = wW3a[j][r]; wW3a[j][r] = 0.f; c1v[r] = wW1a[mt1][nt1][r]; wW1a[mt1][nt1][r] = 0.f; }
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int d3 = g + 8 * (r >> 1), c3 = 8 * j + 2 * q + (r & 1);
          if (d3 < D) oW3[d3 * H + c3] = (flushed_once ? oW3[d3 * H + c3] : 0.0) + un * (double)c3v[r];
          const int h1r = 16 * mt1 + g + 8 * (r >> 1), d1 = 8 * nt1 + 2 * q + (r & 1);
          if (d1 < D) oW1[h1r * D + d1] = (flushed_once ? oW1[h1r * D + d1] : 0.0) + un1 * (double)c1v[r];
        }
      }
    }
#pragma unroll
    for (int k = 0; k < D; ++k) {
      float v = wb3[k];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) v += __shfl_xor_sync(FULL, v, o);
      if (lane == 0) ob3[k] = (flushed_once ? ob3[k] : 0.0) + (double)v;
      wb3[k] = 0.f;
    }
    flushed_once = true;
    since_flush = 0;
  };

  bool alive = false;
  long long slot = gl - n_lanes;   // next static assignment: slot += n_lanes, traj = order[slot]
  long long traj = 0;
  int kstar = 0, seg = 0;
  float Gk = 0.f, mG = 0.f;        // WEIGHTED: -cS, -cG
  float lam[D];
  float xs[BWD_MAX_SEG][D];
  constexpr bool CACHE_DB = NoisePlan<D>::BPP > 1;
  float dbs[CACHE_DB ? BWD_MAX_SEG : 1][D];
  float xck[D];                    // checkpoint of the NEXT round, loaded one round ahead (its latency hides behind a round)
  NoiseCache<D> nc;
  nc.reset();
#pragma unroll
  for (int i = 0; i < D; ++i) { lam[i] = 0.f; xck[i] = A.x0_f[i]; }

  for (;;) {
    while (!alive && slot + n_lanes < A.K) {
      slot += n_lanes;
      traj = A.order ? A.order[slot] : slot;
      const int t = A.T[traj];
      if (t >= 0 && ckpt_covered<RAGGED>(A, traj, t)) {
        alive = true; kstar = t; seg = t / C; Gk = ((const float*)A.G)[traj];
        if constexpr (WEIGHTED) { Gk = __fmul_rn(-1.0f, Gk); mG = __fmul_rn(-1.0f, ((const float*)A.S)[traj]); }
        nc.reset();
#pragma unroll
        for (int i = 0; i < D; ++i) { lam[i] = 0.f; xck[i] = A.path[ckpt_slot<RAGGED>(A, traj, seg) * D + i]; }
      }
    }
    if (!__any_sync(FULL, alive)) break;
    const int seg_start = seg * C;
    const int seg_len = alive ? ((kstar + 1 - seg_start) < C ? (kstar + 1 - seg_start) : C) : 0;
#pragma unroll
    for (int i = 0; i < D; ++i) xs[0][i] = xck[i];
    if (alive && seg > 0) {
#pragma unroll
      for (int i = 0; i < D; ++i)
        xck[i] = RAGGED ? A.path[ckpt_slot<RAGGED>(A, traj, seg - 1) * D + i]
                        : A.path[((long long)traj * A.ckpt_stride + seg - 1) * D + i];     // (the dense kernels' code as it was)
    }

    for (int t = 0; t < 2 * C - 1; ++t) {
      const bool phase_a = t < C - 1;
      const int s = phase_a ? t : (2 * C - 2 - t);
      const bool ok = alive && s < seg_len;
      const int j = seg_start + s;
      float x[D], dB[D];
#pragma unroll
      for (int i = 0; i < D; ++i) x[i] = xs[s][i];
      if constexpr (CACHE_DB) {
        // several Philox blocks per pass: the segment's forward sweep keeps its increments for the reverse sweep
        if (!inject && !phase_a && s < C - 1) {
#pragma unroll
          for (int i = 0; i < D; ++i) dB[i] = dbs[s][i];
        } else {
          nc.get(A, inject, ok, traj, j, dB);
          if (phase_a) {
#pragma unroll
            for (int i = 0; i < D; ++i) dbs[s][i] = dB[i];
          }
        }
      } else {
        nc.get(A, inject, ok, traj, j, dB);
      }
      float u[D];
#pragma unroll
      for (int i = 0; i < D; ++i) u[i] = 0.f;

      if constexpr (DMMA) {
        // the states of the warp's 32 trajectories as float16 hi / lo rows (A operand of layer 1, B operand of dW1)
        __syncwarp();
        stage_row<D>(stage, lane, x, 1.0f);
        __syncwarp();
      }

#pragma unroll 1
      for (int mt = 0; mt < 2; ++mt) {
        const bool my_half = (lane >> 4) == mt;
        // ---- forward of rows 16 mt + g (+ 8) in fragment space
        float xr[2][DMMA ? 1 : D];
        uint32_t xah[4], xal[4];
        float h1[4][4];
        if constexpr (DMMA) {
          load_staged(stage, mt, lane, xah, xal);
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            const float2 bb = *reinterpret_cast<const float2*>(&s_b1[8 * jj + 2 * q]);
            h1[jj][0] = bb.x; h1[jj][1] = bb.y; h1[jj][2] = bb.x; h1[jj][3] = bb.y;
          }
          mma_small_k16(h1, xah, xal, s_sfrag, 0, lane);
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            tanh_pair<FAST>(pack2(h1[jj][0], h1[jj][1]), h1[jj][0], h1[jj][1]);
            tanh_pair<FAST>(pack2(h1[jj][2], h1[jj][3]), h1[jj][2], h1[jj][3]);
          }
        } else {
#pragma unroll
          for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int k = 0; k < D; ++k) xr[h][k] = __shfl_sync(FULL, x[k], 16 * mt + g + 8 * h);
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            const float2 bb = *reinterpret_cast<const float2*>(&s_b1[8 * jj + 2 * q]);
            float z[4] = {bb.x, bb.y, bb.x, bb.y};
#pragma unroll
            for (int k = 0; k < D; ++k) {
              const float2 ww = *reinterpret_cast<const float2*>(&s_W1[k][8 * jj + 2 * q]);
              z[0] = fmaf(xr[0][k], ww.x, z[0]); z[1] = fmaf(xr[0][k], ww.y, z[1]);
              z[2] = fmaf(xr[1][k], ww.x, z[2]); z[3] = fmaf(xr[1][k], ww.y, z[3]);
            }
            tanh_pair<FAST>(pack2(z[0], z[1]), h1[jj][0], h1[jj][1]);
            tanh_pair<FAST>(pack2(z[2], z[3]), h1[jj][2], h1[jj][3]);
          }
        }
        uint32_t a1h[2][4], a1l[2][4];
        acc_to_a_frags<false>(h1, 1.0f, a1h, a1l);
        float h2[4][4];
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          const float2 bb = *reinterpret_cast<const float2*>(&s_b2[8 * jj + 2 * q]);
          h2[jj][0] = bb.x; h2[jj][1] = bb.y; h2[jj][2] = bb.x; h2[jj][3] = bb.y;
        }
        mma_product_w(h2, a1h, a1l, s_wfrag, 0, lane);
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          tanh_pair<FAST>(pack2(h2[jj][0], h2[jj][1]), h2[jj][0], h2[jj][1]);
          tanh_pair<FAST>(pack2(h2[jj][2], h2[jj][3]), h2[jj][2], h2[jj][3]);
        }
        uint32_t h2h[2][4], h2l[2][4];                 // DMMA: h2 as an operand (head, dW3)
        if constexpr (DMMA) {
          acc_to_a_frags<false>(h2, 1.0f, h2h, h2l);
          float uacc[2][4];
#pragma unroll
          for (int nt = 0; nt < 2; ++nt)
#pragma unroll
            for (int r = 0; r < 4; ++r) uacc[nt][r] = 0.f;
          mma_small_k32(uacc, h2h, h2l, s_sfrag, 1, lane);
          store_tile(tile, uacc, g, q);
          __syncwarp();
          if (my_half) {
#pragma unroll
            for (int k = 0; k < D; ++k) u[k] = tile[(lane & 15) * MMA_TILE_PITCH + k] + W.b3[k];
          }
          __syncwarp();
        } else {
          // head: u[row][k] = b3[k] + sum_col W3[k][col] h2[row][col]  (this thread's 8 columns, then the quad)
          float up[2][D];
#pragma unroll
          for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int k = 0; k < D; ++k) up[h][k] = 0.f;
#pragma unroll
          for (int jj = 0; jj < 4; ++jj)
#pragma unroll
            for (int k = 0; k < D; ++k) {
              const float2 w3 = *reinterpret_cast<const float2*>(&s_W3[k][8 * jj + 2 * q]);
              up[0][k] = fmaf(w3.x, h2[jj][0], up[0][k]); up[0][k] = fmaf(w3.y, h2[jj][1], up[0][k]);
              up[1][k] = fmaf(w3.x, h2[jj][2], up[1][k]); up[1][k] = fmaf(w3.y, h2[jj][3], up[1][k]);
            }
#pragma unroll
          for (int k = 0; k < D; ++k) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              up[h][k] += __shfl_xor_sync(FULL, up[h][k], 1);
              up[h][k] += __shfl_xor_sync(FULL, up[h][k], 2);
            }
            const float got = __shfl_sync(FULL, (q & 1) ? up[1][k] : up[0][k], src_lane) + W.b3[k];
            if (my_half) u[k] = got;
          }
        }
        if (phase_a) continue;      // (warp-uniform) the segment's forward sweep needs the action only

        // ---- reverse: a_j at the owner lanes of this half
        float a[D];
        float asum = 0.f;
#pragma unroll
        for (int i = 0; i < D; ++i) {
          float v = 0.f;
          if (ok && my_half) {
            const bool incl = s_exact ? (j < kstar) : true;
            if constexpr (WEIGHTED) v = (j < kstar ? __fmul_rn(mG, u[i]) * A.dt_f : 0.f) - (incl ? Gk * dB[i] : 0.f) + A.sigma_f * A.dt_f * lam[i];
            else v = (j < kstar ? u[i] * A.dt_f : 0.f) - (incl ? Gk * dB[i] : 0.f) + A.sigma_f * A.dt_f * lam[i];
          }
          a[i] = v;
          asum += fabsf(v);
          wb3[i] += v;
        }
        {
          // |dz2| <= sum_k |a_k| max |W3|.  Keep 2^dsh x that bound inside [2^7, 2^15) (float16 tops out at 2^16); when it
          // leaves the window, move the scale and rescale the running sums that live in scaled units (a power of two: exact)
          float mul = F.w3_max;
          if constexpr (DMMA) mul = FS.a_mul;          // the a_k themselves go through float16 too
          const unsigned bits = __reduce_max_sync(FULL, __float_as_uint(asum * mul));   // non-negative floats order as integers
          if (bits != 0u) {
            const int e1 = (int)(bits >> 23) - 126;            // bound < 2^e1
            if (e1 + dsh > 15 || e1 + dsh < 8) {
              int nsh = 14 - e1;
              nsh = nsh > 100 ? 100 : (nsh < -100 ? -100 : nsh);
              const float r = __uint_as_float((unsigned)(127 + nsh - dsh) << 23);
              if constexpr (SACC) {
#pragma unroll
                for (int i = 0; i < NTILES; ++i) {
                  float c[4];
                  acc_load(i, c);
#pragma unroll
                  for (int rr = 0; rr < 4; ++rr) c[rr] *= r;
                  acc_store(i, c);
                }
              } else {
#pragma unroll
                for (int m2 = 0; m2 < 2; ++m2)
#pragma unroll
                  for (int jj = 0; jj < 4; ++jj)
#pragma unroll
                    for (int rr = 0; rr < 4; ++rr) wW2[m2][jj][rr] *= r;
                if constexpr (DMMA) {
#pragma unroll
                  for (int jj = 0; jj < 4; ++jj)
#pragma unroll
                    for (int rr = 0; rr < 4; ++rr) { wW3a[jj][rr] *= r; wW1a[jj >> 1][jj & 1][rr] *= r; }
                }
              }
              dsh = nsh;
            }
          }
        }
        const float dscale = __uint_as_float((unsigned)(127 + dsh) << 23);
        const float dunscale = __uint_as_float((unsigned)(127 - dsh) << 23);
        float dz2[4][4];
        uint32_t a2h[2][4], a2l[2][4];
        float ar[2][DMMA ? 1 : D];
        if constexpr (DMMA) {
          // a 2^dsh of this half's rows through the staging rows (their states are in registers by now)
          if (my_half) stage_row<D>(stage, lane, a, dscale);
          __syncwarp();
          uint32_t aah[4], aal[4];
          load_staged(stage, mt, lane, aah, aal);
          // dh2 = a W3 (scaled); dz2 = dh2 (1 - h2^2); db2 += dz2
#pragma unroll
          for (int jj = 0; jj < 4; ++jj)
#pragma unroll
            for (int r = 0; r < 4; ++r) dz2[jj][r] = 0.f;
          mma_small_k16(dz2, aah, aal, s_sfrag, 2, lane);
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
#pragma unroll
            for (int r = 0; r < 4; ++r) dz2[jj][r] *= fmaf(-h2[jj][r], h2[jj][r], 1.0f);
#pragma unroll
            for (int e = 0; e < 2; ++e) wb2[jj][e] = fmaf(dz2[jj][e] + dz2[jj][2 + e], dunscale, wb2[jj][e]);
          }
          acc_to_a_frags<false>(dz2, 1.0f, a2h, a2l);
          // dW3 += a^T h2 over this half's 16 trajectories (m = d, k = trajectory, n = hidden), in the scaled units of a
          {
            uint32_t th[4], tl[4];
            th[0] = movm_trans(aah[0]); th[1] = movm_trans(aah[2]); th[2] = movm_trans(aah[1]); th[3] = movm_trans(aah[3]);
            tl[0] = movm_trans(aal[0]); tl[1] = movm_trans(aal[2]); tl[2] = movm_trans(aal[1]); tl[3] = movm_trans(aal[3]);
            uint32_t bh[4][2], bl[4][2];
#pragma unroll
            for (int j3 = 0; j3 < 4; ++j3) {
              bh[j3][0] = movm_trans(h2h[j3 >> 1][0 | ((j3 & 1) << 1)]);
              bh[j3][1] = movm_trans(h2h[j3 >> 1][1 | ((j3 & 1) << 1)]);
              bl[j3][0] = movm_trans(h2l[j3 >> 1][0 | ((j3 & 1) << 1)]);
              bl[j3][1] = movm_trans(h2l[j3 >> 1][1 | ((j3 & 1) << 1)]);
            }
            auto run = [&](float (&c)[4][4]) {
#pragma unroll
              for (int j3 = 0; j3 < 4; ++j3) mma16816(c[j3], th, bh[j3][0], bh[j3][1]);
#pragma unroll
              for (int j3 = 0; j3 < 4; ++j3) mma16816(c[j3], tl, bh[j3][0], bh[j3][1]);
#pragma unroll
              for (int j3 = 0; j3 < 4; ++j3) mma16816(c[j3], th, bl[j3][0], bl[j3][1]);
            };
            if constexpr (SACC) {
              float c[4][4];
#pragma unroll
              for (int j3 = 0; j3 < 4; ++j3) acc_load(8 + j3, c[j3]);
              run(c);
#pragma unroll
              for (int j3 = 0; j3 < 4; ++j3) acc_store(8 + j3, c[j3]);
            } else {
              run(wW3a);
            }
          }
        } else {
#pragma unroll
          for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int k = 0; k < D; ++k) ar[h][k] = __shfl_sync(FULL, a[k], 16 * mt + g + 8 * h);
          // dz2 = (W3^T a) (1 - h2^2); dW3 += a (x) h2; db2 += dz2
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            float2 w3[D];
#pragma unroll
            for (int k = 0; k < D; ++k) w3[k] = *reinterpret_cast<const float2*>(&s_W3[k][8 * jj + 2 * q]);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const float hv0 = h2[jj][e], hv1 = h2[jj][2 + e];          // rows g and g + 8
              float dh0 = 0.f, dh1 = 0.f;
#pragma unroll
              for (int k = 0; k < D; ++k) {
                const float w = e ? w3[k].y : w3[k].x;
                dh0 = fmaf(ar[0][k], w, dh0);
                dh1 = fmaf(ar[1][k], w, dh1);
                wW3[jj][e][k] += fmaf(ar[0][k], hv0, ar[1][k] * hv1);
              }
              const float dzA = dh0 * fmaf(-hv0, hv0, 1.0f), dzB = dh1 * fmaf(-hv1, hv1, 1.0f);
              wb2[jj][e] += dzA + dzB;
              dz2[jj][e] = dzA;
              dz2[jj][2 + e] = dzB;
            }
          }
          acc_to_a_frags<true>(dz2, dscale, a2h, a2l);
        }
        // dh1 = dz2 W2  -> dz1 = dh1 (1 - h1^2)   (the weights carry the tanh pre-scale: inv_s)
        float dz1[4][4];
#pragma unroll
        for (int jj = 0; jj < 4; ++jj)
#pragma unroll
          for (int r = 0; r < 4; ++r) dz1[jj][r] = 0.f;
        mma_product_w(dz1, a2h, a2l, s_wfrag, 1, lane);
        if constexpr (DMMA) {
          // dz1 stays in scaled units, 2^(dsh - sh1): it is an operand of dX = dZ1 W1 and of dW1 += dZ1^T X
          const float dn = __uint_as_float((unsigned)(127 - FS.sh1) << 23) * inv_s;
          const float un1 = __uint_as_float((unsigned)(127 - dsh + FS.sh1) << 23);
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
#pragma unroll
            for (int r = 0; r < 4; ++r) dz1[jj][r] *= dn * fmaf(-h1[jj][r], h1[jj][r], 1.0f);
#pragma unroll
            for (int e = 0; e < 2; ++e) wb1[jj][e] = fmaf(dz1[jj][e] + dz1[jj][2 + e], un1, wb1[jj][e]);
          }
          uint32_t d1h[2][4], d1l[2][4];
          acc_to_a_frags<false>(dz1, 1.0f, d1h, d1l);
          float dxacc[2][4];
#pragma unroll
          for (int nt = 0; nt < 2; ++nt)
#pragma unroll
            for (int r = 0; r < 4; ++r) dxacc[nt][r] = 0.f;
          mma_small_k32(dxacc, d1h, d1l, s_sfrag, 3, lane);
          store_tile(tile, dxacc, g, q);
          __syncwarp();
          if (ok && my_half) {
            const float unx = un1 * inv_s;
#pragma unroll
            for (int k = 0; k < D; ++k) {
              const float dx = tile[(lane & 15) * MMA_TILE_PITCH + k] * unx;
              const float hess = A.c4a_f[k] * fmaf(3.0f * x[k], x[k], -1.0f);
              lam[k] = fmaf(lam[k], fmaf(-A.dt_f, hess, 1.0f), dx);
            }
          }
          // dW1 += dz1^T x over this half's 16 trajectories (m = hidden, k = trajectory, n = d)
          {
            uint32_t bxh[2][2], bxl[2][2];
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
              bxh[nt][0] = movm_trans(xah[2 * nt]); bxh[nt][1] = movm_trans(xah[2 * nt + 1]);
              bxl[nt][0] = movm_trans(xal[2 * nt]); bxl[nt][1] = movm_trans(xal[2 * nt + 1]);
            }
#pragma unroll
            for (int mt3 = 0; mt3 < 2; ++mt3) {
              uint32_t ah[4], al[4];
              ah[0] = movm_trans(d1h[mt3][0]); ah[1] = movm_trans(d1h[mt3][2]);
              ah[2] = movm_trans(d1h[mt3][1]); ah[3] = movm_trans(d1h[mt3][3]);
              al[0] = movm_trans(d1l[mt3][0]); al[1] = movm_trans(d1l[mt3][2]);
              al[2] = movm_trans(d1l[mt3][1]); al[3] = movm_trans(d1l[mt3][3]);
              auto run = [&](float (&c)[2][4]) {
#pragma unroll
                for (int nt = 0; nt < 2; ++nt) mma16816(c[nt], ah, bxh[nt][0], bxh[nt][1]);
#pragma unroll
                for (int nt = 0; nt < 2; ++nt) mma16816(c[nt], al, bxh[nt][0], bxh[nt][1]);
#pragma unroll
                for (int nt = 0; nt < 2; ++nt) mma16816(c[nt], ah, bxl[nt][0], bxl[nt][1]);
              };
              if constexpr (SACC) {
                float c[2][4];
                acc_load(12 + 2 * mt3, c[0]); acc_load(13 + 2 * mt3, c[1]);
                run(c);
                acc_store(12 + 2 * mt3, c[0]); acc_store(13 + 2 * mt3, c[1]);
              } else {
                run(wW1a[mt3]);
              }
            }
          }
          __syncwarp();
        } else {
          const float un = dunscale * inv_s;
          float dxp[2][D];
#pragma unroll
          for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int k = 0; k < D; ++k) dxp[h][k] = 0.f;
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            float2 ww[D];
#pragma unroll
            for (int k = 0; k < D; ++k) ww[k] = *reinterpret_cast<const float2*>(&s_W1[k][8 * jj + 2 * q]);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const float hv0 = h1[jj][e], hv1 = h1[jj][2 + e];
              const float dzA = dz1[jj][e] * un * fmaf(-hv0, hv0, 1.0f), dzB = dz1[jj][2 + e] * un * fmaf(-hv1, hv1, 1.0f);
              wb1[jj][e] += dzA + dzB;
#pragma unroll
              for (int k = 0; k < D; ++k) {
                wW1[jj][e][k] += fmaf(dzA, xr[0][k], dzB * xr[1][k]);
                const float w = e ? ww[k].y : ww[k].x;
                dxp[0][k] = fmaf(w, dzA, dxp[0][k]);
                dxp[1][k] = fmaf(w, dzB, dxp[1][k]);
              }
            }
          }
          // state adjoint at the owner lane:  lambda_j = (1 - dt hess) lambda_{j+1} + W1^T dz1 (the pre-scale again: inv_s)
#pragma unroll
          for (int k = 0; k < D; ++k) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              dxp[h][k] += __shfl_xor_sync(FULL, dxp[h][k], 1);
              dxp[h][k] += __shfl_xor_sync(FULL, dxp[h][k], 2);
            }
            const float dx = __shfl_sync(FULL, (q & 1) ? dxp[1][k] : dxp[0][k], src_lane) * inv_s;
            if (ok && my_half) {
              const float hess = A.c4a_f[k] * fmaf(3.0f * x[k], x[k], -1.0f);
              lam[k] = fmaf(lam[k], fmaf(-A.dt_f, hess, 1.0f), dx);
            }
          }
        }
        // dW2 += dz2^T h1 over this half's 16 trajectories (K = trajectory): operands are 8x8 transposes of the
        // fragments built above; the sum runs in the scaled units of dz2
        {
          uint32_t bh[4][2], bl[4][2];     // B[k = trajectory][n = in 8 j3 + g]
#pragma unroll
          for (int j3 = 0; j3 < 4; ++j3) {
            bh[j3][0] = movm_trans(a1h[j3 >> 1][0 | ((j3 & 1) << 1)]);
            bh[j3][1] = movm_trans(a1h[j3 >> 1][1 | ((j3 & 1) << 1)]);
            bl[j3][0] = movm_trans(a1l[j3 >> 1][0 | ((j3 & 1) << 1)]);
            bl[j3][1] = movm_trans(a1l[j3 >> 1][1 | ((j3 & 1) << 1)]);
          }
#pragma unroll
          for (int mt3 = 0; mt3 < 2; ++mt3) {
            uint32_t ah[4], al[4];         // A[m = out 16 mt3 + g (+ 8)][k = trajectory]
            ah[0] = movm_trans(a2h[mt3][0]); ah[1] = movm_trans(a2h[mt3][2]);
            ah[2] = movm_trans(a2h[mt3][1]); ah[3] = movm_trans(a2h[mt3][3]);
            al[0] = movm_trans(a2l[mt3][0]); al[1] = movm_trans(a2l[mt3][2]);
            al[2] = movm_trans(a2l[mt3][1]); al[3] = movm_trans(a2l[mt3][3]);
            // the four accumulators take turns: consecutive HMMAs are independent
            auto run = [&](float (&c)[4][4]) {
#pragma unroll
              for (int j3 = 0; j3 < 4; ++j3) mma16816(c[j3], ah, bh[j3][0], bh[j3][1]);
#pragma unroll
              for (int j3 = 0; j3 < 4; ++j3) mma16816(c[j3], al, bh[j3][0], bh[j3][1]);
#pragma unroll
              for (int j3 = 0; j3 < 4; ++j3) mma16816(c[j3], ah, bl[j3][0], bl[j3][1]);
            };
            if constexpr (SACC) {
              float c[4][4];
#pragma unroll
              for (int j3 = 0; j3 < 4; ++j3) acc_load(4 * mt3 + j3, c[j3]);
              run(c);
#pragma unroll
              for (int j3 = 0; j3 < 4; ++j3) acc_store(4 * mt3 + j3, c[j3]);
            } else {
              run(wW2[mt3]);
            }
          }
        }
      }
      if (phase_a) {
        // X_{j+1} from X_j (same association as K1; u agrees with K1's to rounding, so the recomputed states follow the
        // forward pass's states to ~1e-7 -- the hit index is taken from the forward pass, not re-detected)
        if (alive && s + 1 < seg_len) em_step_f32<D>(A, x, u, dB);
#pragma unroll
        for (int i = 0; i < D; ++i) xs[s + 1][i] = x[i];
        continue;
      }
      if (++since_flush >= MMA_FLUSH_EVERY) flush();
    }
    if (alive) {
      --seg;
      if (seg < 0) alive = false;
    }
  }
  flush();
}

// grad[p] (+)= scale * sum_w partial[w][p], warps in index order
static __global__ void bwd_reduce64_kernel(const double* __restrict__ partial, int n_warps, int P, float scale,
                                           float* __restrict__ grad, int accumulate) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  double acc = 0.0;
  for (int w = 0; w < n_warps; ++w) acc += partial[(long long)w * P + p];
  const float gv = (float)(acc * (double)scale);
  grad[p] = accumulate ? grad[p] + gv : gv;
}

// join: if non-null, the stream waits for this event between the rollout kernel and the reduction that adds into `grad`
// (the warp-per-trajectory kernel working on the longest trajectories on a second stream writes `grad` first)
template <int D, bool WEIGHTED = false, bool RAGGED = false>
int launch_rollout_bwd_mma(const float* params_host, const FwdArgs& args, float scale, float* grad, void* partial,
                           int sm_count, cudaStream_t stream, cudaEvent_t join);

}  // namespace rlsde
