// Policy evaluation of the forward rollout with the 32 x 32 hidden layer on the warp-level tensor cores (hidden width 32).
//
// K1 keeps one trajectory per lane and evaluates its policy with FFMA2 against weights from the constant bank: the
// 32 x 32 layer is 512 of the 544 FFMA2 of a warp-pass and ~300 LDCU feed them (profiles/r02/sass/fwd_d1_h32.txt), so
// the FMA pipe, the MUFU pipe (the precise tanh: EX2 + RCP per activation) and issue were all ~70-75 % busy.  Here the
// warp's 32 trajectories form the rows of one 32 x 32 tile and layer 2 is 48 `mma.sync.m16n8k16` (SASS HMMA.16816.F32):
// two m16 tiles x four n8 tiles x two k16 chunks x three products hi.hi + lo.hi + hi.lo of float16 splits with fp32
// accumulation (the split K2m uses, rollout_bwd_mma.cuh).  Layer 1 and the head stay on the CUDA cores, in fragment
// layout, so nothing goes through shared memory except the constant tables.
//
// Row <-> lane mapping.  Row g + 8 b of the tile (g = lane >> 2, b = 0..3) is the trajectory of lane 4 g + b.  A lane's
// fragment rows are g, g + 8, g + 16, g + 24 -- the four trajectories of its own quad -- and its fragment columns are the
// same eight hidden units 8 j + 2 q + e (j = 0..3, e = 0, 1, q = lane & 3) in the A operand of layer 2 and in the
// accumulators.  So a lane computes layer 1 for its 4 rows x 8 columns (32 activations, as in K1), the head is 8 FMAs
// per row over the lane's columns, and a two-step reduce-scatter inside the quad leaves each lane with its own
// trajectory's action: row b's sum is (p0 + p2) + (p1 + p3) of the four lanes' partials in every lane that forms it.
//
// Every row's result depends only on that row's input and the weights.  The warp-per-trajectory kernel continues a
// handed-over trajectory by putting its state in all 32 rows (rollout_warp.cuh, RESUME): it gets K1's action bit for bit
// (and evaluates only what differs, REPL below).
#pragma once
#include <cmath>
#include <cstring>
#include <cuda_fp16.h>
#include "common.cuh"

namespace rlsde {

// ------------------------------------------------------------------ float16 split helpers (shared with K2m and K1u)
inline uint16_t f32_to_f16_bits(float f) {      // round to nearest even, host side
  uint32_t x;
  memcpy(&x, &f, 4);
  const uint32_t sign = (x >> 16) & 0x8000u;
  const int32_t exp = (int32_t)((x >> 23) & 0xff) - 127 + 15;
  uint32_t man = x & 0x7fffffu;
  if (((x >> 23) & 0xff) == 0xff) return (uint16_t)(sign | 0x7c00u | (man ? 0x200u : 0));
  if (exp >= 31) return (uint16_t)(sign | 0x7c00u);
  if (exp <= 0) {
    if (exp < -10) return (uint16_t)sign;
    man |= 0x800000u;
    const int shift = 14 - exp;
    uint32_t h = man >> shift;
    const uint32_t rem = man & ((1u << shift) - 1u), half = 1u << (shift - 1);
    if (rem > half || (rem == half && (h & 1u))) ++h;
    return (uint16_t)(sign | h);
  }
  uint32_t h = ((uint32_t)exp << 10) | (man >> 13);
  const uint32_t rem = man & 0x1fffu;
  if (rem > 0x1000u || (rem == 0x1000u && (h & 1u))) ++h;
  return (uint16_t)(sign | h);
}
inline float f16_bits_to_f32(uint16_t h) {
  const uint32_t sign = (uint32_t)(h & 0x8000u) << 16;
  uint32_t exp = (h >> 10) & 0x1f, man = h & 0x3ffu;
  uint32_t x;
  if (exp == 0) {
    if (man == 0) { x = sign; }
    else {
      int e = -1;
      do { ++e; man <<= 1; } while (!(man & 0x400u));
      x = sign | ((uint32_t)(127 - 15 - e) << 23) | ((man & 0x3ffu) << 13);
    }
  } else if (exp == 31) {
    x = sign | 0x7f800000u | (man << 13);
  } else {
    x = sign | ((exp - 15 + 127) << 23) | (man << 13);
  }
  float f;
  memcpy(&f, &x, 4);
  return f;
}
// host: a, b -> float16 pairs hi, lo with a ~ hi + lo (a in the low half)
inline void split_pair_host(float a, float b, uint32_t& hi, uint32_t& lo) {
  const uint16_t ah = f32_to_f16_bits(a), bh = f32_to_f16_bits(b);
  const uint16_t al = f32_to_f16_bits(a - f16_bits_to_f32(ah)), bl = f32_to_f16_bits(b - f16_bits_to_f32(bh));
  hi = (uint32_t)ah | ((uint32_t)bh << 16);
  lo = (uint32_t)al | ((uint32_t)bl << 16);
}

// W2 (pre-scaled like MlpConst::W2t) as the B operand of the products H W2^T (k = in, n = out) and dZ2 W2 (k = out,
// n = in), float16 hi / lo in fragment order:
//   frag[p][hl][kk][jp][lane] = {b0, b1 of n-tile 2 jp, b0, b1 of n-tile 2 jp + 1}   for k-chunk kk
// (p = 0 is all the forward rollout needs; the reverse pass, K2m, uses both)
template <int D, int H>
inline void pack_w2_frags(const MlpConst<D, H>& W, int n_products, uint32_t (*frag)[2][2][2][32][4]) {
  static_assert(H == 32, "one 32 x 32 tile");
  auto w = [&](int o, int i) { return W.W2t[i][o]; };            // W2[out][in]
  for (int p = 0; p < n_products; ++p)
    for (int kk = 0; kk < 2; ++kk)
      for (int jp = 0; jp < 2; ++jp)
        for (int lane = 0; lane < 32; ++lane) {
          const int g = lane >> 2, q = lane & 3;
          for (int jj = 0; jj < 2; ++jj) {
            const int n = 8 * (2 * jp + jj) + g, k0 = 16 * kk + 2 * q;
            for (int b = 0; b < 2; ++b) {
              const int k = k0 + 8 * b;
              const float e0 = p == 0 ? w(n, k) : w(k, n), e1 = p == 0 ? w(n, k + 1) : w(k + 1, n);
              split_pair_host(e0, e1, frag[p][0][kk][jp][lane][2 * jj + b], frag[p][1][kk][jp][lane][2 * jj + b]);
            }
          }
        }
}

__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// x0, x1 -> float16 pairs hi, lo with x ~ hi + lo  (x0 in the low half).  The residual x - hi is one packed subtraction
// (FADD2; it rounds like the two scalar ones): F2FP, 2 HADD2.F32, FADD2, F2FP per pair.
__device__ __forceinline__ void split_pair(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(x0, x1);
  const float2 hf = __half22float2(h);
  float l0, l1;
  unpack2(sub2(pack2(x0, x1), pack2(hf.x, hf.y)), l0, l1);
  const __half2 l = __floats2half2_rn(l0, l1);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}
// acc[j] += A (hi + lo) x B (hi + lo from the shared-memory fragment table of product p), dropping lo x lo.
// Issue order: the four accumulators take turns, so consecutive HMMAs are independent (dependent ones are 4 apart).
__device__ __forceinline__ void mma_product_w(float (&acc)[4][4], const uint32_t (&ah)[2][4], const uint32_t (&al)[2][4],
                                              const uint4* __restrict__ wfrag, int p, int lane) {
#pragma unroll
  for (int kk = 0; kk < 2; ++kk) {
    const uint4 bh0 = wfrag[(((p * 2 + 0) * 2 + kk) * 2 + 0) * 32 + lane];
    const uint4 bh1 = wfrag[(((p * 2 + 0) * 2 + kk) * 2 + 1) * 32 + lane];
    const uint4 bl0 = wfrag[(((p * 2 + 1) * 2 + kk) * 2 + 0) * 32 + lane];
    const uint4 bl1 = wfrag[(((p * 2 + 1) * 2 + kk) * 2 + 1) * 32 + lane];
    mma16816(acc[0], ah[kk], bh0.x, bh0.y); mma16816(acc[1], ah[kk], bh0.z, bh0.w);
    mma16816(acc[2], ah[kk], bh1.x, bh1.y); mma16816(acc[3], ah[kk], bh1.z, bh1.w);
    mma16816(acc[0], al[kk], bh0.x, bh0.y); mma16816(acc[1], al[kk], bh0.z, bh0.w);
    mma16816(acc[2], al[kk], bh1.x, bh1.y); mma16816(acc[3], al[kk], bh1.z, bh1.w);
    mma16816(acc[0], ah[kk], bl0.x, bl0.y); mma16816(acc[1], ah[kk], bl0.z, bl0.w);
    mma16816(acc[2], ah[kk], bl1.x, bl1.y); mma16816(acc[3], ah[kk], bl1.z, bl1.w);
  }
}

// ------------------------------------------------------------------ the forward policy image
// Built from the MlpConst image K1 itself would be launched with (pack_mlp_const_folded for the precise tanh,
// pack_mlp_const for the fast one), so both arithmetics take the same rounded weights.
//   frag: W2 as the B operand of layer 2 (pack_w2_frags, p = 0)
//   col[q][f][j][e]: the parameters of hidden unit 8 j + 2 q + e for the lanes with lane & 3 == q, f = W1 rows (D), b1,
//                    b2, W3 rows (D) -- a lane reads its 8 columns with LDS.128
template <int D>
struct alignas(16) MlpMma {
  static constexpr int NF = 2 * D + 2;
  uint32_t frag[2][2][2][32][4];
  float col[4][NF][4][2];
  float b3[(D + 3) & ~3];
};
template <int D>
inline void pack_mlp_mma(const MlpConst<D, 32>& W, MlpMma<D>& out) {
  pack_w2_frags<D, 32>(W, 1, reinterpret_cast<uint32_t (*)[2][2][2][32][4]>(&out.frag));
  for (int q = 0; q < 4; ++q)
    for (int j = 0; j < 4; ++j)
      for (int e = 0; e < 2; ++e) {
        const int c = 8 * j + 2 * q + e;
        for (int i = 0; i < D; ++i) {
          out.col[q][i][j][e] = W.W1t[i][c];
          out.col[q][D + 2 + i][j][e] = W.W3[i][c];
        }
        out.col[q][D][j][e] = W.b1[c];
        out.col[q][D + 1][j][e] = W.b2[c];
      }
  for (int k = 0; k < ((D + 3) & ~3); ++k) out.b3[k] = W.b3[k];
}
// Where the clamp of rsig_group cannot bind, proven on the host (in double) from the folded image the kernel is launched
// with, so that the kernel may leave it out (rsig_group<G, false>) and compute the same bits:
//   layer 2: its inputs are r in [0, 1], so z2_n <= b2_n + sum_k max(W2_nk, 0) =: z2_max.  The launcher takes the
//            clamp-free kernel when z2_max <= RCP_GROUP_SAFE_Z;
//   layer 1: z1_j = b1_j + sum_i W1_ji x_i <= b1_j + (sum_i |W1_ji|) max_i |x_i|, which stays <= RCP_GROUP_SAFE_Z while
//            max_i |x_i| <= x1_max (negative: for no x).  A warp whose 32 states all satisfy it skips the clamp in layer 1.
template <int D, int H>
inline void fwd_mma_clamp_bounds(const MlpConst<D, H>& W, double& z2_max, double& x1_max) {
  z2_max = -HUGE_VAL;
  for (int n = 0; n < H; ++n) {
    double z = (double)W.b2[n];
    for (int k = 0; k < H; ++k) z += W.W2t[k][n] > 0.0f ? (double)W.W2t[k][n] : 0.0;
    z2_max = z > z2_max ? z : z2_max;
  }
  x1_max = HUGE_VAL;
  for (int j = 0; j < H; ++j) {
    double a = 0.0;
    for (int i = 0; i < D; ++i) a += fabs((double)W.W1t[i][j]);
    const double room = RCP_GROUP_SAFE_Z - (double)W.b1[j];
    if (room < 0.0) x1_max = -1.0;
    else if (a > 0.0 && room / a < x1_max) x1_max = room / a;
  }
}

// what a block copies to shared memory at its start (16-byte words): the fragment table, then the column table
constexpr int MLP_MMA_FRAG_WORDS = 2 * 2 * 2 * 32;
template <int D>
constexpr int mlp_mma_smem_words() { return (int)(offsetof(MlpMma<D>, b3) / 16); }

// activations of two packed pairs of pre-activations of one row: r = 1 / (2^z + 1) on a pack_mlp_const_folded image, with
// one reciprocal per RLSDE_FWD_RCP_GROUP of them (rsig_group; CLAMP = false only where fwd_mma_clamp_bounds proves the
// clamp cannot bind), tanh otherwise.  Which activations share a reciprocal depends only on the layer and the hidden
// units, never on the lane or the row: the REPL continuation below computes the same groups as the full tile.
template <bool FAST, bool CLAMP = true>
__device__ __forceinline__ void act_group_mma(u64 za, u64 zb, float& a0, float& a1, float& a2, float& a3) {
  if constexpr (FAST) {
    tanh_pair<true>(za, a0, a1);
    tanh_pair<true>(zb, a2, a3);
  } else {
    rsig_group<RLSDE_FWD_RCP_GROUP, CLAMP>(za, zb, a0, a1, a2, a3);
  }
}

// layer 1 of rows g + 8 (2 mt + h), h = 0, 1 (inputs xr[h]) straight into the A-fragment layout of layer 2: a[kk][r4] holds
// row h = r4 & 1, columns of j = 2 kk + (r4 >> 1); the four columns of one (t, h) are one activation group
template <int D, bool FAST, bool REPL, bool CLAMP>
__device__ __forceinline__ void layer1_mma(const float4* col, const float (&xr)[2][D], uint32_t (&ah)[2][4],
                                           uint32_t (&al)[2][4]) {
#pragma unroll
  for (int t = 0; t < 2; ++t) {                  // t = kk: j = 2 t, 2 t + 1
    const float4 bb = col[D * 2 + t];
    float4 ww[D];
#pragma unroll
    for (int i = 0; i < D; ++i) ww[i] = col[i * 2 + t];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (REPL && h == 1) {
        ah[t][1] = ah[t][0]; al[t][1] = al[t][0]; ah[t][3] = ah[t][2]; al[t][3] = al[t][2];
        continue;
      }
      u64 z0 = pack2(bb.x, bb.y), z1 = pack2(bb.z, bb.w);
#pragma unroll
      for (int i = 0; i < D; ++i) {
        fma2(z0, pack2(xr[h][i], xr[h][i]), pack2(ww[i].x, ww[i].y));
        fma2(z1, pack2(xr[h][i], xr[h][i]), pack2(ww[i].z, ww[i].w));
      }
      float a[4];
      act_group_mma<FAST, CLAMP>(z0, z1, a[0], a[1], a[2], a[3]);
      split_pair(a[0], a[1], ah[t][h], al[t][h]);
      split_pair(a[2], a[3], ah[t][2 + h], al[t][2 + h]);
    }
  }
}

// u = policy(x) of the trajectory of this lane; all 32 lanes of the warp must take part (x and u of the other lanes'
// trajectories come and go through the quad).  s_frag / s_col: the block's shared-memory copy of MlpMma<D>.
// REPL: every lane holds the same trajectory (the warp-per-trajectory continuation), so all 32 rows are equal: one m16
// tile and one row per lane are evaluated and copied to the others -- the values the full tile would hold, at a quarter of
// the MUFU and half of the HMMA work on the latency path of a lone trajectory.
// CLAMP2 = false: layer 2 without the clamp of rsig_group (the host has proven z2_max <= RCP_GROUP_SAFE_Z);
// clamp1 = false: layer 1 without it (warp-uniform: every lane's state is within x1_max).  Precise tanh only.
template <int D, bool FAST, bool REPL = false, bool CLAMP2 = true>
__device__ __forceinline__ void mlp_forward_mma(const uint4* __restrict__ s_frag, const float4* __restrict__ s_col,
                                                const float (&b3)[(D + 3) & ~3], int lane, const float (&x)[D],
                                                float (&u)[D], bool clamp1 = true) {
  static_assert(FAST || RLSDE_FWD_FOLDED, "the precise tanh is evaluated on the folded image");
  constexpr unsigned FULL = 0xffffffffu;
  constexpr int NF = MlpMma<D>::NF;
  const int q = lane & 3, quad = lane & ~3;
  const float4* col = s_col + q * NF * 2;          // [f][j pair]: float4 = columns of j = 2 t and 2 t + 1
  float part[D][4];                                // head partials of rows g + 8 b over this lane's 8 columns
#pragma unroll
  for (int mt = 0; mt < (REPL ? 1 : 2); ++mt) {
    // rows g + 8 (2 mt + h), h = 0, 1: the trajectories of lanes quad + 2 mt + h
    float xr[2][D];
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int i = 0; i < D; ++i) xr[h][i] = __shfl_sync(FULL, x[i], quad | (2 * mt + h));
    uint32_t ah[2][4], al[2][4];
    if (!FAST && !clamp1) layer1_mma<D, FAST, REPL, false>(col, xr, ah, al);
    else layer1_mma<D, FAST, REPL, true>(col, xr, ah, al);
    // layer 2 on the tensor cores, accumulators initialised to the bias
    float acc[4][4];
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const float4 bb = col[(D + 1) * 2 + t];
      acc[2 * t][0] = bb.x; acc[2 * t][1] = bb.y; acc[2 * t][2] = bb.x; acc[2 * t][3] = bb.y;
      acc[2 * t + 1][0] = bb.z; acc[2 * t + 1][1] = bb.w; acc[2 * t + 1][2] = bb.z; acc[2 * t + 1][3] = bb.w;
    }
    mma_product_w(acc, ah, al, s_frag, 0, lane);
    // activation groups: the columns of n-tiles j and j + 1 (j = 0, 2) of one row
#pragma unroll
    for (int j = 0; j < 4; j += 2) {
      act_group_mma<FAST, CLAMP2>(pack2(acc[j][0], acc[j][1]), pack2(acc[j + 1][0], acc[j + 1][1]),
                                  acc[j][0], acc[j][1], acc[j + 1][0], acc[j + 1][1]);
      if constexpr (REPL) {
        acc[j][2] = acc[j][0]; acc[j][3] = acc[j][1]; acc[j + 1][2] = acc[j + 1][0]; acc[j + 1][3] = acc[j + 1][1];
      } else {
        act_group_mma<FAST, CLAMP2>(pack2(acc[j][2], acc[j][3]), pack2(acc[j + 1][2], acc[j + 1][3]),
                                    acc[j][2], acc[j][3], acc[j + 1][2], acc[j + 1][3]);
      }
    }
    // head partials: sum over this lane's 8 columns, as one packed accumulator per row (even / odd columns)
#pragma unroll
    for (int i = 0; i < D; ++i) {
      u64 p[2] = {0ull, 0ull};
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const float4 w3 = col[(D + 2 + i) * 2 + t];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          fma2(p[h], pack2(acc[2 * t][2 * h], acc[2 * t][2 * h + 1]), pack2(w3.x, w3.y));
          fma2(p[h], pack2(acc[2 * t + 1][2 * h], acc[2 * t + 1][2 * h + 1]), pack2(w3.z, w3.w));
        }
      }
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        float lo, hi;
        unpack2(p[h], lo, hi);
        part[i][2 * mt + h] = __fadd_rn(lo, hi);
      }
    }
  }
  if constexpr (REPL) {
#pragma unroll
    for (int i = 0; i < D; ++i) { part[i][2] = part[i][0]; part[i][3] = part[i][1]; }
  }
  // quad reduce-scatter: over lane bit 1, then bit 0; lane q ends with row q's sum (p0 + p2) + (p1 + p3)
  const bool b1 = (q & 2) != 0, b0 = (q & 1) != 0;
#pragma unroll
  for (int i = 0; i < D; ++i) {
    const float k0 = b1 ? part[i][2] : part[i][0], k1 = b1 ? part[i][3] : part[i][1];
    const float s0 = b1 ? part[i][0] : part[i][2], s1 = b1 ? part[i][1] : part[i][3];
    const float r0 = __fadd_rn(k0, __shfl_xor_sync(FULL, s0, 2));
    const float r1 = __fadd_rn(k1, __shfl_xor_sync(FULL, s1, 2));
    const float keep = b0 ? r1 : r0, send = b0 ? r0 : r1;
    u[i] = __fadd_rn(__fadd_rn(keep, __shfl_xor_sync(FULL, send, 1)), b3[i]);
  }
}

}  // namespace rlsde
