// Device-side building blocks shared by the rollout kernels (sm_100a).
//
//  * Philox4x32-10 counter-based generator + Box-Muller normals: the Brownian increments the
//    reference draws with torch.randn / np.random.randn (environments.py:145,208) become a pure
//    function of (seed, global trajectory id, pass index, coordinate), so results do not depend
//    on how trajectories are scheduled onto lanes or sharded over GPUs.
//  * packed fp32 arithmetic (fma.rn.f32x2 -> SASS FFMA2): two FMAs per issue slot, with the
//    activation as a scalar-broadcast register operand and the weight pair as a uniform-register
//    operand loaded from the constant bank (measured in tools/microbench/layer.cu).
//  * tanh: "precise" = 1 - 2 / (2^(c x) + 1) (MUFU.EX2 + MUFU.RCP, ~3e-7 abs. error) and
//    "fast" = tanh.approx (MUFU.TANH, 2^-11 rel. error).
#pragma once
#include <cstdint>
#include <type_traits>
#include <cuda_runtime.h>

namespace rlsde {

typedef unsigned long long u64;

// diagnostics: every launcher reports the kernels it enqueued (rlsde_launch_count in the C ABI)
void note_kernel_launches(int n);

// ------------------------------------------------------------------ packed fp32 helpers
__device__ __forceinline__ u64 pack2(float lo, float hi) {
  u64 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(u64 v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
// acc += a * w   (lane-wise on the two packed floats)
__device__ __forceinline__ void fma2(u64& acc, u64 a, u64 w) {
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(w));
}
__device__ __forceinline__ u64 fma2r(u64 a, u64 b, u64 c) {
  u64 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ u64 add2(u64 a, u64 b) {
  u64 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ u64 sub2(u64 a, u64 b) {
  u64 d;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ u64 mul2(u64 a, u64 b) {
  u64 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}

// ------------------------------------------------------------------ MUFU wrappers
__device__ __forceinline__ float mufu_ex2(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float mufu_rcp(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float mufu_tanh(float x) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float mufu_lg2(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float mufu_sqrt(float x) { float y; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float mufu_sin(float x) { float y; asm("sin.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float mufu_cos(float x) { float y; asm("cos.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// 2 log2(e): hidden-layer weights and biases are pre-multiplied by this on the host for the
// precise tanh, so that tanh(z) = 1 - 2 / (2^(z') + 1) with z' the accumulated pre-activation.
#define RLSDE_TWO_LOG2E 2.8853900817779268
// forward-only thread-per-trajectory kernel: hidden layers pass r = 1 / (exp(2 z) + 1) on, the "1 - 2 r" of the tanh is
// folded into the next layer's weights (see rsig_pair); 0 = evaluate tanh itself, as the reverse-pass kernels do
#ifndef RLSDE_FWD_FOLDED
#define RLSDE_FWD_FOLDED 1
#endif

// tanh of a packed pair of (pre-scaled) pre-activations.  One asm block per pair: keeping the
// statement count of the fully unrolled step body low matters for compile time with -lineinfo.
template <bool FAST>
__device__ __forceinline__ void tanh_pair(u64 acc, float& t0, float& t1) {
  if constexpr (FAST) {
    asm("{\n\t.reg .f32 a0, a1;\n\t"
        "mov.b64 {a0, a1}, %2;\n\t"
        "tanh.approx.f32 %0, a0;\n\ttanh.approx.f32 %1, a1;\n\t}"
        : "=f"(t0), "=f"(t1) : "l"(acc));
  } else {
    asm("{\n\t.reg .f32 a0, a1, e0, e1, d0, d1, r0, r1;\n\t.reg .b64 p, q;\n\t"
        "mov.b64 {a0, a1}, %2;\n\t"
        "ex2.approx.ftz.f32 e0, a0;\n\tex2.approx.ftz.f32 e1, a1;\n\t"
        "mov.b64 p, {e0, e1};\n\tadd.rn.f32x2 p, p, %3;\n\tmov.b64 {d0, d1}, p;\n\t"
        "rcp.approx.ftz.f32 r0, d0;\n\trcp.approx.ftz.f32 r1, d1;\n\t"
        "mov.b64 q, {r0, r1};\n\tfma.rn.f32x2 q, q, %4, %3;\n\tmov.b64 {%0, %1}, q;\n\t}"
        : "=f"(t0), "=f"(t1) : "l"(acc), "l"(0x3f8000003f800000ull), "l"(0xc0000000c0000000ull));
  }
}

// r = 1 / (2^a + 1) of a packed pair of pre-scaled pre-activations: the precise tanh without its last step,
// tanh = 1 - 2 r.  The forward-only kernel feeds r to the next layer, whose weights carry the -2 and whose bias carries
// the row sums (pack_mlp_const_folded): one FFMA2 per pair less on the pipe that bounds that kernel.
__device__ __forceinline__ void rsig_pair(u64 acc, float& r0, float& r1) {
  asm("{\n\t.reg .f32 a0, a1, e0, e1, d0, d1;\n\t.reg .b64 p;\n\t"
      "mov.b64 {a0, a1}, %2;\n\t"
      "ex2.approx.ftz.f32 e0, a0;\n\tex2.approx.ftz.f32 e1, a1;\n\t"
      "mov.b64 p, {e0, e1};\n\tadd.rn.f32x2 p, p, %3;\n\tmov.b64 {d0, d1}, p;\n\t"
      "rcp.approx.ftz.f32 %0, d0;\n\trcp.approx.ftz.f32 %1, d1;\n\t}"
      : "=f"(r0), "=f"(r1) : "l"(acc), "l"(0x3f8000003f800000ull));
}

// rsig_pair of two packed pairs za = {z0, z1}, zb = {z2, z3} with one MUFU.RCP per G activations instead of one each
// (G = RLSDE_FWD_RCP_GROUP; the tensor-core forward policy, mlp_mma.cuh):
//   G = 2:  p = da db (packed),  R = {1 / p.x, 1 / p.y},  ra = R db,  rb = R da
//   G = 4:  p = da db,  R = 1 / (p.x p.y),  Q = {R p.y, R p.x} = {1 / p.x, 1 / p.y},  ra = Q db,  rb = Q da
// with d = 2^z + 1 >= 1, so no product can become subnormal.  A product can overflow, which makes the reciprocal 0 and the
// smaller members' r 0 (or NaN): z is clamped to 63 (G = 2) / 31 (G = 4) first, so that the product of G of them stays
// below 2^126.  The clamp moves r by at most 2^-31 (r < 2^-31 on both sides of it).
// Error: the group adds 2 (G = 2) / 4 (G = 4) float32 roundings to each r.  With correctly rounded EX2 and RCP, over
// z in [-200, 200], |r - 1 / (2^z + 1)| <= k 2^-24 (r + 2^-31) + 2^-31 with k = 3.5 (G = 2) / 4.5 (G = 4), against 2.5
// ungrouped (tests/test_fwd_grouped_rcp.py restates the arithmetic); MUFU.EX2 / RCP add their own few ulp as before.  So
// tanh = 1 - 2 r moves by at most ~2 ulp of 1 (~2.4e-7) more than with G = 1.
// CLAMP = false leaves the clamp out.  Only for inputs known to stay <= RCP_GROUP_SAFE_Z (fwd_mma_clamp_bounds): there
// the clamp is the identity, so both forms give the same bits.
#ifndef RLSDE_FWD_RCP_GROUP
#define RLSDE_FWD_RCP_GROUP 4
#endif
template <int G>
struct RcpGroup {
  static_assert(G == 1 || G == 2 || G == 4, "RLSDE_FWD_RCP_GROUP is 1, 2 or 4");
  static constexpr float ZMAX = G == 4 ? 31.0f : 63.0f;   // the clamp on z (unused for G = 1)
};
// the bound a host-side proof must establish before CLAMP = false: one below the smallest clamp, which leaves room for
// the float32 / tensor-core rounding of z against its bound computed in double
constexpr double RCP_GROUP_SAFE_Z = 30.0;
template <int G, bool CLAMP = true>
__device__ __forceinline__ void rsig_group(u64 za, u64 zb, float& r0, float& r1, float& r2, float& r3) {
  if constexpr (G == 1) {
    rsig_pair(za, r0, r1);
    rsig_pair(zb, r2, r3);
  } else {
    float z[4];
    unpack2(za, z[0], z[1]);
    unpack2(zb, z[2], z[3]);
    if constexpr (CLAMP) {
#pragma unroll
      for (int i = 0; i < 4; ++i) asm("min.NaN.f32 %0, %0, %1;" : "+f"(z[i]) : "f"(RcpGroup<G>::ZMAX));   // NaN stays NaN
    }
    const u64 one = 0x3f8000003f800000ull;
    const u64 da = add2(pack2(mufu_ex2(z[0]), mufu_ex2(z[1])), one);
    const u64 db = add2(pack2(mufu_ex2(z[2]), mufu_ex2(z[3])), one);
    float px, py;
    unpack2(mul2(da, db), px, py);
    u64 q;
    if constexpr (G == 2) {
      q = pack2(mufu_rcp(px), mufu_rcp(py));
    } else {
      const float R = mufu_rcp(__fmul_rn(px, py));
      q = pack2(__fmul_rn(R, py), __fmul_rn(R, px));
    }
    unpack2(mul2(q, db), r0, r1);
    unpack2(mul2(q, da), r2, r3);
  }
}

// acc[o .. o+7] (8 packed accumulators = 16 outputs) += h * w[2o .. 2o+15]
#define RLSDE_FMA2X8(acc, o, h, w)                                                                                  \
  asm("{\n\t.reg .b64 hh, w0, w1, w2, w3, w4, w5, w6, w7;\n\t"                                                       \
      "mov.b64 hh, {%8, %8};\n\t"                                                                                    \
      "mov.b64 w0, {%9, %10};\n\tmov.b64 w1, {%11, %12};\n\tmov.b64 w2, {%13, %14};\n\tmov.b64 w3, {%15, %16};\n\t"   \
      "mov.b64 w4, {%17, %18};\n\tmov.b64 w5, {%19, %20};\n\tmov.b64 w6, {%21, %22};\n\tmov.b64 w7, {%23, %24};\n\t"  \
      "fma.rn.f32x2 %0, hh, w0, %0;\n\tfma.rn.f32x2 %1, hh, w1, %1;\n\t"                                             \
      "fma.rn.f32x2 %2, hh, w2, %2;\n\tfma.rn.f32x2 %3, hh, w3, %3;\n\t"                                             \
      "fma.rn.f32x2 %4, hh, w4, %4;\n\tfma.rn.f32x2 %5, hh, w5, %5;\n\t"                                             \
      "fma.rn.f32x2 %6, hh, w6, %6;\n\tfma.rn.f32x2 %7, hh, w7, %7;\n\t}"                                            \
      : "+l"(acc[(o) + 0]), "+l"(acc[(o) + 1]), "+l"(acc[(o) + 2]), "+l"(acc[(o) + 3]), "+l"(acc[(o) + 4]),          \
        "+l"(acc[(o) + 5]), "+l"(acc[(o) + 6]), "+l"(acc[(o) + 7])                                                   \
      : "f"(h), "f"((w)[2 * (o) + 0]), "f"((w)[2 * (o) + 1]), "f"((w)[2 * (o) + 2]), "f"((w)[2 * (o) + 3]),          \
        "f"((w)[2 * (o) + 4]), "f"((w)[2 * (o) + 5]), "f"((w)[2 * (o) + 6]), "f"((w)[2 * (o) + 7]),                  \
        "f"((w)[2 * (o) + 8]), "f"((w)[2 * (o) + 9]), "f"((w)[2 * (o) + 10]), "f"((w)[2 * (o) + 11]),                \
        "f"((w)[2 * (o) + 12]), "f"((w)[2 * (o) + 13]), "f"((w)[2 * (o) + 14]), "f"((w)[2 * (o) + 15]))

// acc (one packed accumulator) += sum_{j = o .. o+11, step 2} {h[j], h[j+1]} * {w[j], w[j+1]}   (12 activations)
#define RLSDE_DOT2X6(acc, o, h, w)                                                                                  \
  asm("{\n\t.reg .b64 a, b;\n\t"                                                                                     \
      "mov.b64 a, {%1, %2};\n\tmov.b64 b, {%13, %14};\n\tfma.rn.f32x2 %0, a, b, %0;\n\t"                             \
      "mov.b64 a, {%3, %4};\n\tmov.b64 b, {%15, %16};\n\tfma.rn.f32x2 %0, a, b, %0;\n\t"                             \
      "mov.b64 a, {%5, %6};\n\tmov.b64 b, {%17, %18};\n\tfma.rn.f32x2 %0, a, b, %0;\n\t"                             \
      "mov.b64 a, {%7, %8};\n\tmov.b64 b, {%19, %20};\n\tfma.rn.f32x2 %0, a, b, %0;\n\t"                             \
      "mov.b64 a, {%9, %10};\n\tmov.b64 b, {%21, %22};\n\tfma.rn.f32x2 %0, a, b, %0;\n\t"                            \
      "mov.b64 a, {%11, %12};\n\tmov.b64 b, {%23, %24};\n\tfma.rn.f32x2 %0, a, b, %0;\n\t}"                          \
      : "+l"(acc)                                                                                                    \
      : "f"((h)[(o) + 0]), "f"((h)[(o) + 1]), "f"((h)[(o) + 2]), "f"((h)[(o) + 3]), "f"((h)[(o) + 4]),               \
        "f"((h)[(o) + 5]), "f"((h)[(o) + 6]), "f"((h)[(o) + 7]), "f"((h)[(o) + 8]), "f"((h)[(o) + 9]),               \
        "f"((h)[(o) + 10]), "f"((h)[(o) + 11]), "f"((w)[(o) + 0]), "f"((w)[(o) + 1]), "f"((w)[(o) + 2]),             \
        "f"((w)[(o) + 3]), "f"((w)[(o) + 4]), "f"((w)[(o) + 5]), "f"((w)[(o) + 6]), "f"((w)[(o) + 7]),               \
        "f"((w)[(o) + 8]), "f"((w)[(o) + 9]), "f"((w)[(o) + 10]), "f"((w)[(o) + 11]))

// ------------------------------------------------------------------ Philox4x32-10
struct Philox4 { uint32_t x, y, z, w; };

__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                          uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    const uint32_t n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    const uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return Philox4{c0, c1, c2, c3};
}

// Noise addressing.  The increments of one trajectory form the flat sequence m = pass * d + coordinate.
// One Philox block yields 4 normals: block index b = m / 4, slot = m % 4.  Counter = (traj_lo, traj_hi,
// b_lo, b_hi | stream tag), key = seed.  (oracle/rlsde_oracle.c uses the same mapping.)
#define RLSDE_PHILOX_TAG 0x52534445u /* "RSDE" */

// 4 increments dB = sqrt(dt) * N(0,1) for noise block b of trajectory traj.
// scale2 = -2 * dt * ln(2)   (so that r = sqrt(scale2 * log2(u1)) = sqrt(dt) * sqrt(-2 ln u1))
__device__ __forceinline__ void noise_block(uint64_t seed, uint64_t traj, uint32_t b, float scale2, float (&z)[4]) {
  const Philox4 r = philox4x32_10((uint32_t)traj, (uint32_t)(traj >> 32), b, RLSDE_PHILOX_TAG,
                                  (uint32_t)seed, (uint32_t)(seed >> 32));
  const float kTwoM32 = 2.3283064365386963e-10f, kHalfUlp = 1.1641532182693481e-10f;
  const float u0 = fmaf((float)r.x, kTwoM32, kHalfUlp);   // (0, 1]
  const float u1 = fmaf((float)r.y, kTwoM32, kHalfUlp);
  const float u2 = fmaf((float)r.z, kTwoM32, kHalfUlp);
  const float u3 = fmaf((float)r.w, kTwoM32, kHalfUlp);
  const float ra = mufu_sqrt(scale2 * mufu_lg2(u0));
  const float rb = mufu_sqrt(scale2 * mufu_lg2(u2));
  const float ta = 6.2831853071795865f * u1, tb = 6.2831853071795865f * u3;
  z[0] = ra * mufu_cos(ta);
  z[1] = ra * mufu_sin(ta);
  z[2] = rb * mufu_cos(tb);
  z[3] = rb * mufu_sin(tb);
}

// ------------------------------------------------------------------ policy parameters in the constant bank
// Hidden layers are stored input-major ("transposed") so that the unrolled inner loop over outputs
// walks contiguous constants (LDCU.128 -> four weights per uniform load); the head keeps the
// state_dict layout (output-major) and is evaluated as packed dot products.
template <int D, int H>
struct alignas(16) MlpConst {
  static_assert(H % 16 == 0, "hidden width must be a multiple of 16");
  float W1t[D][H];    // W1t[i][j] = s * policy.0.weight[j][i]
  float b1[H];        //             s * policy.0.bias
  float W2t[H][H];    // W2t[i][j] = s * policy.2.weight[j][i]
  float b2[H];
  float W3[D][H];     // policy.4.weight
  float b3[(D + 3) & ~3];
};

// host: state_dict-ordered flat parameters -> MlpConst;  s = 2 log2(e) for the precise tanh, 1 for the fast one
template <int D, int H>
inline void pack_mlp_const(const float* p, bool fast_tanh, MlpConst<D, H>& out) {
  const double s = fast_tanh ? 1.0 : RLSDE_TWO_LOG2E;
  const float* W1 = p;              // (H, D)
  const float* b1 = W1 + H * D;
  const float* W2 = b1 + H;         // (H, H)
  const float* b2 = W2 + H * H;
  const float* W3 = b2 + H;         // (D, H)
  const float* b3 = W3 + D * H;
  for (int i = 0; i < D; ++i)
    for (int j = 0; j < H; ++j) out.W1t[i][j] = (float)(s * (double)W1[j * D + i]);
  for (int j = 0; j < H; ++j) out.b1[j] = (float)(s * (double)b1[j]);
  for (int i = 0; i < H; ++i)
    for (int j = 0; j < H; ++j) out.W2t[i][j] = (float)(s * (double)W2[j * H + i]);
  for (int j = 0; j < H; ++j) out.b2[j] = (float)(s * (double)b2[j]);
  for (int k = 0; k < D; ++k)
    for (int j = 0; j < H; ++j) out.W3[k][j] = W3[k * H + j];
  for (int k = 0; k < ((D + 3) & ~3); ++k) out.b3[k] = (k < D) ? b3[k] : 0.0f;
}

// The same for the forward-only kernel with the precise tanh: hidden layers hand r = (1 - tanh) / 2 to the next layer, so
//   z2 = b2 + W2 h1 = (b2 + W2 1) + (-2 W2) r1,     u = b3 + W3 h2 = (b3 + W3 1) + (-2 W3) r2
// -- the factor is a power of two (exact), the folded biases are formed in double and rounded once.
template <int D, int H>
inline void pack_mlp_const_folded(const float* p, MlpConst<D, H>& out) {
  pack_mlp_const<D, H>(p, false, out);
  const float* W2 = p + H * D + H;  // (H, H)
  const float* b2 = W2 + H * H;
  const float* W3 = b2 + H;         // (D, H)
  const float* b3 = W3 + D * H;
  for (int j = 0; j < H; ++j) {
    double rs = 0.0;
    for (int i = 0; i < H; ++i) { rs += (double)W2[j * H + i]; out.W2t[i][j] = -2.0f * out.W2t[i][j]; }
    out.b2[j] = (float)(RLSDE_TWO_LOG2E * ((double)b2[j] + rs));
  }
  for (int k = 0; k < D; ++k) {
    double rs = 0.0;
    for (int j = 0; j < H; ++j) { rs += (double)W3[k * H + j]; out.W3[k][j] = -2.0f * W3[k * H + j]; }
    out.b3[k] = (float)((double)b3[k] + rs);
  }
}

// One row of constant-bank weights into a local array through explicit 16-byte loads.  (SASS is the
// same LDCU.128 either way; with scalar loads the front end's compile time grows quadratically in
// the number of constant loads of the fully unrolled kernels.)
template <int N>
__device__ __forceinline__ void load_row(const float (&src)[N], float (&w)[N]) {
  static_assert(N % 4 == 0, "rows are padded to 16 bytes");
#pragma unroll
  for (int q = 0; q < N / 4; ++q) {
    const float4 t = reinterpret_cast<const float4*>(&src[0])[q];
    w[4 * q] = t.x; w[4 * q + 1] = t.y; w[4 * q + 2] = t.z; w[4 * q + 3] = t.w;
  }
}

// hidden activations of one layer: hout = tanh(bias + Wt^T hin)   (IN inputs, H outputs)
template <int IN, int H, bool FAST, bool RSIG = false>
__device__ __forceinline__ void dense_tanh(const float (&Wt)[IN][H], const float (&b)[H], const float (&hin)[IN],
                                           float (&hout)[H]) {
  // Outputs are produced in slabs of 16 (8 packed accumulators): the MUFU work (tanh) of one slab is
  // independent of the FFMA2 stream of the next, so the two pipes can overlap inside one warp.
#ifndef RLSDE_DENSE_SLAB
#define RLSDE_DENSE_SLAB 256
#endif
  constexpr int SLAB = (RLSDE_DENSE_SLAB < H) ? RLSDE_DENSE_SLAB : H;   // outputs per slab (multiple of 16)
#pragma unroll
  for (int s0 = 0; s0 < H; s0 += SLAB) {
    u64 acc[SLAB / 2];
#pragma unroll
    for (int q = 0; q < SLAB / 4; ++q) {
      const float4 t = reinterpret_cast<const float4*>(&b[s0])[q];
      acc[2 * q] = pack2(t.x, t.y);
      acc[2 * q + 1] = pack2(t.z, t.w);
    }
#pragma unroll
    for (int i = 0; i < IN; ++i) {
      float w[SLAB];
#pragma unroll
      for (int q = 0; q < SLAB / 4; ++q) {
        const float4 t = reinterpret_cast<const float4*>(&Wt[i][s0])[q];
        w[4 * q] = t.x; w[4 * q + 1] = t.y; w[4 * q + 2] = t.z; w[4 * q + 3] = t.w;
      }
#pragma unroll
      for (int o = 0; o < SLAB / 2; o += 8) RLSDE_FMA2X8(acc, o, hin[i], w);
    }
#pragma unroll
    for (int j = 0; j < SLAB / 2; ++j) {
      if constexpr (RSIG) rsig_pair(acc[j], hout[s0 + 2 * j], hout[s0 + 2 * j + 1]);
      else tanh_pair<FAST>(acc[j], hout[s0 + 2 * j], hout[s0 + 2 * j + 1]);
    }
  }
}

// a = policy(x): two tanh layers of width H (FFMA2 with broadcast activations) and a linear head
// (packed dot products).  h1 / h2 are returned for the reverse pass.
template <int D, int H, bool FAST>
__device__ __forceinline__ void mlp_forward_keep(const MlpConst<D, H>& W, const float (&x)[D], float (&h1)[H],
                                                 float (&h2)[H], float (&u)[D]) {
  dense_tanh<D, H, FAST>(W.W1t, W.b1, x, h1);
  dense_tanh<H, H, FAST>(W.W2t, W.b2, h1, h2);
#pragma unroll
  for (int k = 0; k < D; ++k) {
    u64 acc = pack2(W.b3[k], 0.0f);
    float w[H];
    load_row<H>(W.W3[k], w);
#pragma unroll
    for (int o = 0; o < H; o += 16) {
      RLSDE_DOT2X6(acc, o, h2, w);   // 12 of the 16 activations of this slab (30-operand asm limit)
      u64 a = pack2(h2[o + 12], h2[o + 13]), b = pack2(w[o + 12], w[o + 13]);
      fma2(acc, a, b);
      a = pack2(h2[o + 14], h2[o + 15]); b = pack2(w[o + 14], w[o + 15]);
      fma2(acc, a, b);
    }
    float lo, hi;
    unpack2(acc, lo, hi);
    u[k] = lo + hi;
  }
}

template <int D, int H, bool FAST>
__device__ __forceinline__ void mlp_forward(const MlpConst<D, H>& W, const float (&x)[D], float (&u)[D]) {
  float h1[H], h2[H];
  mlp_forward_keep<D, H, FAST>(W, x, h1, h2, u);
}

// the head of mlp_forward_keep on its own
template <int D, int H>
__device__ __forceinline__ void mlp_head(const MlpConst<D, H>& W, const float (&h2)[H], float (&u)[D]) {
#pragma unroll
  for (int k = 0; k < D; ++k) {
    u64 acc = pack2(W.b3[k], 0.0f);
    float w[H];
    load_row<H>(W.W3[k], w);
#pragma unroll
    for (int o = 0; o < H; o += 16) {
      RLSDE_DOT2X6(acc, o, h2, w);
      u64 a = pack2(h2[o + 12], h2[o + 13]), b = pack2(w[o + 12], w[o + 13]);
      fma2(acc, a, b);
      a = pack2(h2[o + 14], h2[o + 15]); b = pack2(w[o + 14], w[o + 15]);
      fma2(acc, a, b);
    }
    float lo, hi;
    unpack2(acc, lo, hi);
    u[k] = lo + hi;
  }
}

// a = policy(x) from a pack_mlp_const_folded image (precise tanh, forward only)
template <int D, int H>
__device__ __forceinline__ void mlp_forward_folded(const MlpConst<D, H>& W, const float (&x)[D], float (&u)[D]) {
  float r1[H], r2[H];
  dense_tanh<D, H, false, true>(W.W1t, W.b1, x, r1);
  dense_tanh<H, H, false, true>(W.W2t, W.b2, r1, r2);
  mlp_head<D, H>(W, r2, u);
}

// ------------------------------------------------------------------ host-side launch helpers
// A runtime flag as a compile-time one: f(std::true_type{}) if b holds and ALLOWED, else f(std::false_type{}).  Where
// ALLOWED is false the true branch is never instantiated, so a pruned kernel variant is never compiled; the C ABI refuses
// such flags before it launches.
template <bool ALLOWED = true, class F>
static inline int with_flag(bool b, F&& f) {
  if constexpr (ALLOWED) {
    if (b) return f(std::true_type{});
  }
  return f(std::false_type{});
}

// Grid of a kernel that runs one trajectory per thread: one warp per block for small batches, so that the warps spread
// over the SMs (latency-bound regime); otherwise a persistent grid of 128-thread blocks, as many as are co-resident with
// smem bytes of dynamic shared memory each (at most cap per SM when cap >= 1).  Sets block; returns the grid.
template <class Kern>
static long long persistent_grid(Kern kern, long long K, int sm_count, size_t smem, int cap, int& block) {
  long long grid;
  block = 128;
  if (K <= (long long)sm_count * 128) {
    block = 32;
    grid = (K + 31) / 32;
  } else {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, block, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
    if (cap >= 1 && cap < per_sm) per_sm = cap;
    grid = (long long)sm_count * per_sm;
    const long long need = (K + block - 1) / block;
    if (grid > need) grid = need;
  }
  return grid < 1 ? 1 : grid;
}

}  // namespace rlsde
