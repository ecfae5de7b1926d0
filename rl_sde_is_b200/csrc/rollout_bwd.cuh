// K2: fused reverse (adjoint) pass of the REINFORCE surrogate loss through the whole rollout.
//
// Replaces eff_loss.backward() (reinforce_deterministic_core.py:240), i.e. autograd walking ~25
// nodes per pass of sample_loss_vectorized (:52-88; states are never detached, :88), for
//     L = scale * sum_k ( -G_k - sg(G_k) S_k )                                   (:91)
// Per trajectory, for j = k* .. 0 with lambda_{k*+1} = 0 (SURVEY.md Appendix C):
//     a_j      = [j<k*] u_j dt - G dB_{j+1} [j<=k*, or j<k* with RLSDE_F_STOCH_INT_EXACT] + sigma dt lambda_{j+1}
//     theta_bar += (d policy / d theta)(X_j)^T a_j
//     lambda_j = (1 - dt 4 alpha (3 X_j^2 - 1)) * lambda_{j+1} + (d policy / d x)(X_j)^T a_j
// (unscaled; `scale` is applied in the final reduction).
// WEIGHTED (rlsde_rollout_bwd_weighted): L = scale * sum_k (cG_k G_k + cS_k S_k) for per-trajectory coefficients, i.e.
//     a_j      = -cG [j<k*] u_j dt + cS dB_{j+1} [same condition as above] + sigma dt lambda_{j+1}
// (the comment above em_step_f32); the unweighted kernels are the case cG = -1, cS = -G, folded at compile time.
//
// Mapping: one trajectory per thread, processed segment by segment from the last checkpoint
// backwards.  A round = phase A (recompute the segment's states X_j from its checkpoint, identical
// arithmetic to K1) + phase B (walk the segment in reverse: recompute the activations, backpropagate).
// All lanes of a warp are in the same phase at the same time, so the 32 trajectories stay in lock
// step although their lengths differ.  dB is regenerated from Philox, never stored.
//
// Parameter gradients are sums over (trajectory, pass) of outer products.  Each pass, the warp's 32
// lanes stage their (delta, activation) vectors in XOR-swizzled shared memory and every lane
// accumulates one column of the 32x32 (HxH) block in registers: an in-warp 32 x 32 x 32 product on
// FFMA2, broadcast LDS.128 for the deltas.  Per-warp partial gradients go to global memory at the end
// and a second kernel sums them in a fixed order (deterministic; trajectories are assigned to lanes
// statically for the same reason).
#pragma once
#include "rollout_fwd.cuh"

namespace rlsde {

constexpr int BWD_MAX_WARPS = 148 * 16;          // upper bound on warps in the backward grid
constexpr int BWD_MAX_PARAMS = 4608;             // >= P for every compiled shape (d=2, H=64: 4482)
constexpr int BWD_MAX_SEG = 32;                  // largest ckpt_every the backward pass accepts
// two disjoint partial areas: [0, A) for the thread-per-trajectory kernel (float or double partials of a shape with
// P <= 2304 parameters at hidden width 32), [A, A + B) for the warp-per-trajectory kernel that takes the longest
// trajectories concurrently on a second stream
inline size_t bwd_partial_main_bytes() { return (size_t)BWD_MAX_WARPS * BWD_MAX_PARAMS * sizeof(float); }
inline size_t bwd_partial_aux_bytes() { return (size_t)BWD_MAX_WARPS * (BWD_MAX_PARAMS / 2) * sizeof(float); }
inline size_t bwd_workspace_bytes() { return bwd_partial_main_bytes() + bwd_partial_aux_bytes(); }

// acc[o .. o+3] (4 packed accumulators) += h * {w0, w1, w2, w3} with packed weights in registers
#define RLSDE_FMA2X4_REG(acc, o, h, w0, w1, w2, w3)                                                   \
  asm("{\n\t.reg .b64 hh;\n\tmov.b64 hh, {%4, %4};\n\t"                                                \
      "fma.rn.f32x2 %0, hh, %5, %0;\n\tfma.rn.f32x2 %1, hh, %6, %1;\n\t"                               \
      "fma.rn.f32x2 %2, hh, %7, %2;\n\tfma.rn.f32x2 %3, hh, %8, %3;\n\t}"                              \
      : "+l"(acc[(o) + 0]), "+l"(acc[(o) + 1]), "+l"(acc[(o) + 2]), "+l"(acc[(o) + 3])                 \
      : "f"(h), "l"(w0), "l"(w1), "l"(w2), "l"(w3))

// acc (packed) += sum_{q<4} v[o+q] (packed register pairs) * {w[2(o+q)], w[2(o+q)+1]} (constant bank)
#define RLSDE_DOTP4(acc, v, o, w)                                                                     \
  asm("{\n\t.reg .b64 b;\n\t"                                                                          \
      "mov.b64 b, {%5, %6};\n\tfma.rn.f32x2 %0, %1, b, %0;\n\t"                                        \
      "mov.b64 b, {%7, %8};\n\tfma.rn.f32x2 %0, %2, b, %0;\n\t"                                        \
      "mov.b64 b, {%9, %10};\n\tfma.rn.f32x2 %0, %3, b, %0;\n\t"                                       \
      "mov.b64 b, {%11, %12};\n\tfma.rn.f32x2 %0, %4, b, %0;\n\t}"                                     \
      : "+l"(acc)                                                                                      \
      : "l"(v[(o) + 0]), "l"(v[(o) + 1]), "l"(v[(o) + 2]), "l"(v[(o) + 3]),                            \
        "f"((w)[2 * (o) + 0]), "f"((w)[2 * (o) + 1]), "f"((w)[2 * (o) + 2]), "f"((w)[2 * (o) + 3]),    \
        "f"((w)[2 * (o) + 4]), "f"((w)[2 * (o) + 5]), "f"((w)[2 * (o) + 6]), "f"((w)[2 * (o) + 7]))

// Layout of a [32 lanes][H] float tile in shared memory.  Both variants make a lane writing its own row with STS.128, a
// broadcast read of one row and a read of one column element per lane conflict-free:
//   PAD = false: XOR swizzle at float4 granularity (no extra memory, ~1 450 integer instructions per pass for addresses);
//   PAD = true:  rows padded to H + 4 floats (plain addresses).
// Measured (tools/bench_train.py): at d = 1, where the kernel runs 4 blocks per SM, the padded layout is 19 % faster
// (57.7 -> 46.8 ms: with four warps per scheduler the instruction count is what limits), at d = 2..4 with 3 blocks per SM
// 14 % faster; at 2 blocks per SM (d = 10) the swizzle is 3-5 % faster (the address arithmetic fills issue slots that
// would idle anyway).
constexpr bool bwd_tiles_padded(int D) { return D <= 4; }
template <int H, bool PAD>
__device__ __forceinline__ int swz(int row, int col) {
  if constexpr (PAD) return row * (H + 4) + col;
  else return row * H + ((((col >> 2) ^ (row & 7)) << 2) | (col & 3));
}
template <int H, bool PAD>
__host__ __device__ constexpr int tile_floats() { return 32 * (H + (PAD ? 4 : 0)); }

template <int H, bool PAD>
__device__ __forceinline__ void stage_row(float* tile, int lane, const float (&v)[H]) {
#pragma unroll
  for (int q = 0; q < H / 4; ++q)
    *reinterpret_cast<float4*>(tile + swz<H, PAD>(lane, 4 * q)) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
}

// cached Philox block per lane for out-of-order (reverse) access to the increments
template <int D>
struct NoiseCache {
  static constexpr int SPB = NoisePlan<D>::SPB;
  static constexpr int BPP = NoisePlan<D>::BPP;
  float z[NoisePlan<D>::NZ];
  long long blk;
  __device__ __forceinline__ void reset() { blk = -1; }
  __device__ __forceinline__ void get(const FwdArgs& A, bool inject, bool ok, long long traj, int j, float (&dB)[D]) {
    if (inject) {
      const long long row = (long long)j * A.K_global + (A.traj_offset + traj);
#pragma unroll
      for (int i = 0; i < D; ++i) dB[i] = (ok && j < A.noise_steps) ? __ldg(A.noise + row * D + i) : 0.f;
      return;
    }
    const long long want = j / SPB;
    if (ok && want != blk) {
      const unsigned long long gt = (unsigned long long)(A.traj_offset + traj);
#pragma unroll
      for (int q = 0; q < BPP; ++q) {
        float zz[4];
        noise_block(A.seed, gt, (unsigned)want * BPP + q, A.noise_scale2, zz);
#pragma unroll
        for (int s = 0; s < 4; ++s) z[4 * q + s] = zz[s];
      }
      blk = want;
    }
    const int sub = j % SPB;
#pragma unroll
    for (int i = 0; i < D; ++i) {
      float v = z[i];
#pragma unroll
      for (int s = 1; s < SPB; ++s) v = (sub == s) ? z[s * D + i] : v;
      dB[i] = v;
    }
  }
};

// The weighted kernels (WEIGHTED = true) read the coefficients from FwdArgs fields no reverse pass reads otherwise: cS_k from
// A.G (where the unweighted kernels read G_k, the negated coefficient of dB), cG_k from A.S.  They evaluate the unweighted
// kernels' expression for a_j with G_k replaced by -cS_k and u_j by RN(-cG_k u_j), both negations and the product formed
// with __fmul_rn (opaque to the compiler's rewriting).  With (cG, cS) = (-1, -G) they are exact and the expression keeps
// its shape, so the compiler's choices (which products it contracts into FMAs differs between kernels and dimensions)
// and hence every rounding are the unweighted kernels': the gradient is bit for bit that of rlsde_rollout_bwd.
// f32 Euler-Maruyama pass, identical association to K1
template <int D>
__device__ __forceinline__ void em_step_f32(const FwdArgs& A, float (&x)[D], const float (&u)[D], const float (&dB)[D]) {
#pragma unroll
  for (int i = 0; i < D; ++i) {
    const float xi = x[i];
    const float g = __fmul_rn(__fmul_rn(A.c4a_f[i], xi), __fsub_rn(__fmul_rn(xi, xi), 1.0f));
    const float drift = __fmul_rn(__fadd_rn(-g, __fmul_rn(A.sigma_f, u[i])), A.dt_f);
    x[i] = __fadd_rn(__fadd_rn(xi, drift), __fmul_rn(A.sigma_f, dB[i]));
  }
}

// Resident blocks per SM the register allocation aims for.  Measured on B200 (K = 4e5 / 2e5, tools/bench_train.py):
//   d = 1:  2 blocks (210 registers) 63.3 ms, 3 blocks (168) 61.4 ms, 4 blocks (128, 16 B of spills) 58.2 ms
//   d = 10: 2 blocks 22.4 ms, 3 blocks 27.4 ms, 4 blocks 29.8 ms (the wider head spills)
//   d = 2 (K = 2e5): 2 blocks + swizzled tiles 8.0 ms, 3 blocks + padded tiles 7.0 ms; d = 10: 20.3 vs 20.9 ms
// unroll factor of the three 32-row inner products of a warp-pass (B200, d = 1 K = 4e5: 2 -> 36.6 ms, 4 -> 35.3, 8 -> 35.2, 32 -> 48.7; d = 10: 48.9 / 47.8 / 49.7)
#ifndef RLSDE_BWD_UNROLL
#define RLSDE_BWD_UNROLL 4
#endif
constexpr int kBwdUnroll = RLSDE_BWD_UNROLL;
#ifndef RLSDE_BWD_MIN_BLOCKS
#define RLSDE_BWD_MIN_BLOCKS(D) ((D) == 1 ? 4 : ((D) <= 4 ? 3 : 2))
#endif

// Per-warp partial gradient layout = state_dict order: W1 (H,D), b1 (H), W2 (H,H), b2 (H), W3 (D,H), b3 (D)
// RAGGED: the checkpoints come from the ragged store (ckpt_slot, rollout_fwd.cuh)
template <int D, int H, bool FAST, bool WEIGHTED = false, bool RAGGED = false>
__global__ void __launch_bounds__(128, RLSDE_BWD_MIN_BLOCKS(D)) rollout_bwd_kernel(const __grid_constant__ MlpConst<D, H> W,
                                                          const __grid_constant__ FwdArgs A, float* __restrict__ partial) {
  static_assert(H == 32 || H == 64, "column-per-lane accumulation needs H in {32, 64}");
  constexpr int CPL = H / 32;                 // columns of the HxH block owned by a lane
  constexpr bool PAD = bwd_tiles_padded(D);
  constexpr unsigned FULL = 0xffffffffu;
  constexpr int P = D * H + H + H * H + H + H * D + D;
  extern __shared__ __align__(16) float smem[];
  const int lane = threadIdx.x & 31;
  const int warp_in_block = threadIdx.x >> 5;
  const int warps_per_block = blockDim.x >> 5;
  float* tileH1 = smem + (size_t)warp_in_block * (2 * tile_floats<H, PAD>() + 64 * D);  // first-layer activations [32][H]
  float* tileB = tileH1 + tile_floats<H, PAD>();                                        // h2, then dz2, then dz1  [32][H]
  float* vecA = tileB + tile_floats<H, PAD>();                                          // a or x                  [32][D]
  const bool inject = (A.flags & RLSDE_F_NOISE_INJECTED) != 0;
  const bool s_exact = (A.flags & RLSDE_F_STOCH_INT_EXACT) != 0;
  const int C = A.ckpt_every;
  const float inv_s = FAST ? 1.0f : (float)(1.0 / RLSDE_TWO_LOG2E);
  const long long n_lanes = (long long)gridDim.x * blockDim.x;
  const long long gl = (long long)blockIdx.x * blockDim.x + threadIdx.x;

  // persistent per-lane gradient accumulators (column `lane + 32 c` of each block)
  u64 gW2[CPL][H / 2];
  // the small blocks are sums with heavy cancellation (G dB terms): their per-pass fp32 partials are added
  // into fp64 accumulators (one conversion + DADD per accumulator per pass)
  double gb2[CPL], gb1[CPL], gW1[CPL][D], gW3[CPL][D], gb3 = 0.0;
#pragma unroll
  for (int c = 0; c < CPL; ++c) {
    gb2[c] = 0.0; gb1[c] = 0.0;
#pragma unroll
    for (int j = 0; j < H / 2; ++j) gW2[c][j] = 0ull;
#pragma unroll
    for (int i = 0; i < D; ++i) { gW1[c][i] = 0.0; gW3[c][i] = 0.0; }
  }

  bool alive = false;
  long long slot = gl - n_lanes;   // next static assignment: slot += n_lanes, traj = order[slot]
  long long traj = 0;
  int kstar = 0, seg = 0;
  float Gk = 0.f, mG = 0.f;        // WEIGHTED: -cS, -cG
  float lam[D];
  float xs[BWD_MAX_SEG][D];
  NoiseCache<D> nc;
  nc.reset();
#pragma unroll
  for (int i = 0; i < D; ++i) lam[i] = 0.f;

  for (;;) {
    // ---- work assignment: static round robin over `order` (trajectories sorted by length, longest first, so
    // that the 32 lanes of a warp walk trajectories of similar length and every lane gets a similar total);
    // static => deterministic gradients.  Unfinished trajectories are skipped.
    while (!alive && slot + n_lanes < A.K) {
      slot += n_lanes;
      traj = A.order ? A.order[slot] : slot;
      const int t = A.T[traj];
      if (t >= 0 && ckpt_covered<RAGGED>(A, traj, t)) {
        alive = true; kstar = t; seg = t / C; Gk = ((const float*)A.G)[traj];
        if constexpr (WEIGHTED) { Gk = __fmul_rn(-1.0f, Gk); mG = __fmul_rn(-1.0f, ((const float*)A.S)[traj]); }
        nc.reset();
#pragma unroll
        for (int i = 0; i < D; ++i) lam[i] = 0.f;
      }
    }
    if (!__any_sync(FULL, alive)) break;
    const int seg_start = seg * C;
    const int seg_len = alive ? ((kstar + 1 - seg_start) < C ? (kstar + 1 - seg_start) : C) : 0;

    // ---- one round over the segment.  Micro-steps t = 0 .. C-2 are phase A (advance the state from
    // the checkpoint, keeping X_j in xs[]), t = C-1 .. 2C-2 are phase B (reverse sweep).  Both phases
    // share one copy of the policy-forward code; the branch on the phase is warp-uniform.
    {
#pragma unroll
      for (int i = 0; i < D; ++i) xs[0][i] = alive ? A.path[ckpt_slot<RAGGED>(A, traj, seg) * D + i] : A.x0_f[i];
    }
    for (int t = 0; t < 2 * C - 1; ++t) {
      const bool phase_a = t < C - 1;
      const int s = phase_a ? t : (2 * C - 2 - t);
      const bool ok = alive && s < seg_len;
      const int j = seg_start + s;
      float x[D], a[D];
#pragma unroll
      for (int i = 0; i < D; ++i) x[i] = xs[s][i];
      u64 dz2[H / 2];
      {
        float h2[H], u[D], dB[D];
        {
          float h1[H];
          mlp_forward_keep<D, H, FAST>(W, x, h1, h2, u);
          if (!phase_a) stage_row<H, PAD>(tileH1, lane, h1);   // h1 leaves the registers here; re-read when needed
        }
        nc.get(A, inject, ok, traj, j, dB);
        if (phase_a) {
          // X_{j+1} from X_j with K1's environment arithmetic; the policy is K1's up to the rounding of its folded tanh
          // (RLSDE_FWD_FOLDED), so the recomputed states are the forward pass's states to ~1 ulp per pass
          if (alive && s + 1 < seg_len) em_step_f32<D>(A, x, u, dB);
#pragma unroll
          for (int i = 0; i < D; ++i) xs[s + 1][i] = x[i];
          continue;
        }
#pragma unroll
        for (int i = 0; i < D; ++i) {
          float v = 0.f;
          if (ok) {
            const bool incl = s_exact ? (j < kstar) : true;
            if constexpr (WEIGHTED) v = (j < kstar ? __fmul_rn(mG, u[i]) * A.dt_f : 0.f) - (incl ? Gk * dB[i] : 0.f) + A.sigma_f * A.dt_f * lam[i];
            else v = (j < kstar ? u[i] * A.dt_f : 0.f) - (incl ? Gk * dB[i] : 0.f) + A.sigma_f * A.dt_f * lam[i];
          }
          a[i] = v;
        }
        // head: dW3[k][col] += a_k h2[col], db3[k] += a_k;  dh2 = W3^T a;  dz2 = dh2 (1 - h2^2)
        stage_row<H, PAD>(tileB, lane, h2);
#pragma unroll
        for (int i = 0; i < D; ++i) vecA[lane * D + i] = a[i];
        __syncwarp();
        {
          float pW3[CPL][D], pb3 = 0.f;
#pragma unroll
          for (int c = 0; c < CPL; ++c)
#pragma unroll
            for (int i = 0; i < D; ++i) pW3[c][i] = 0.f;
#pragma unroll(kBwdUnroll)
          for (int r = 0; r < 32; ++r) {
            float ar[D];
#pragma unroll
            for (int i = 0; i < D; ++i) ar[i] = vecA[r * D + i];
#pragma unroll
            for (int c = 0; c < CPL; ++c) {
              const float hv = tileB[swz<H, PAD>(r, lane + 32 * c)];
#pragma unroll
              for (int i = 0; i < D; ++i) pW3[c][i] = fmaf(ar[i], hv, pW3[c][i]);
            }
            if (lane < D) pb3 += vecA[r * D + lane];
          }
#pragma unroll
          for (int c = 0; c < CPL; ++c)
#pragma unroll
            for (int i = 0; i < D; ++i) gW3[c][i] += (double)pW3[c][i];
          gb3 += (double)pb3;
        }
#pragma unroll
        for (int jj = 0; jj < H / 2; ++jj) dz2[jj] = 0ull;
#pragma unroll
        for (int k = 0; k < D; ++k) {
          float w[H];
          load_row<H>(W.W3[k], w);
#pragma unroll
          for (int o = 0; o < H / 2; o += 8) RLSDE_FMA2X8(dz2, o, a[k], w);
        }
#pragma unroll
        for (int jj = 0; jj < H / 2; ++jj) {
          float d0, d1;
          unpack2(dz2[jj], d0, d1);
          dz2[jj] = pack2(d0 * fmaf(-h2[2 * jj], h2[2 * jj], 1.0f), d1 * fmaf(-h2[2 * jj + 1], h2[2 * jj + 1], 1.0f));
        }
      }
      __syncwarp();

      // hidden-hidden block: dW2[:, col] += dz2 h1[col], db2[col] += dz2[col]
#pragma unroll
      for (int q = 0; q < H / 4; ++q)
        *reinterpret_cast<ulonglong2*>(tileB + swz<H, PAD>(lane, 4 * q)) = make_ulonglong2(dz2[2 * q], dz2[2 * q + 1]);
      __syncwarp();
      float pb2[CPL];
#pragma unroll
      for (int c = 0; c < CPL; ++c) pb2[c] = 0.f;
#pragma unroll(kBwdUnroll)
      for (int r = 0; r < 32; ++r) {
        float hv[CPL];
#pragma unroll
        for (int c = 0; c < CPL; ++c) {
          hv[c] = tileH1[swz<H, PAD>(r, lane + 32 * c)];
          pb2[c] += tileB[swz<H, PAD>(r, lane + 32 * c)];
        }
#pragma unroll
        for (int q = 0; q < H / 4; q += 2) {
          const ulonglong2 w0 = *reinterpret_cast<const ulonglong2*>(tileB + swz<H, PAD>(r, 4 * q));
          const ulonglong2 w1 = *reinterpret_cast<const ulonglong2*>(tileB + swz<H, PAD>(r, 4 * q + 4));
#pragma unroll
          for (int c = 0; c < CPL; ++c) RLSDE_FMA2X4_REG(gW2[c], 2 * q, hv[c], w0.x, w0.y, w1.x, w1.y);
        }
      }
#pragma unroll
      for (int c = 0; c < CPL; ++c) gb2[c] += (double)pb2[c];
      __syncwarp();
      // dh1 = W2^T dz2 (dot form on the input-major, pre-scaled W2t);  dz1 = dh1 (1 - h1^2), streamed
      // four at a time into tileB (the dz2 tile is dead now) while dx = W1^T dz1 accumulates on the fly
      float dxa[D];
#pragma unroll
      for (int i = 0; i < D; ++i) dxa[i] = 0.f;
#pragma unroll
      for (int q = 0; q < H / 4; ++q) {
        const float4 hq = *reinterpret_cast<const float4*>(tileH1 + swz<H, PAD>(lane, 4 * q));
        const float hloc[4] = {hq.x, hq.y, hq.z, hq.w};
        float dq[4], w1q[D][4];
#pragma unroll
        for (int d = 0; d < D; ++d) {
          const float4 t = reinterpret_cast<const float4*>(&W.W1t[d][0])[q];
          w1q[d][0] = t.x; w1q[d][1] = t.y; w1q[d][2] = t.z; w1q[d][3] = t.w;
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int i = 4 * q + e;
          u64 acc = 0ull;
          float w[H];
          load_row<H>(W.W2t[i], w);
#pragma unroll
          for (int o = 0; o < H / 2; o += 4) RLSDE_DOTP4(acc, dz2, o, w);
          float lo, hi;
          unpack2(acc, lo, hi);
          dq[e] = (lo + hi) * inv_s * fmaf(-hloc[e], hloc[e], 1.0f);
#pragma unroll
          for (int d = 0; d < D; ++d) dxa[d] = fmaf(w1q[d][e], dq[e], dxa[d]);
        }
        *reinterpret_cast<float4*>(tileB + swz<H, PAD>(lane, 4 * q)) = make_float4(dq[0], dq[1], dq[2], dq[3]);
      }
#pragma unroll
      for (int i = 0; i < D; ++i) vecA[lane * D + i] = x[i];
      __syncwarp();

      // input block: dW1[col][i] += dz1[col] x_i, db1[col] += dz1[col]
      {
        float pb1[CPL], pW1[CPL][D];
#pragma unroll
        for (int c = 0; c < CPL; ++c) {
          pb1[c] = 0.f;
#pragma unroll
          for (int i = 0; i < D; ++i) pW1[c][i] = 0.f;
        }
#pragma unroll(kBwdUnroll)
        for (int r = 0; r < 32; ++r) {
          float xr[D];
#pragma unroll
          for (int i = 0; i < D; ++i) xr[i] = vecA[r * D + i];
#pragma unroll
          for (int c = 0; c < CPL; ++c) {
            const float dv = tileB[swz<H, PAD>(r, lane + 32 * c)];
            pb1[c] += dv;
#pragma unroll
            for (int i = 0; i < D; ++i) pW1[c][i] = fmaf(dv, xr[i], pW1[c][i]);
          }
        }
#pragma unroll
        for (int c = 0; c < CPL; ++c) {
          gb1[c] += (double)pb1[c];
#pragma unroll
          for (int i = 0; i < D; ++i) gW1[c][i] += (double)pW1[c][i];
        }
      }
      __syncwarp();
      if (ok) {
#pragma unroll
        for (int i = 0; i < D; ++i) {
          const float dx = dxa[i] * inv_s;
          // d x_{j+1} / d x_j = 1 - dt * hessian,  hessian = 4 alpha (3 x^2 - 1)
          const float hess = A.c4a_f[i] * fmaf(3.0f * x[i], x[i], -1.0f);
          lam[i] = fmaf(lam[i], fmaf(-A.dt_f, hess, 1.0f), dx);
        }
      }
    }
    if (alive) {
      --seg;
      if (seg < 0) alive = false;
    }
  }

  // ---- per-warp partial gradient: in-warp sums are already formed (each lane owns whole columns)
  const long long gw = (long long)blockIdx.x * warps_per_block + warp_in_block;
  float* out = partial + gw * P;
  float* oW1 = out;
  float* ob1 = oW1 + H * D;
  float* oW2 = ob1 + H;
  float* ob2 = oW2 + H * H;
  float* oW3 = ob2 + H;
  float* ob3 = oW3 + D * H;
#pragma unroll
  for (int c = 0; c < CPL; ++c) {
    const int col = lane + 32 * c;
#pragma unroll
    for (int i = 0; i < D; ++i) { oW1[col * D + i] = (float)gW1[c][i]; oW3[i * H + col] = (float)gW3[c][i]; }
    ob1[col] = (float)gb1[c];
    ob2[col] = (float)gb2[c];
#pragma unroll
    for (int jj = 0; jj < H / 2; ++jj) {
      float lo, hi;
      unpack2(gW2[c][jj], lo, hi);
      oW2[(2 * jj) * H + col] = lo;        // dW2[j][i]: j = output (delta) index, i = input (column) index
      oW2[(2 * jj + 1) * H + col] = hi;
    }
  }
  if (lane < D) ob3[lane] = (float)gb3;
}

template <int D, int H, bool WEIGHTED = false, bool RAGGED = false>
int launch_rollout_bwd(const float* params_host, const FwdArgs& args, float scale, float* grad, float* partial,
                       int sm_count, cudaStream_t stream);

}  // namespace rlsde
