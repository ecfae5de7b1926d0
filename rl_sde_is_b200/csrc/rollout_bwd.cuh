// Reverse (adjoint) pass of the REINFORCE surrogate loss through the whole rollout: what every reverse family (K2m, K2w,
// K2x, K2u) computes, and the pieces they share.
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

}  // namespace rlsde
