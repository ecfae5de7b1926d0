// Per-trajectory state and ONE environment pass with the reference's arithmetic, for kernels in which a thread owns a
// trajectory but the policy is evaluated elsewhere (rollout_umma.cuh: on the tensor cores).  The pass is K1's
// (rollout_fwd.cuh; SURVEY.md Appendix A): hit test on the CURRENT state, the stochastic integral also on the detecting
// pass, reward / Euler-Maruyama update with torch's (f32) or NumPy's (f64 state, RLSDE_F_STATE_F64) association and no
// FMA contraction, so that, given the same action and increment, next state / reward are bit-identical to the
// reference's.  Replaces one env.step[_torch] call (environments.py:139-162, 201-226) plus the bookkeeping around it in
// sample_loss_vectorized (reinforce_deterministic_core.py:58-88) / test_policy_vectorized (approximate_methods.py:604-638).
#pragma once
#include "rollout_fwd.cuh"

namespace rlsde {

// Cell of the 1-D state grid of cfg.n_grid / grid_lo / grid_hi / grid_h that holds x (state precision, widened to double):
// idx = floor((clip(x, lo, hi) - lo) / h), clamped to [0, n_grid - 1]   (environments.py:318-321).  The l2 error of
// TrajOwner::pass and the tabulated control of rollout_fwd_tab_kernel (fwd_tab_d1.cu) both index with it.
__device__ __forceinline__ long long grid_index(const FwdArgs& A, double x) {
  const double xc = x < A.grid_lo ? A.grid_lo : (x > A.grid_hi ? A.grid_hi : x);
  const long long gi = (long long)floor((xc - A.grid_lo) / A.grid_h);
  return gi < 0 ? 0 : (gi >= A.n_grid ? A.n_grid - 1 : gi);
}

// BRIDGE: the Brownian-bridge hit test between passes (bridge_project, rollout_fwd.cuh; d = 1 only)
// RAGGED: checkpoints go to the ragged store (ckpt_slot, rollout_fwd.cuh)
template <int D, bool F64, bool BRIDGE = false, bool RAGGED = false>
struct TrajOwner {
  typedef typename RealT<F64>::type real;
  static constexpr int SPB = NoisePlan<D>::SPB;
  static constexpr int BPP = NoisePlan<D>::BPP;
  static constexpr int NZ = NoisePlan<D>::NZ;
  bool alive, exhausted;
  long long traj;
  int k, ck;
  real x[D];
  real G, S, L2;
  float z[NZ];
  double inv_s2dt;

  __device__ __forceinline__ void init(const FwdArgs& A) {
    alive = false; exhausted = false; traj = 0; k = 0; ck = 0; G = 0; S = 0; L2 = 0;
    inv_s2dt = BRIDGE ? bridge_inv_s2dt(A) : 0.0;
#pragma unroll
    for (int i = 0; i < D; ++i) x[i] = F64 ? (real)A.x0_d[i] : (real)A.x0_f[i];
#pragma unroll
    for (int i = 0; i < NZ; ++i) z[i] = 0.f;
  }
  __device__ __forceinline__ void start(const FwdArgs& A, long long idx) {
    traj = idx; k = 0; ck = 0; alive = true; G = 0; S = 0; L2 = 0;
#pragma unroll
    for (int i = 0; i < D; ++i) x[i] = F64 ? (real)A.x0_d[i] : (real)A.x0_f[i];
  }
  __device__ __forceinline__ void write_out(const FwdArgs& A, real Sout, real logw_S, int t_out) {
    if (F64) {
      ((double*)A.G)[traj] = (double)G; ((double*)A.S)[traj] = (double)Sout;
      if (A.l2) ((double*)A.l2)[traj] = (double)L2;
      if (A.logw) ((double*)A.logw)[traj] = (double)G - (double)logw_S;
    } else {
      ((float*)A.G)[traj] = (float)G; ((float*)A.S)[traj] = (float)Sout;
      if (A.l2) ((float*)A.l2)[traj] = (float)L2;
      if (A.logw) ((float*)A.logw)[traj] = (float)G - (float)logw_S;
    }
    A.T[traj] = t_out;
  }
  // one pass with action u; call only while alive
  __device__ __forceinline__ void pass(const FwdArgs& A, const float (&u)[D], long long lim) {
    const bool inject = (A.flags & RLSDE_F_NOISE_INJECTED) != 0;
    const bool s_exact = (A.flags & RLSDE_F_STOCH_INT_EXACT) != 0;
    const bool store_path = (A.flags & RLSDE_F_STORE_PATH) != 0 && A.path != nullptr;
    const bool want_l2 = (D == 1) && A.policy_opt != nullptr && A.l2 != nullptr;
    float dB[D];
    if (inject) {
      const long long row = (long long)k * A.K_global + (A.traj_offset + traj);
#pragma unroll
      for (int i = 0; i < D; ++i) dB[i] = k < lim ? __ldg(A.noise + row * D + i) : 0.f;
    } else {
      if ((k % SPB) == 0) {
        const unsigned long long gt = (unsigned long long)(A.traj_offset + traj);
#pragma unroll
        for (int q = 0; q < BPP; ++q) {
          float zz[4];
          noise_block(A.seed, gt, (unsigned)(k / SPB) * BPP + q, A.noise_scale2, zz);
#pragma unroll
          for (int s = 0; s < 4; ++s) z[4 * q + s] = zz[s];
        }
      }
      const int sub = k % SPB;
#pragma unroll
      for (int i = 0; i < D; ++i) {
        float v = z[i];
#pragma unroll
        for (int s = 1; s < SPB; ++s) v = (sub == s) ? z[s * D + i] : v;
        dB[i] = v;
      }
    }
    bool hit;
    if (A.hit_rule == RLSDE_HIT_X0_IN_LB_RB) {
      hit = F64 ? ((double)x[0] >= A.lb_d && (double)x[0] <= A.rb_d) : ((float)x[0] >= A.lb_f && (float)x[0] <= A.rb_f);
    } else {
      hit = true;
#pragma unroll
      for (int i = 0; i < D; ++i) hit = hit && (F64 ? ((double)x[i] >= A.lb_d) : ((float)x[i] >= A.lb_f));
    }
    real su = 0;
    float n2 = 0.f;
#pragma unroll
    for (int i = 0; i < D; ++i) {
      su = (i == 0) ? mul_rn((real)u[i], (real)dB[i]) : add_rn(su, mul_rn((real)u[i], (real)dB[i]));
      n2 = (i == 0) ? __fmul_rn(u[i], u[i]) : __fadd_rn(n2, __fmul_rn(u[i], u[i]));
    }
    const real S_prev = S;
    S = add_rn(S, su);
    if (want_l2) {
      const long long gi = grid_index(A, (double)x[0]);
      const float du = __fsub_rn(u[0], __ldg(A.policy_opt + gi));
      L2 = F64 ? (real)__dadd_rn((double)L2, __dmul_rn((double)__fmul_rn(du, du), A.dt_d))
               : (real)__fadd_rn((float)L2, __fmul_rn(__fmul_rn(du, du), A.dt_f));
    }
    if (store_path) {
      if (ck == 0) {
        const int ci = A.ckpt_log2 >= 0 ? (k >> A.ckpt_log2) : (k / A.ckpt_every);
        const long long row = ckpt_slot<RAGGED>(A, traj, ci);
        if (ckpt_writable<RAGGED>(A, traj, row)) {
          float* dst = A.path + row * D;
#pragma unroll
          for (int i = 0; i < D; ++i) dst[i] = (float)x[i];
        }
        ck = A.ckpt_every;
      }
      --ck;
    }
    if (hit) {
      write_out(A, s_exact ? S_prev : S, S_prev, k);
      alive = false;
      return;
    }
    const float nn = (D == 1) ? n2 : __fmul_rn(sqrtf(n2), sqrtf(n2));
    if (F64) G = (real)__dadd_rn((double)G, -__dmul_rn(__dadd_rn(1.0, (double)__fmul_rn(0.5f, nn)), A.dt_d));
    else G = (real)__fadd_rn((float)G, -__fmul_rn(__fadd_rn(1.0f, __fmul_rn(0.5f, nn)), A.dt_f));
    const real x_prev = x[0];
#pragma unroll
    for (int i = 0; i < D; ++i) {
      if (F64) {
        const double xi = (double)x[i];
        double g;
        if (k == 0) {   // numpy promotion on the float32 initial state (SURVEY App. A-5), as in K1
          const float xs_ = (float)xi;
          g = (D == 1) ? (double)__fmul_rn(__fmul_rn(A.c4a_f[i], xs_), __fsub_rn(__fmul_rn(xs_, xs_), 1.0f))
                       : __dmul_rn(__dmul_rn(A.c4a_d[i], xi), (double)__fsub_rn(__fmul_rn(xs_, xs_), 1.0f));
        } else {
          g = __dmul_rn(__dmul_rn(A.c4a_d[i], xi), __dsub_rn(__dmul_rn(xi, xi), 1.0));
        }
        const double drift = __dmul_rn(__dadd_rn(-g, __dmul_rn(A.sigma_d, (double)u[i])), A.dt_d);
        x[i] = (real)__dadd_rn(__dadd_rn(xi, drift), __dmul_rn(A.sigma_d, (double)dB[i]));
      } else {
        const float xi = (float)x[i];
        const float g = __fmul_rn(__fmul_rn(A.c4a_f[i], xi), __fsub_rn(__fmul_rn(xi, xi), 1.0f));
        const float drift = __fmul_rn(__fadd_rn(-g, __fmul_rn(A.sigma_f, u[i])), A.dt_f);
        x[i] = (real)__fadd_rn(__fadd_rn(xi, drift), __fmul_rn(A.sigma_f, dB[i]));
      }
    }
    if constexpr (BRIDGE) bridge_project(A, inv_s2dt, (unsigned long long)(A.traj_offset + traj), k, x_prev, x[0]);
    ++k;
    if (k >= lim) {       // not detected within the pass budget: flagged, never garbage
      write_out(A, S, S, -1);
      alive = false;
    }
  }
};

}  // namespace rlsde
