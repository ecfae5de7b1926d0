// K1w / K2w: latency-oriented variants of the rollout kernels for SMALL batches (e.g. the reference's
// REINFORCE configuration, K = 100: reinforce_deterministic_core.py:226-243), where one trajectory per thread
// cannot fill the machine and an iteration costs (longest trajectory) x (latency of one pass).
//
// One WARP per trajectory, hidden width 32: lane j owns hidden unit j.  Its weight rows live in registers for
// the whole launch; the 32 activations of a layer are exchanged through 128 bytes of shared memory per warp
// (one STS + eight broadcast LDS.128); the head and the state adjoint are butterfly reductions.  A pass costs
// ~400 cycles (forward) instead of the ~5 500 cycles a lone warp of the thread-per-trajectory kernel needs
// (there, every FFMA2 pair waits for an LDCU.128: profiles/r01/README.md).
//
// Semantics are those of K1 and of the reverse pass (rollout_fwd.cuh, rollout_bwd.cuh): same per-pass arithmetic with the
// reference's association for the environment step, same Philox stream, same outputs.  The dot products are
// summed in a different order than in K1, so per-trajectory values agree with K1 to rounding (~1e-6 relative),
// not bit for bit; the reverse kernel recomputes the forward pass with THIS kernel's arithmetic.
#pragma once
#include "rollout_bwd.cuh"

namespace rlsde {

constexpr int WARP_H = 32;

template <bool FAST>
__device__ __forceinline__ float tanh_scalar(float zp) {   // zp = pre-activation, pre-scaled by 2 log2(e) unless FAST
  if constexpr (FAST) return mufu_tanh(zp);
  return fmaf(-2.0f, mufu_rcp(mufu_ex2(zp) + 1.0f), 1.0f);
}

__device__ __forceinline__ float warp_sum(float v) {        // identical result in every lane
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// all 32 values of a lane-distributed vector, through this warp's 32-float slot of shared memory
__device__ __forceinline__ void warp_allgather(float* slot, int lane, float mine, float (&all)[WARP_H]) {
  slot[lane] = mine;
  __syncwarp();
#pragma unroll
  for (int q = 0; q < WARP_H / 4; ++q) {
    const float4 t = reinterpret_cast<const float4*>(slot)[q];
    all[4 * q] = t.x; all[4 * q + 1] = t.y; all[4 * q + 2] = t.z; all[4 * q + 3] = t.w;
  }
  __syncwarp();
}

// Pin a value in a register: without this the compiler re-materialises the lane-owned weights every pass with
// lane-indexed constant loads (LDC c[0][lane*4 + ...]), which serialise 32-way and dominated the pass latency.
__device__ __forceinline__ void pin(float& v) { asm volatile("" : "+f"(v)); }

// lane-owned policy parameters (pre-scaled like MlpConst)
template <int D>
struct LaneParams {
  float w1[D], b1;            // row `lane` of W1, bias
  float w2row[WARP_H], b2;    // row `lane` of W2: weights into hidden unit `lane`
  float w3[D];                // column `lane` of W3
  float b3[D];                // head bias (uniform)
  // narrow heads: the whole of W3 in every lane, so that each lane can sum the head itself (see warp_policy)
  static constexpr bool HEAD_LOCAL = D <= 2;
  float w3all[HEAD_LOCAL ? D : 1][WARP_H];
  __device__ __forceinline__ void load(const MlpConst<D, WARP_H>& W, int lane) {   // W: kernel parameter or device memory
#pragma unroll
    for (int i = 0; i < D; ++i) { w1[i] = W.W1t[i][lane]; w3[i] = W.W3[i][lane]; b3[i] = W.b3[i]; pin(w1[i]); pin(w3[i]); }
    if constexpr (HEAD_LOCAL) {
#pragma unroll
      for (int i = 0; i < D; ++i)
#pragma unroll
        for (int j = 0; j < WARP_H; ++j) { w3all[i][j] = W.W3[i][j]; pin(w3all[i][j]); }
    }
    b1 = W.b1[lane]; pin(b1);
    b2 = W.b2[lane]; pin(b2);
#pragma unroll
    for (int i = 0; i < WARP_H; ++i) { w2row[i] = W.W2t[i][lane]; pin(w2row[i]); }
  }
};

// policy forward for one state (replicated in all lanes): returns u (replicated), this lane's h1 / h2 and all h1
template <int D, bool FAST>
__device__ __forceinline__ void warp_policy(const LaneParams<D>& P, float* slot, int lane, const float (&x)[D], float& h1,
                                            float (&h1_all)[WARP_H], float& h2, float (&u)[D]) {
  float z = P.b1;
#pragma unroll
  for (int i = 0; i < D; ++i) z = fmaf(x[i], P.w1[i], z);
  h1 = tanh_scalar<FAST>(z);
  warp_allgather(slot, lane, h1, h1_all);
  float a0 = P.b2, a1 = 0.f, a2 = 0.f, a3 = 0.f;            // four chains
#pragma unroll
  for (int i = 0; i < WARP_H; i += 4) {
    a0 = fmaf(h1_all[i], P.w2row[i], a0);
    a1 = fmaf(h1_all[i + 1], P.w2row[i + 1], a1);
    a2 = fmaf(h1_all[i + 2], P.w2row[i + 2], a2);
    a3 = fmaf(h1_all[i + 3], P.w2row[i + 3], a3);
  }
  h2 = tanh_scalar<FAST>((a0 + a1) + (a2 + a3));
  if constexpr (LaneParams<D>::HEAD_LOCAL) {
    // head: a second exchange through shared memory and four FMA chains per lane (~100 cycles) instead of a five-level
    // shuffle butterfly (~150 cycles) on the critical path of the pass
    float h2_all[WARP_H];
    warp_allgather(slot, lane, h2, h2_all);
#pragma unroll
    for (int k = 0; k < D; ++k) {
      float c0 = P.b3[k], c1 = 0.f, c2 = 0.f, c3 = 0.f;
#pragma unroll
      for (int j = 0; j < WARP_H; j += 4) {
        c0 = fmaf(h2_all[j], P.w3all[k][j], c0);
        c1 = fmaf(h2_all[j + 1], P.w3all[k][j + 1], c1);
        c2 = fmaf(h2_all[j + 2], P.w3all[k][j + 2], c2);
        c3 = fmaf(h2_all[j + 3], P.w3all[k][j + 3], c3);
      }
      u[k] = (c0 + c1) + (c2 + c3);
    }
  } else {
#pragma unroll
    for (int k = 0; k < D; ++k) u[k] = P.b3[k] + warp_sum(P.w3[k] * h2);
  }
}

// Same policy with K1's summation orders (rollout_fwd.cuh / common.cuh): one FMA chain per hidden unit over the inputs
// in index order, the head as two chains over the even / odd activations added at the end.  ~70 cycles slower per pass
// than warp_policy, but bit-identical to the thread-per-trajectory kernel, so a trajectory that K1 hands over (the last
// long trajectories of a launch) continues exactly as K1 would have continued it.
// (With RLSDE_FWD_FOLDED, K1 hands r = 1 / (exp(2 z) + 1) from layer to layer and its weight image carries the rest of the
// tanh: P and W are then loaded from a pack_mlp_const_folded image and the activation here stops at r as well.)
template <bool FAST>
__device__ __forceinline__ float act_like_k1(float zp) {
  if constexpr (!FAST && RLSDE_FWD_FOLDED) return mufu_rcp(mufu_ex2(zp) + 1.0f);
  return tanh_scalar<FAST>(zp);
}
template <int D, bool FAST>
__device__ __forceinline__ void warp_policy_exact(const LaneParams<D>& P, const MlpConst<D, WARP_H>& W, float* slot, int lane,
                                                  const float (&x)[D], float (&u)[D]) {
  float z = P.b1;
#pragma unroll
  for (int i = 0; i < D; ++i) z = fmaf(x[i], P.w1[i], z);
  float all[WARP_H];
  warp_allgather(slot, lane, act_like_k1<FAST>(z), all);
  float a = P.b2;
#pragma unroll
  for (int i = 0; i < WARP_H; ++i) a = fmaf(all[i], P.w2row[i], a);
  warp_allgather(slot, lane, act_like_k1<FAST>(a), all);
#pragma unroll
  for (int k = 0; k < D; ++k) {
    float lo = W.b3[k], hi = 0.0f;
#pragma unroll
    for (int j = 0; j < WARP_H; j += 2) {
      lo = fmaf(all[j], W.W3[k][j], lo);
      hi = fmaf(all[j + 1], W.W3[k][j + 1], hi);
    }
    u[k] = __fadd_rn(lo, hi);
  }
}

// ------------------------------------------------------------------------------------------------ forward
// RESUME = true: the work items are the continuation records K1 left in the ring when it handed the last live
// trajectories of its launch over (rollout_fwd.cuh); they are continued with K1's arithmetic: warp_policy_exact, or with
// MMA (K1 evaluated its policy with mlp_forward_mma) the same tensor-core sequence with the trajectory's state in all
// 32 rows of the tile.
// BRIDGE: the Brownian-bridge hit test between passes (bridge_project, rollout_fwd.cuh; d = 1 only)
// RAGGED: checkpoints go to the ragged store (ckpt_slot, rollout_fwd.cuh)
template <int D, bool F64, bool FAST, bool RESUME, bool MMA = false, bool BRIDGE = false, bool RAGGED = false>
__global__ void __launch_bounds__(128, (D <= 2 ? 4 : 1)) rollout_fwd_warp_kernel(const __grid_constant__ MlpConst<D, WARP_H> W_param,
                                                               const MlpConst<D, WARP_H>* __restrict__ W_dev,
                                                               const __grid_constant__ FwdArgs A,
                                                               const __grid_constant__ typename FwdMmaSel<D, MMA>::type M) {
  static_assert(!MMA || RESUME, "the tensor-core policy continues K1's trajectories");
  // the policy comes by value (host parameters) or, for the device-resident training loop, from device memory
  const MlpConst<D, WARP_H>& W = W_dev != nullptr ? *W_dev : W_param;
  typedef typename RealT<F64>::type real;
  constexpr int SPB = NoisePlan<D>::SPB;
  constexpr int BPP = NoisePlan<D>::BPP;
  __shared__ __align__(16) float slots[4][WARP_H];
  __shared__ uint4 s_mma[MMA ? mlp_mma_smem_words<D>() : 1];
  if constexpr (MMA) {
    for (int i = threadIdx.x; i < mlp_mma_smem_words<D>(); i += blockDim.x) s_mma[i] = reinterpret_cast<const uint4*>(&M)[i];
    __syncthreads();
  }
  const int lane = threadIdx.x & 31;
  float* slot = slots[threadIdx.x >> 5];
  const long long n_warps = (long long)gridDim.x * (blockDim.x >> 5);
  const long long gw = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const bool inject = (A.flags & RLSDE_F_NOISE_INJECTED) != 0;
  const bool s_exact = (A.flags & RLSDE_F_STOCH_INT_EXACT) != 0;
  const bool store_path = (A.flags & RLSDE_F_STORE_PATH) != 0 && A.path != nullptr;
  const bool want_l2 = (D == 1) && A.policy_opt != nullptr && A.l2 != nullptr;
  const long long lim = inject ? (A.noise_steps < A.n_steps_lim ? A.noise_steps : A.n_steps_lim) : A.n_steps_lim;
  const double inv_s2dt = BRIDGE ? bridge_inv_s2dt(A) : 0.0;
  LaneParams<D> P;
  P.load(W, lane);

  typedef ContRec<D, F64> Rec;
  // RESUME: the records K1 appended when it handed its tail over; none if its launch went for time slices instead
  // (q_ctrl[5] == 1: the ring then holds the FIFO's consumed records)
  const long long n_items = RESUME ? (A.q_ctrl[5] == 1 ? 0 : (long long)A.q_ctrl[1]) : A.K;
  // fresh batches: static round robin (deterministic reverse-pass partials rely on nothing here, but it is free);
  // resumed tails: lengths differ by orders of magnitude, so warps take records from a counter as they become free
  auto next_item = [&](long long prev) -> long long {
    if constexpr (RESUME) {
      unsigned long long i = 0;
      if (lane == 0) i = atomicAdd(A.q_ctrl + 3, 1ull);
      return (long long)__shfl_sync(0xffffffffu, i, 0);
    } else {
      return prev < 0 ? gw : prev + n_warps;
    }
  };
  for (long long item = next_item(-1); item < n_items; item = next_item(item)) {
    long long traj = item;
    int k_first = 0;
    real x[D];
    real G = 0, S = 0, L2 = 0;
    if constexpr (RESUME) {
      const Rec* r = reinterpret_cast<const Rec*>(A.q_ring) + item;
      traj = r->traj; k_first = r->k; G = r->G; S = r->S; L2 = r->L2;
#pragma unroll
      for (int i = 0; i < D; ++i) x[i] = r->x[i];
    } else {
#pragma unroll
      for (int i = 0; i < D; ++i) x[i] = F64 ? (real)A.x0_d[i] : (real)A.x0_f[i];
    }
    float z[NoisePlan<D>::NZ];
    long long t_out = -1;
    int ck = 0;
    if (RESUME && store_path) {
      const int rem = k_first % A.ckpt_every;
      ck = rem ? A.ckpt_every - rem : 0;
    }
    for (int k = k_first; k < (int)lim; ++k) {
      if (!inject && (k % SPB) == 0) {
        const unsigned long long gt = (unsigned long long)(A.traj_offset + traj);
#pragma unroll
        for (int q = 0; q < BPP; ++q) {
          float zz[4];
          noise_block(A.seed, gt, (unsigned)(k / SPB) * BPP + q, A.noise_scale2, zz);
#pragma unroll
          for (int s = 0; s < 4; ++s) z[4 * q + s] = zz[s];
        }
      }
      float xf[D], u[D], dB[D];
#pragma unroll
      for (int i = 0; i < D; ++i) xf[i] = (float)x[i];
      if constexpr (MMA) {
        mlp_forward_mma<D, FAST, true>(s_mma, reinterpret_cast<const float4*>(s_mma + MLP_MMA_FRAG_WORDS), M.b3, lane, xf, u);
      } else if constexpr (RESUME) {
        warp_policy_exact<D, FAST>(P, W, slot, lane, xf, u);
      } else {
        float h1, h2, h1_all[WARP_H];
        warp_policy<D, FAST>(P, slot, lane, xf, h1, h1_all, h2, u);
      }
      if (inject) {
        const long long row = (long long)k * A.K_global + (A.traj_offset + traj);
#pragma unroll
        for (int i = 0; i < D; ++i) dB[i] = __ldg(A.noise + row * D + i);
      } else {
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
        double xc = (double)x[0];
        xc = xc < A.grid_lo ? A.grid_lo : (xc > A.grid_hi ? A.grid_hi : xc);
        long long gi = (long long)floor((xc - A.grid_lo) / A.grid_h);
        gi = gi < 0 ? 0 : (gi >= A.n_grid ? A.n_grid - 1 : gi);
        const float du = __fsub_rn(u[0], __ldg(A.policy_opt + gi));
        L2 = F64 ? (real)__dadd_rn((double)L2, __dmul_rn((double)__fmul_rn(du, du), A.dt_d))
                 : (real)__fadd_rn((float)L2, __fmul_rn(__fmul_rn(du, du), A.dt_f));
      }
      if (store_path) {
        if (ck == 0) {
          const int ci = A.ckpt_log2 >= 0 ? (k >> A.ckpt_log2) : (k / A.ckpt_every);      // no integer division per pass
          const long long row = ckpt_slot<RAGGED>(A, traj, ci);
          if (ckpt_writable<RAGGED>(A, traj, row)) {
#pragma unroll
            for (int i = 0; i < D; ++i)
              if (lane == i) A.path[row * D + i] = (float)x[i];
          }
          ck = A.ckpt_every;
        }
        --ck;
      }
      if (hit) {
        S = s_exact ? S_prev : S;
        t_out = k;
        if (lane == 0 && A.logw) {
          if (F64) ((double*)A.logw)[traj] = (double)G - (double)S_prev;
          else ((float*)A.logw)[traj] = (float)G - (float)S_prev;
        }
        break;
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
            const float xs = (float)xi;
            g = (D == 1) ? (double)__fmul_rn(__fmul_rn(A.c4a_f[i], xs), __fsub_rn(__fmul_rn(xs, xs), 1.0f))
                         : __dmul_rn(__dmul_rn(A.c4a_d[i], xi), (double)__fsub_rn(__fmul_rn(xs, xs), 1.0f));
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
    }
    if (lane == 0) {
      if (t_out < 0 && A.logw) {
        if (F64) ((double*)A.logw)[traj] = (double)G - (double)S;
        else ((float*)A.logw)[traj] = (float)G - (float)S;
      }
      if (F64) {
        ((double*)A.G)[traj] = (double)G; ((double*)A.S)[traj] = (double)S;
        if (A.l2) ((double*)A.l2)[traj] = (double)L2;
      } else {
        ((float*)A.G)[traj] = (float)G; ((float*)A.S)[traj] = (float)S;
        if (A.l2) ((float*)A.l2)[traj] = (float)L2;
      }
      A.T[traj] = (int)t_out;
    }
  }
}

// ------------------------------------------------------------------------------------------------ reverse
// Needs every state (ckpt_every == 1).  Lane j accumulates row j of dW2 / dW1, column j of dW3, entry j of db1 / db2.
// WEIGHTED: per-trajectory coefficients (rollout_bwd.cuh, the comment above em_step_f32).
// RAGGED: the states come from the ragged store (ckpt_slot, rollout_fwd.cuh)
template <int D, bool FAST, bool WEIGHTED = false, bool RAGGED = false>
__global__ void __launch_bounds__(128) rollout_bwd_warp_kernel(const __grid_constant__ MlpConst<D, WARP_H> W_param,
                                                               const MlpConst<D, WARP_H>* __restrict__ W_dev,
                                                               const __grid_constant__ FwdArgs A, float* __restrict__ partial) {
  const MlpConst<D, WARP_H>& W = W_dev != nullptr ? *W_dev : W_param;
  constexpr int H = WARP_H;
  constexpr int P_ = D * H + H + H * H + H + H * D + D;
  __shared__ __align__(16) float slots[4][WARP_H];
  const int lane = threadIdx.x & 31;
  float* slot = slots[threadIdx.x >> 5];
  const long long n_warps = (long long)gridDim.x * (blockDim.x >> 5);
  const long long gw = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const bool inject = (A.flags & RLSDE_F_NOISE_INJECTED) != 0;
  const bool s_exact = (A.flags & RLSDE_F_STOCH_INT_EXACT) != 0;
  const float inv_s = FAST ? 1.0f : (float)(1.0 / RLSDE_TWO_LOG2E);
  LaneParams<D> P;
  P.load(W, lane);
  float w2col[H];                       // column `lane` of W2 (pre-scaled): weights OUT of hidden unit `lane`
#pragma unroll
  for (int j = 0; j < H; ++j) { w2col[j] = W.W2t[lane][j]; pin(w2col[j]); }
  float gW2[H], gW1[D], gW3[D], gb1 = 0.f, gb2 = 0.f, gb3[D];
#pragma unroll
  for (int i = 0; i < H; ++i) gW2[i] = 0.f;
#pragma unroll
  for (int i = 0; i < D; ++i) { gW1[i] = 0.f; gW3[i] = 0.f; gb3[i] = 0.f; }
  NoiseCache<D> nc;

  // static round robin over the (optionally length-sorted) list: deterministic per-warp partial sums
  for (long long item = gw; item < A.K; item += n_warps) {
    const long long traj = A.order ? A.order[item] : item;
    const int kstar = A.T[traj];
    if (kstar < 0 || !ckpt_covered<RAGGED>(A, traj, kstar)) continue;
    const float Gk = ((const float*)A.G)[traj];                       // WEIGHTED: cS
    const float nS = WEIGHTED ? __fmul_rn(-1.0f, Gk) : 0.f;
    const float mG = WEIGHTED ? __fmul_rn(-1.0f, ((const float*)A.S)[traj]) : 0.f;
    float lam[D];
#pragma unroll
    for (int i = 0; i < D; ++i) lam[i] = 0.f;
    nc.reset();
    // X_j is loaded one pass ahead: the load's latency (~500 cycles) overlaps the previous pass's arithmetic instead
    // of heading the dependency chain of its own pass
    const float* xp = A.path + ckpt_slot<RAGGED>(A, traj, 0) * D;
    float x_next[D];
#pragma unroll
    for (int i = 0; i < D; ++i) x_next[i] = xp[(long long)kstar * D + i];
    for (int j = kstar; j >= 0; --j) {
      float x[D], u[D], h1, h2, h1_all[H], dB[D], a[D];
#pragma unroll
      for (int i = 0; i < D; ++i) x[i] = x_next[i];
      if (j > 0) {
#pragma unroll
        for (int i = 0; i < D; ++i) x_next[i] = xp[(long long)(j - 1) * D + i];
      }
      warp_policy<D, FAST>(P, slot, lane, x, h1, h1_all, h2, u);
      nc.get(A, inject, true, traj, j, dB);
      float dh2 = 0.f;
#pragma unroll
      for (int i = 0; i < D; ++i) {
        const bool incl = s_exact ? (j < kstar) : true;
        if constexpr (WEIGHTED) a[i] = (j < kstar ? __fmul_rn(mG, u[i]) * A.dt_f : 0.f) - (incl ? nS * dB[i] : 0.f) + A.sigma_f * A.dt_f * lam[i];
        else a[i] = (j < kstar ? u[i] * A.dt_f : 0.f) - (incl ? Gk * dB[i] : 0.f) + A.sigma_f * A.dt_f * lam[i];
        gW3[i] = fmaf(a[i], h2, gW3[i]);
        gb3[i] += a[i];
        dh2 = fmaf(P.w3[i], a[i], dh2);
      }
      const float dz2 = dh2 * fmaf(-h2, h2, 1.0f);
      gb2 += dz2;
#pragma unroll
      for (int i = 0; i < H; ++i) gW2[i] = fmaf(dz2, h1_all[i], gW2[i]);
      float dz2_all[H];
      warp_allgather(slot, lane, dz2, dz2_all);
      float c0 = 0.f, c1 = 0.f, c2 = 0.f, c3 = 0.f;
#pragma unroll
      for (int jj = 0; jj < H; jj += 4) {
        c0 = fmaf(w2col[jj], dz2_all[jj], c0);
        c1 = fmaf(w2col[jj + 1], dz2_all[jj + 1], c1);
        c2 = fmaf(w2col[jj + 2], dz2_all[jj + 2], c2);
        c3 = fmaf(w2col[jj + 3], dz2_all[jj + 3], c3);
      }
      const float dz1 = ((c0 + c1) + (c2 + c3)) * inv_s * fmaf(-h1, h1, 1.0f);
      gb1 += dz1;
#pragma unroll
      for (int i = 0; i < D; ++i) {
        gW1[i] = fmaf(dz1, x[i], gW1[i]);
        const float dx = warp_sum(P.w1[i] * dz1) * inv_s;
        const float hess = A.c4a_f[i] * fmaf(3.0f * x[i], x[i], -1.0f);
        lam[i] = fmaf(lam[i], fmaf(-A.dt_f, hess, 1.0f), dx);
      }
    }
  }
  float* out = partial + gw * P_;
  float* oW1 = out;
  float* ob1 = oW1 + H * D;
  float* oW2 = ob1 + H;
  float* ob2 = oW2 + H * H;
  float* oW3 = ob2 + H;
  float* ob3 = oW3 + D * H;
#pragma unroll
  for (int i = 0; i < D; ++i) { oW1[lane * D + i] = gW1[i]; oW3[i * H + lane] = gW3[i]; }
  ob1[lane] = gb1;
  ob2[lane] = gb2;
#pragma unroll
  for (int i = 0; i < H; ++i) oW2[lane * H + i] = gW2[i];
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < D; ++i) ob3[i] = gb3[i];
  }
}

// largest batch routed to the warp-per-trajectory kernels (above it one trajectory per thread fills the GPU better)
inline long long warp_path_max_k(int sm_count) { return (long long)sm_count * 16; }

// params_host == nullptr: the policy is read from W_dev (an MlpConst<D, WARP_H> in device memory, see pack_mlp_const_dev)
// RAGGED: the ragged checkpoint store (float32 state only, no Brownian-bridge test: the caller refuses both)
template <int D, bool RAGGED = false>
int launch_rollout_fwd_warp(const float* params_host, const void* W_dev, const FwdArgs& args, int sm_count, cudaStream_t stream);
template <int D, bool WEIGHTED = false, bool RAGGED = false>
int launch_rollout_bwd_warp(const float* params_host, const void* W_dev, const FwdArgs& args, float scale, float* grad,
                            float* partial, int sm_count, cudaStream_t stream);
// continues the trajectories the thread-per-trajectory kernel left in args.q_ring (args.q_ctrl[1] records)
template <int D, bool RAGGED = false>
int launch_rollout_fwd_warp_resume(const float* params_host, const FwdArgs& args, int sm_count, cudaStream_t stream);
// theta_dev (flat float32, state_dict order) -> MlpConst<D, WARP_H> in device memory, same rounding as the host packer
template <int D>
int launch_pack_mlp_const_dev(const float* theta_dev, void* W_dev, bool fast_tanh, cudaStream_t stream);
inline size_t mlp_const_bytes_max() { return sizeof(MlpConst<RLSDE_MAX_D, WARP_H>); }

}  // namespace rlsde
