// K1x / K2x: rollout kernels for WIDE policies (hidden width 64, 128, 256 -- the reference's reinforce() default is 256,
// reinforce_deterministic_core.py:102), where the hidden-hidden layer no longer fits a thread's registers or the
// constant bank and a pass becomes a small dense contraction per TILE of trajectories.
//
// Same semantics, Philox stream and outputs as K1 and the reverse pass (rollout_fwd.cuh, rollout_bwd.cuh); what changes is the mapping:
//   * a block of 128 threads advances a tile of M = 32 (or 16) trajectories in lock step; warp w owns rows
//     R w .. R w + R - 1 of the tile (R = 8 or 4), lane l owns the hidden units l, l + 32, l + 64, ...;
//   * activations of the tile live in shared memory unit-major ([unit][trajectory], rows padded to 36 floats: row
//     writes by 32 lanes, broadcast row reads and float4 column reads are all conflict-free);
//   * the H x H weights are streamed from global memory (L2-resident: 256 KB at H = 256) through a double-buffered
//     shared-memory stage of 32 input rows (cp.async) and consumed by an R x (H / 32) register tile per thread:
//     per input row one broadcast LDS.128 (R activations) + H/32 LDS.32 (weights) for R H/32 FFMA;
//   * the per-trajectory scalar work (state, hit test, accumulators, Philox increments) is done by the tile's "owner"
//     threads (thread t < M owns trajectory t) with K1's arithmetic, so given the same action the environment pass is
//     bit-identical to torch / NumPy; finished trajectories are replaced from the global work counter (lane refill).
// The policy is summed in fp32 FFMA in input order (as K1 does), so a wide policy is evaluated to the same rounding as
// the narrow ones.  Reverse pass (K2x): recomputed forward + two more tile contractions (dZ2 W2 and the outer product
// dZ2^T H1, accumulated into a block-private H x H partial in global memory), static assignment of length-sorted
// trajectories to tiles, per-block partials added in index order: deterministic gradients.  ckpt_every must be 1.
#pragma once
#include <cuda_pipeline_primitives.h>
#include "rollout_bwd.cuh"

namespace rlsde {

// Device copy of a wide policy (float32, in the caller's workspace):
//   W1t [D][H], b1 [H], W2t [H][H] (input-major), W2 [H][H] (output-major), b2 [H], W3 [D][H], b3 [D rounded up to 4]
// hidden layers pre-scaled by 2 log2(e) for the precise tanh, exactly like MlpConst.
template <int D, int H>
struct WideParams {
  static constexpr size_t o_W1t = 0;
  static constexpr size_t o_b1 = o_W1t + (size_t)D * H;
  static constexpr size_t o_W2t = o_b1 + H;
  static constexpr size_t o_W2 = o_W2t + (size_t)H * H;
  static constexpr size_t o_b2 = o_W2 + (size_t)H * H;
  static constexpr size_t o_W3 = o_b2 + H;
  static constexpr size_t o_b3 = o_W3 + (size_t)D * H;
  static constexpr size_t count = o_b3 + ((D + 3) & ~3);
};
constexpr size_t WIDE_PARAM_BYTES_MAX = (2 * 256 * 256 + 2 * RLSDE_MAX_D * 256 + 2 * 256 + RLSDE_MAX_D) * sizeof(float);

template <int D, int H>
inline void pack_wide_params(const float* p, bool fast_tanh, float* out) {
  typedef WideParams<D, H> L;
  const double s = fast_tanh ? 1.0 : RLSDE_TWO_LOG2E;
  const float* W1 = p;              // (H, D)
  const float* b1 = W1 + H * D;
  const float* W2 = b1 + H;         // (H, H)
  const float* b2 = W2 + H * H;
  const float* W3 = b2 + H;         // (D, H)
  const float* b3 = W3 + D * H;
  for (int i = 0; i < D; ++i)
    for (int j = 0; j < H; ++j) out[L::o_W1t + (size_t)i * H + j] = (float)(s * (double)W1[j * D + i]);
  for (int j = 0; j < H; ++j) out[L::o_b1 + j] = (float)(s * (double)b1[j]);
  for (int i = 0; i < H; ++i)
    for (int j = 0; j < H; ++j) {
      const float w = (float)(s * (double)W2[j * H + i]);      // W2[out = j][in = i]
      out[L::o_W2t + (size_t)i * H + j] = w;
      out[L::o_W2 + (size_t)j * H + i] = w;
    }
  for (int j = 0; j < H; ++j) out[L::o_b2 + j] = (float)(s * (double)b2[j]);
  for (int k = 0; k < D; ++k)
    for (int j = 0; j < H; ++j) out[L::o_W3 + (size_t)k * H + j] = W3[k * H + j];
  for (int k = 0; k < ((D + 3) & ~3); ++k) out[L::o_b3 + k] = k < D ? b3[k] : 0.0f;
}

constexpr int WIDE_THREADS = 128;
constexpr int WIDE_KC = 32;                 // input rows per weight stage
constexpr int WIDE_LD = 36;                 // row pitch of the [unit][trajectory] activation tiles (floats)

template <int H>
__host__ __device__ constexpr size_t wide_fwd_smem_bytes() {
  // activations h1 [H][LD] + two weight stages [KC][H] + x / u exchange [32][RLSDE_MAX_D] x 2
  return ((size_t)H * WIDE_LD + 2 * (size_t)WIDE_KC * H + 2 * 32 * RLSDE_MAX_D) * sizeof(float);
}
template <int H>
__host__ __device__ constexpr size_t wide_bwd_smem_bytes() {
  // h1 and dz2 tiles + two weight stages + x / u / a / dx exchange
  return (2 * (size_t)H * WIDE_LD + 2 * (size_t)WIDE_KC * H + 4 * 32 * RLSDE_MAX_D) * sizeof(float);
}

// one stage of WIDE_KC rows x H floats, global -> shared, 16 bytes per cp.async, whole block
template <int H>
__device__ __forceinline__ void wide_stage_load(float* dst, const float* __restrict__ src) {
  constexpr int N16 = WIDE_KC * H / 4;
  for (int i = threadIdx.x; i < N16; i += WIDE_THREADS)
    __pipeline_memcpy_async(reinterpret_cast<float4*>(dst) + i, reinterpret_cast<const float4*>(src) + i, 16);
  __pipeline_commit();
}

// acc[r][c] += sum_i A[i][row0 + r] * Wg[i][lane + 32 c]   for i in [0, H): A = activation tile in shared memory
// ([unit][trajectory], pitch WIDE_LD), Wg = H x H weights in global memory with the contraction index leading.
// Weights go through the two shared-memory stages; all threads of the block must call this together.
template <int H, int R>
__device__ __forceinline__ void wide_tile_gemm(float (&acc)[R][H / 32], const float* __restrict__ A, const float* __restrict__ Wg,
                                               float* stage, int row0, int lane) {
  constexpr int CPL = H / 32;
  constexpr int NCH = H / WIDE_KC;
  wide_stage_load<H>(stage, Wg);
  for (int ch = 0; ch < NCH; ++ch) {
    float* cur = stage + (size_t)(ch & 1) * WIDE_KC * H;
    if (ch + 1 < NCH) {
      wide_stage_load<H>(stage + (size_t)((ch + 1) & 1) * WIDE_KC * H, Wg + (size_t)(ch + 1) * WIDE_KC * H);
      __pipeline_wait_prior(1);
    } else {
      __pipeline_wait_prior(0);
    }
    __syncthreads();
#pragma unroll 4
    for (int ii = 0; ii < WIDE_KC; ++ii) {
      const float* arow = A + (size_t)(ch * WIDE_KC + ii) * WIDE_LD + row0;
      float a[R];
#pragma unroll
      for (int r4 = 0; r4 < R / 4; ++r4) {
        const float4 t = *reinterpret_cast<const float4*>(arow + 4 * r4);
        a[4 * r4] = t.x; a[4 * r4 + 1] = t.y; a[4 * r4 + 2] = t.z; a[4 * r4 + 3] = t.w;
      }
      const float* wrow = cur + (size_t)ii * H + lane;
#pragma unroll
      for (int c = 0; c < CPL; ++c) {
        const float w = wrow[32 * c];
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r][c] = fmaf(a[r], w, acc[r][c]);
      }
    }
    __syncthreads();                 // the stage just consumed is the target of the load issued next round
  }
}

template <bool FAST>
__device__ __forceinline__ float wide_tanh(float zp) {      // zp pre-scaled by 2 log2(e) unless FAST
  if constexpr (FAST) return mufu_tanh(zp);
  return fmaf(-2.0f, mufu_rcp(mufu_ex2(zp) + 1.0f), 1.0f);
}

// h1 tile: h1[unit][traj] = tanh(b1 + W1 x) for the warp's R rows and the lane's H / 32 units, written unit-major
template <int D, int H, int R, bool FAST>
__device__ __forceinline__ void wide_layer1(const float* __restrict__ Wp, const float* xS, float* h1S, int row0, int lane) {
  typedef WideParams<D, H> L;
  float xr[R][D];
#pragma unroll
  for (int r = 0; r < R; ++r)
#pragma unroll
    for (int k = 0; k < D; ++k) xr[r][k] = xS[(row0 + r) * RLSDE_MAX_D + k];
#pragma unroll
  for (int c = 0; c < H / 32; ++c) {
    const int unit = lane + 32 * c;
    const float b = __ldg(Wp + L::o_b1 + unit);
    float w[D];
#pragma unroll
    for (int k = 0; k < D; ++k) w[k] = __ldg(Wp + L::o_W1t + (size_t)k * H + unit);
    float hv[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      float z = b;
#pragma unroll
      for (int k = 0; k < D; ++k) z = fmaf(xr[r][k], w[k], z);
      hv[r] = wide_tanh<FAST>(z);
    }
#pragma unroll
    for (int r4 = 0; r4 < R / 4; ++r4)
      *reinterpret_cast<float4*>(h1S + (size_t)unit * WIDE_LD + row0 + 4 * r4) = make_float4(hv[4 * r4], hv[4 * r4 + 1], hv[4 * r4 + 2], hv[4 * r4 + 3]);
  }
}

// head: u[row][k] = b3[k] + sum_unit W3[k][unit] h2[row][unit]; the warp holds all units of its rows -> butterfly sums,
// lane 0 writes uS[row][k]
template <int D, int H, int R>
__device__ __forceinline__ void wide_head(const float* __restrict__ Wp, const float (&h2)[R][H / 32], float* uS, int row0, int lane) {
  typedef WideParams<D, H> L;
#pragma unroll
  for (int k = 0; k < D; ++k) {
    float w3[H / 32];
#pragma unroll
    for (int c = 0; c < H / 32; ++c) w3[c] = __ldg(Wp + L::o_W3 + (size_t)k * H + lane + 32 * c);
#pragma unroll
    for (int r = 0; r < R; ++r) {
      float v = 0.f;
#pragma unroll
      for (int c = 0; c < H / 32; ++c) v = fmaf(w3[c], h2[r][c], v);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) uS[(row0 + r) * RLSDE_MAX_D + k] = v + __ldg(Wp + L::o_b3 + k);
    }
  }
}

// ------------------------------------------------------------------------------------------------ forward
// BRIDGE: the Brownian-bridge hit test between passes (bridge_project, rollout_fwd.cuh; d = 1 only)
template <int D, int H, int R, bool F64, bool FAST, bool BRIDGE = false, bool RAGGED = false>
__global__ void __launch_bounds__(WIDE_THREADS, 1) rollout_fwd_wide_kernel(const float* __restrict__ Wp, const __grid_constant__ FwdArgs A) {
  typedef typename RealT<F64>::type real;
  typedef WideParams<D, H> L;
  constexpr int M = 4 * R;                  // trajectories per tile (4 warps x R rows)
  constexpr int SPB = NoisePlan<D>::SPB;
  constexpr int BPP = NoisePlan<D>::BPP;
  constexpr int NZ = NoisePlan<D>::NZ;
  extern __shared__ __align__(16) float smem[];
  float* h1S = smem;
  float* stage = h1S + (size_t)H * WIDE_LD;
  float* xS = stage + 2 * (size_t)WIDE_KC * H;
  float* uS = xS + 32 * RLSDE_MAX_D;
  __shared__ int s_live;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int row0 = warp * R;
  const bool owner = threadIdx.x < M;
  const bool inject = (A.flags & RLSDE_F_NOISE_INJECTED) != 0;
  const bool s_exact = (A.flags & RLSDE_F_STOCH_INT_EXACT) != 0;
  const bool store_path = (A.flags & RLSDE_F_STORE_PATH) != 0 && A.path != nullptr;
  const bool want_l2 = (D == 1) && A.policy_opt != nullptr && A.l2 != nullptr;
  const long long lim = inject ? (A.noise_steps < A.n_steps_lim ? A.noise_steps : A.n_steps_lim) : A.n_steps_lim;
  const double inv_s2dt = BRIDGE ? bridge_inv_s2dt(A) : 0.0;

  // owner state
  bool alive = false, exhausted = false;
  long long traj = 0;
  int k = 0, ck = 0;
  real x[D];
  real G = 0, S = 0, L2 = 0;
  float z[NZ];
#pragma unroll
  for (int i = 0; i < D; ++i) x[i] = F64 ? (real)A.x0_d[i] : (real)A.x0_f[i];
#pragma unroll
  for (int i = 0; i < NZ; ++i) z[i] = 0.f;

  for (;;) {
    // ---- owners: take the next trajectory if idle (warp 0 holds all owners: M <= 32)
    if (warp == 0) {
      const unsigned need = __ballot_sync(0xffffffffu, owner && !alive && !exhausted);
      if (need) {
        unsigned long long base = 0;
        const int leader = __ffs(need) - 1;
        if (lane == leader) base = atomicAdd(A.counter, (unsigned long long)__popc(need));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (owner && !alive && !exhausted) {
          const long long idx = (long long)base + __popc(need & ((1u << lane) - 1u));
          if (idx < A.K) {
            traj = idx; k = 0; ck = 0; alive = true; G = 0; S = 0; L2 = 0;
#pragma unroll
            for (int i = 0; i < D; ++i) x[i] = F64 ? (real)A.x0_d[i] : (real)A.x0_f[i];
          } else {
            exhausted = true;
          }
        }
      }
      const unsigned live = __ballot_sync(0xffffffffu, alive);
      if (lane == 0) s_live = live != 0u;
      if (owner) {
#pragma unroll
        for (int i = 0; i < D; ++i) xS[lane * RLSDE_MAX_D + i] = (float)x[i];
      }
    }
    __syncthreads();
    if (!s_live) break;

    // ---- policy for the whole tile
    wide_layer1<D, H, R, FAST>(Wp, xS, h1S, row0, lane);
    __syncthreads();
    float acc[R][H / 32];
#pragma unroll
    for (int c = 0; c < H / 32; ++c) {
      const float b = __ldg(Wp + L::o_b2 + lane + 32 * c);
#pragma unroll
      for (int r = 0; r < R; ++r) acc[r][c] = b;
    }
    wide_tile_gemm<H, R>(acc, h1S, Wp + L::o_W2t, stage, row0, lane);
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int c = 0; c < H / 32; ++c) acc[r][c] = wide_tanh<FAST>(acc[r][c]);
    wide_head<D, H, R>(Wp, acc, uS, row0, lane);
    __syncthreads();

    // ---- owners: one environment pass, K1's arithmetic (rollout_fwd.cuh)
    if (owner && alive) {
      float u[D], dB[D];
#pragma unroll
      for (int i = 0; i < D; ++i) u[i] = uS[lane * RLSDE_MAX_D + i];
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
        const real Sout = s_exact ? S_prev : S;
        if (F64) {
          ((double*)A.G)[traj] = (double)G; ((double*)A.S)[traj] = (double)Sout;
          if (A.l2) ((double*)A.l2)[traj] = (double)L2;
          if (A.logw) ((double*)A.logw)[traj] = (double)G - (double)S_prev;
        } else {
          ((float*)A.G)[traj] = (float)G; ((float*)A.S)[traj] = (float)Sout;
          if (A.l2) ((float*)A.l2)[traj] = (float)L2;
          if (A.logw) ((float*)A.logw)[traj] = (float)G - (float)S_prev;
        }
        A.T[traj] = k;
        alive = false;
      } else {
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
          if (F64) {
            ((double*)A.G)[traj] = (double)G; ((double*)A.S)[traj] = (double)S;
            if (A.l2) ((double*)A.l2)[traj] = (double)L2;
            if (A.logw) ((double*)A.logw)[traj] = (double)G - (double)S;
          } else {
            ((float*)A.G)[traj] = (float)G; ((float*)A.S)[traj] = (float)S;
            if (A.l2) ((float*)A.l2)[traj] = (float)L2;
            if (A.logw) ((float*)A.logw)[traj] = (float)G - (float)S;
          }
          A.T[traj] = -1;
          alive = false;
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ reverse
// Block-private partial gradient in global memory: state_dict order, float32 [P].  The H x H block is updated in place
// every pass (read-modify-write by the thread that owns the element); the small blocks are kept in registers / shared
// memory and written at the end.
// WEIGHTED: per-trajectory coefficients (rollout_bwd.cuh, the comment above em_step_f32)
// RAGGED: the states come from the ragged store (ckpt_slot, rollout_fwd.cuh)
template <int D, int H, int R, bool FAST, bool WEIGHTED = false, bool RAGGED = false>
__global__ void __launch_bounds__(WIDE_THREADS, 1) rollout_bwd_wide_kernel(const float* __restrict__ Wp, const __grid_constant__ FwdArgs A,
                                                                           float* __restrict__ partial) {
  typedef WideParams<D, H> L;
  constexpr int M = 4 * R;
  constexpr int CPL = H / 32;
  constexpr int P = D * H + H + H * H + H + H * D + D;
  extern __shared__ __align__(16) float smem[];
  float* h1S = smem;                                   // [H][LD]
  float* dzS = h1S + (size_t)H * WIDE_LD;              // [H][LD]  dz2 of the tile
  float* stage = dzS + (size_t)H * WIDE_LD;
  float* xS = stage + 2 * (size_t)WIDE_KC * H;
  float* uS = xS + 32 * RLSDE_MAX_D;
  float* aS = uS + 32 * RLSDE_MAX_D;
  float* dxS = aS + 32 * RLSDE_MAX_D;
  __shared__ int s_live;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int row0 = warp * R;
  const bool owner = threadIdx.x < M;
  const bool inject = (A.flags & RLSDE_F_NOISE_INJECTED) != 0;
  const bool s_exact = (A.flags & RLSDE_F_STOCH_INT_EXACT) != 0;
  const float inv_s = FAST ? 1.0f : (float)(1.0 / RLSDE_TWO_LOG2E);
  float* const out = partial + (size_t)blockIdx.x * P;
  float* const oW1 = out;
  float* const ob1 = oW1 + H * D;
  float* const oW2 = ob1 + H;
  float* const ob2 = oW2 + H * H;
  float* const oW3 = ob2 + H;
  float* const ob3 = oW3 + D * H;
  for (int i = threadIdx.x; i < P; i += WIDE_THREADS) out[i] = 0.f;

  // per-thread partials of the small blocks: the lane's units, summed over the warp's rows (and over passes)
  float gb1[CPL], gb2[CPL], gW1[CPL][D], gW3[CPL][D], gb3[D];
#pragma unroll
  for (int c = 0; c < CPL; ++c) {
    gb1[c] = 0.f; gb2[c] = 0.f;
#pragma unroll
    for (int i = 0; i < D; ++i) { gW1[c][i] = 0.f; gW3[c][i] = 0.f; }
  }
#pragma unroll
  for (int i = 0; i < D; ++i) gb3[i] = 0.f;

  // owner state: static assignment, tile by tile over the (length-sorted) order => deterministic
  bool alive = false;
  long long traj = 0;
  int kstar = 0, j = 0;
  float Gk = 0.f, mG = 0.f;        // WEIGHTED: -cS, -cG
  float lam[D];
  NoiseCache<D> nc;
  nc.reset();
#pragma unroll
  for (int i = 0; i < D; ++i) lam[i] = 0.f;
  long long tile = (long long)blockIdx.x - gridDim.x;
  __syncthreads();

  for (;;) {
    if (warp == 0) {
      unsigned live = __ballot_sync(0xffffffffu, alive);
      while (!live) {                                 // the whole tile is done: take the next one
        tile += gridDim.x;
        if (tile * M >= A.K) break;
        const long long slot = tile * M + lane;
        if (owner && slot < A.K) {
          traj = A.order ? A.order[slot] : slot;
          const int t = A.T[traj];
          if (t >= 0 && ckpt_covered<RAGGED>(A, traj, t)) {
            alive = true; kstar = t; j = t; Gk = ((const float*)A.G)[traj];
            if constexpr (WEIGHTED) { Gk = __fmul_rn(-1.0f, Gk); mG = __fmul_rn(-1.0f, ((const float*)A.S)[traj]); }
            nc.reset();
#pragma unroll
            for (int i = 0; i < D; ++i) lam[i] = 0.f;
          }
        }
        live = __ballot_sync(0xffffffffu, alive);
      }
      if (lane == 0) s_live = live != 0u;
      if (owner) {
#pragma unroll
        for (int i = 0; i < D; ++i) xS[lane * RLSDE_MAX_D + i] = alive ? A.path[ckpt_slot<RAGGED>(A, traj, j) * D + i] : A.x0_f[i];
      }
    }
    __syncthreads();
    if (!s_live) break;

    // ---- recomputed forward of the tile
    wide_layer1<D, H, R, FAST>(Wp, xS, h1S, row0, lane);
    __syncthreads();
    float acc[R][CPL];
#pragma unroll
    for (int c = 0; c < CPL; ++c) {
      const float b = __ldg(Wp + L::o_b2 + lane + 32 * c);
#pragma unroll
      for (int r = 0; r < R; ++r) acc[r][c] = b;
    }
    wide_tile_gemm<H, R>(acc, h1S, Wp + L::o_W2t, stage, row0, lane);
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int c = 0; c < CPL; ++c) acc[r][c] = wide_tanh<FAST>(acc[r][c]);        // h2
    wide_head<D, H, R>(Wp, acc, uS, row0, lane);
    __syncthreads();

    // ---- owners: a_j
    if (warp == 0 && owner) {
      float dB[D];
      nc.get(A, inject, alive, traj, j, dB);
#pragma unroll
      for (int i = 0; i < D; ++i) {
        float v = 0.f;
        if (alive) {
          const bool incl = s_exact ? (j < kstar) : true;
          if constexpr (WEIGHTED)
            v = (j < kstar ? __fmul_rn(mG, uS[lane * RLSDE_MAX_D + i]) * A.dt_f : 0.f) - (incl ? Gk * dB[i] : 0.f) + A.sigma_f * A.dt_f * lam[i];
          else v = (j < kstar ? uS[lane * RLSDE_MAX_D + i] * A.dt_f : 0.f) - (incl ? Gk * dB[i] : 0.f) + A.sigma_f * A.dt_f * lam[i];
        }
        aS[lane * RLSDE_MAX_D + i] = v;
        gb3[i] += v;
      }
    }
    __syncthreads();

    // ---- dz2 = (W3^T a)(1 - h2^2); dW3 += a (x) h2; db2 += dz2; dz2 tile to shared memory (unit-major)
    {
      float ar[R][D];
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int i = 0; i < D; ++i) ar[r][i] = aS[(row0 + r) * RLSDE_MAX_D + i];
#pragma unroll
      for (int c = 0; c < CPL; ++c) {
        const int unit = lane + 32 * c;
        float w3[D];
#pragma unroll
        for (int i = 0; i < D; ++i) w3[i] = __ldg(Wp + L::o_W3 + (size_t)i * H + unit);
        float dz[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const float hv = acc[r][c];
          float dh = 0.f;
#pragma unroll
          for (int i = 0; i < D; ++i) {
            dh = fmaf(ar[r][i], w3[i], dh);
            gW3[c][i] = fmaf(ar[r][i], hv, gW3[c][i]);
          }
          dz[r] = dh * fmaf(-hv, hv, 1.0f);
          gb2[c] += dz[r];
        }
#pragma unroll
        for (int r4 = 0; r4 < R / 4; ++r4)
          *reinterpret_cast<float4*>(dzS + (size_t)unit * WIDE_LD + row0 + 4 * r4) = make_float4(dz[4 * r4], dz[4 * r4 + 1], dz[4 * r4 + 2], dz[4 * r4 + 3]);
      }
    }
    __syncthreads();

    // ---- dh1 = dz2 W2 (contraction over the output units: W2 output-major) -> dz1 = dh1 (1 - h1^2) / s
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int c = 0; c < CPL; ++c) acc[r][c] = 0.f;
    wide_tile_gemm<H, R>(acc, dzS, Wp + L::o_W2, stage, row0, lane);
    {
      float dxp[R][D];
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int i = 0; i < D; ++i) dxp[r][i] = 0.f;
#pragma unroll
      for (int c = 0; c < CPL; ++c) {
        const int unit = lane + 32 * c;
        float w1[D];
#pragma unroll
        for (int i = 0; i < D; ++i) w1[i] = __ldg(Wp + L::o_W1t + (size_t)i * H + unit);
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const float hv = h1S[(size_t)unit * WIDE_LD + row0 + r];
          const float dz = acc[r][c] * inv_s * fmaf(-hv, hv, 1.0f);
          gb1[c] += dz;
#pragma unroll
          for (int i = 0; i < D; ++i) {
            gW1[c][i] = fmaf(dz, xS[(row0 + r) * RLSDE_MAX_D + i], gW1[c][i]);
            dxp[r][i] = fmaf(w1[i], dz, dxp[r][i]);
          }
        }
      }
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int i = 0; i < D; ++i) {
          float v = dxp[r][i];
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
          if (lane == 0) dxS[(row0 + r) * RLSDE_MAX_D + i] = v * inv_s;
        }
    }

    // ---- dW2[u][i] += sum_t dz2[t][u] h1[t][i]: both tiles are trajectory-contiguous.  Warp w takes the output-unit
    // groups u0 = 8 (w + 4 n); lane l the input units l + 32 c.  The running sum is the block-private partial in global
    // memory (L2-resident), read-modify-written by the one thread that owns the element.
    for (int ug = warp; ug < H / 8; ug += 4) {
      const int u0 = 8 * ug;
      float w2[8][CPL];
#pragma unroll
      for (int a8 = 0; a8 < 8; ++a8)
#pragma unroll
        for (int c = 0; c < CPL; ++c) w2[a8][c] = 0.f;
#pragma unroll
      for (int t4 = 0; t4 < M / 4; ++t4) {
        float4 dzv[8];
#pragma unroll
        for (int a8 = 0; a8 < 8; ++a8) dzv[a8] = *reinterpret_cast<const float4*>(dzS + (size_t)(u0 + a8) * WIDE_LD + 4 * t4);
#pragma unroll
        for (int c = 0; c < CPL; ++c) {
          const float4 hv = *reinterpret_cast<const float4*>(h1S + (size_t)(lane + 32 * c) * WIDE_LD + 4 * t4);
#pragma unroll
          for (int a8 = 0; a8 < 8; ++a8) {
            w2[a8][c] = fmaf(dzv[a8].x, hv.x, w2[a8][c]);
            w2[a8][c] = fmaf(dzv[a8].y, hv.y, w2[a8][c]);
            w2[a8][c] = fmaf(dzv[a8].z, hv.z, w2[a8][c]);
            w2[a8][c] = fmaf(dzv[a8].w, hv.w, w2[a8][c]);
          }
        }
      }
#pragma unroll
      for (int a8 = 0; a8 < 8; ++a8)
#pragma unroll
        for (int c = 0; c < CPL; ++c) {
          float* dst = oW2 + (size_t)(u0 + a8) * H + lane + 32 * c;
          *dst = *dst + w2[a8][c];
        }
    }
    __syncthreads();

    // ---- owners: adjoint state and next pass
    if (warp == 0 && owner && alive) {
      const float* xp = xS + lane * RLSDE_MAX_D;
#pragma unroll
      for (int i = 0; i < D; ++i) {
        const float hess = A.c4a_f[i] * fmaf(3.0f * xp[i], xp[i], -1.0f);
        lam[i] = fmaf(lam[i], fmaf(-A.dt_f, hess, 1.0f), dxS[lane * RLSDE_MAX_D + i]);
      }
      --j;
      if (j < 0) alive = false;
    }
    __syncthreads();
  }

  // ---- small blocks: sum the four warps' register partials through shared memory (fixed order), then to the partial
  __syncthreads();
  float* red = smem;                                    // [4 warps][(2 + 2 D) H]
#pragma unroll
  for (int c = 0; c < CPL; ++c) {
    const int unit = lane + 32 * c;
    float* base = red + (size_t)warp * (2 + 2 * D) * H;
    base[unit] = gb1[c];
    base[H + unit] = gb2[c];
#pragma unroll
    for (int i = 0; i < D; ++i) { base[(2 + i) * H + unit] = gW1[c][i]; base[(2 + D + i) * H + unit] = gW3[c][i]; }
  }
  if (warp == 0) {
#pragma unroll
    for (int i = 0; i < D; ++i) {
      float v = gb3[i];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) ob3[i] = v;
    }
  }
  __syncthreads();
  for (int e = threadIdx.x; e < (2 + 2 * D) * H; e += WIDE_THREADS) {
    const float v = ((red[e] + red[(size_t)(2 + 2 * D) * H + e]) + red[(size_t)2 * (2 + 2 * D) * H + e]) + red[(size_t)3 * (2 + 2 * D) * H + e];
    const int blk = e / H, unit = e % H;
    if (blk == 0) ob1[unit] = v;
    else if (blk == 1) ob2[unit] = v;
    else if (blk < 2 + D) oW1[unit * D + (blk - 2)] = v;
    else oW3[(blk - 2 - D) * H + unit] = v;
  }
}

// grad[p] (+)= scale * sum_b partial[b][p], blocks in index order
static __global__ void wide_reduce_kernel(const float* __restrict__ partial, int n_blocks, int P, float scale, float* __restrict__ grad,
                                          int accumulate) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  double acc = 0.0;
  for (int b = 0; b < n_blocks; ++b) acc += (double)partial[(size_t)b * P + p];
  const float g = (float)(acc * (double)scale);
  grad[p] = accumulate ? grad[p] + g : g;
}

// params_dev: WideParams<D, H> buffer in the caller's workspace (filled from params_host by the launcher).
// RAGGED: the ragged checkpoint store (float32 state only, no Brownian-bridge test: the caller refuses both)
template <int D, int H, bool RAGGED = false>
int launch_rollout_fwd_wide(const float* params_host, float* params_dev, const FwdArgs& args, int sm_count, cudaStream_t stream);
template <int D, int H, bool WEIGHTED = false, bool RAGGED = false>
int launch_rollout_bwd_wide(const float* params_host, float* params_dev, const FwdArgs& args, float scale, float* grad, float* partial,
                            size_t partial_bytes, int sm_count, cudaStream_t stream);

}  // namespace rlsde
