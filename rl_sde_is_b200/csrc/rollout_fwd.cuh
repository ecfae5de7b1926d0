// K1: fused forward rollout (policy MLP + Euler-Maruyama pass + hit bookkeeping + running
// work / stochastic-integral accumulation), one trajectory per thread, state in registers for
// the whole rollout, lane refill from a global work counter.
//
// Replaces the per-pass Python loops of sample_loss_vectorized (reinforce_deterministic_core.py:52-88),
// test_policy_vectorized (approximate_methods.py:597-638) and estimate_fht_vectorized (:667-688),
// i.e. one model.forward + env.step[_torch] (environments.py:139-162,201-226) per pass.
//
// Per-pass semantics (SURVEY.md Appendix A):
//   u = policy(X_k);  hit = X_k in target set (CURRENT state);  S += u . dB_{k+1} (also on the hit pass);
//   hit  -> record (G, S, k) and retire;   else G += -(1 + |u|^2/2) dt;  X_{k+1} = X_k + (-gradV + sigma u) dt + sigma dB.
// Arithmetic of the pass is written with the reference's association and without FMA contraction
// so that, given the same action and increment, next state / reward are bit-identical to torch's
// (f32) or numpy's (f64, RLSDE_F_STATE_F64) results.
//
// Scheduling: a warp's 32 lanes run 32 independent trajectories in lock step.  A lane whose
// trajectory retires takes the next work item (warp-aggregated atomicAdd) at the next noise-block
// boundary, so lanes stay busy until the work runs out.
//
// Time slicing.  Trajectory lengths are unknown in advance and bounded only by n_steps_lim, so with
// run-to-completion scheduling the launch ends with a tail of (longest trajectory) x (time of a pass): the
// last-started long trajectory runs on an otherwise empty GPU (measured: 4.3 ms of a 27.5 ms launch at
// 1e6 trajectories, whatever the batch size).  Instead a trajectory runs for at most `q_quantum` passes
// per slice; a lane whose slice is over appends the trajectory's state (24 B at d = 1) to a FIFO in
// global memory and takes the next item.  Items are served in order -- first all fresh trajectories,
// then their continuations in the order they were queued -- which makes the schedule breadth-first: all
// trajectories advance together and the tail shrinks to a few quanta.  (Warps do not advance at the same pace -- with
// eight warps per scheduler some execute 8 000 passes while others execute 700 in the same launch -- so the last
// slice of a trajectory that sits in a starved warp is what ends the launch: short slices, 8 passes at n_steps_lim =
// 1000, measured best; they cost ~3 % in steady state.)  The FIFO is a ring of records with
// a sequence word per slot (producer: write, fence, publish epoch; consumer: claim an index, poll its
// slot between passes, never blocking the warp's other lanes); the launch ends when every trajectory has
// reported completion.  Per-trajectory arithmetic does not depend on the slicing: results are bit-identical.
#pragma once
#include <type_traits>
#include "common.cuh"
#include "mlp_mma.cuh"
#include "../../include/rlsde.h"

namespace rlsde {

template <bool F64> struct RealT { typedef float type; };
template <> struct RealT<true> { typedef double type; };

struct FwdArgs {
  // environment (both precisions are precomputed on the host the way torch / numpy round them)
  float c4a_f[RLSDE_MAX_D];     // float32(4 * alpha_i)
  double c4a_d[RLSDE_MAX_D];    // 4 * alpha_i
  float x0_f[RLSDE_MAX_D];
  double x0_d[RLSDE_MAX_D];
  float sigma_f, dt_f, lb_f, rb_f;
  double sigma_d, dt_d, lb_d, rb_d;
  float noise_scale2;           // -2 dt ln 2
  int hit_rule;
  // work
  long long K, traj_offset, K_global;
  unsigned long long seed;
  long long n_steps_lim, noise_steps;
  unsigned flags;
  int ckpt_every;
  int ckpt_log2;                 // log2(ckpt_every) if it is a power of two (checkpoint index = k >> ckpt_log2), else -1
  long long ckpt_stride;
  long long n_grid;
  double grid_lo, grid_hi, grid_h;
  // buffers
  const float* noise;
  const float* policy_opt;
  void* G;
  void* S;
  int* T;
  void* l2;
  void* logw;
  float* path;
  unsigned long long* counter;   // work counter of THIS launch (zeroed by the host wrapper)
  const long long* order;        // reverse pass: processing order of the trajectories (or nullptr = identity)
  int grad_accumulate;           // reverse pass: add this launch's gradient to grad instead of overwriting it
  int blocks_per_sm_cap;         // > 0: cap on resident blocks per SM of the thread-per-trajectory forward kernel (tuning)
  int policy_mma;                // 1: the thread-per-trajectory forward kernel evaluates the policy with mlp_forward_mma (and
                                 // the kernel that continues its handed-over trajectories does the same), 0: with FFMA2
  float mma_x1_max;              // set by the launcher: mlp_forward_mma skips the layer-1 clamp of a warp whose states all
                                 // have max_i |x_i| <= this (fwd_mma_clamp_bounds)
  // ---- transition stream (replay-buffer sampler, approximate_methods.py:513-545): trajectory `t` writes the tuple of
  //      its pass k at slot tr_base[t] + k of the five arrays below.  nullptr = no stream.
  //      path_base (kernels instantiated with RAGGED only, which never carry the stream): the ragged checkpoint store,
  //      trajectory t owns rows [path_base[t], path_base[t + 1]) of `path` (ckpt_slot).  One field for both keeps the
  //      struct, and so the code of every kernel compiled without RAGGED, unchanged.
  union {
    const long long* tr_base;
    const long long* path_base;
  };
  float* tr_state;               // [n][d]  state the pass starts from
  float* tr_action;              // [n][d]
  float* tr_reward;              // [n]
  float* tr_next;                // [n][d]  state after the pass (also computed on the pass that detects the hit)
  unsigned char* tr_done;        // [n]
  // ---- time-sliced scheduling (see the header comment).  q_ring == nullptr: every trajectory runs to completion.
  unsigned char* q_ring;               // ring of ContRec<D, F64> records, all-zero at launch
  long long q_cap;                     // records in the ring: a power of two >= K + lanes of the grid
  int q_cap_log2;
  unsigned long long* q_ctrl;          // [0] items claimed (== counter), [1] continuation records queued, [2] trajectories
                                       // completed, [3] records taken by the resume kernel, [4] trajectories that ran into
                                       // the pass budget, [5] tail strategy of an adaptive launch
  int q_quantum;                       // passes per slice (0: run to completion)
  int q_adaptive;                      // 1: start run-to-completion and pick the tail strategy from what the launch sees:
                                       //    q_ctrl[5] = 1 (time slices) once >= 5 % of the completed trajectories ran into the
                                       //    pass budget, = 2 (hand-off) if the work runs out first
  long long q_handoff;                 // > 0 (run-to-completion only): once all trajectories have been started and at most
                                       // this many are still live, they are left in the ring for the warp-per-trajectory
                                       // kernel, which advances a lone trajectory ~5x faster (rollout_warp.cuh, RESUME)
};

// State of an in-flight trajectory: everything a lane needs to continue it (x, accumulators, pass index).
template <int D, bool F64>
struct alignas(8) ContRec {
  long long traj;
  int k;
  int seq;            // 0: never used; e > 0: holds the e-th record of this slot; -e: that record has been taken
  typename RealT<F64>::type x[D];
  typename RealT<F64>::type G, S, L2;
};

// Row of `path` that holds checkpoint ci (the state X_{ci * ckpt_every}) of trajectory traj: the dense store
// path[K][ckpt_stride][d], or (RAGGED, rlsde_rollout_fwd_ragged / rlsde_rollout_bwd_ragged) the ragged one, in which the
// trajectory owns rows [path_base[traj], path_base[traj + 1]).  A ragged writer drops a checkpoint that falls outside
// them (ckpt_writable); a ragged reverse pass takes a trajectory only if they hold all its checkpoints (ckpt_covered).
template <bool RAGGED>
__device__ __forceinline__ long long ckpt_slot(const FwdArgs& A, long long traj, int ci) {
  if constexpr (RAGGED) return A.path_base[traj] + ci;
  else return traj * A.ckpt_stride + ci;
}
template <bool RAGGED>
__device__ __forceinline__ bool ckpt_writable(const FwdArgs& A, long long traj, long long slot) {
  if constexpr (RAGGED) return slot < A.path_base[traj + 1];
  else return true;
}
template <bool RAGGED>
__device__ __forceinline__ bool ckpt_covered(const FwdArgs& A, long long traj, int kstar) {
  if constexpr (RAGGED) return A.path_base[traj] + kstar / A.ckpt_every < A.path_base[traj + 1];
  else return true;
}

__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }

// ---- Brownian-bridge hit test between passes (RLSDE_F_HIT_BRIDGE, d = 1).  Every rollout kernel that carries out a pass
// (K1 below, the warp / wide kernels and TrajOwner::pass) calls bridge_project after the Euler-Maruyama update of a pass
// whose state a = X_k was not a hit, with b = X_{k+1}.  Within the pass the drift is frozen, so conditioned on its end
// points the path is a Brownian bridge whatever the drift, and it reaches a barrier c that both end points lie beyond with
// probability p = exp(-2 (c - a)(c - b) / (sigma^2 dt)).  Endpoints on opposite sides of [lb, rb] (rb = +inf under
// RLSDE_HIT_ALL_GE_LB) crossed for certain; b inside the target is left to the next pass's hit test.  A crossing moves
// X_{k+1} onto the barrier on a's side, where the next pass's ordinary hit test detects it, so no new per-trajectory state
// exists and continuation records carry it unchanged.  U is drawn from its own Philox stream, counter (traj_lo, traj_hi,
// pass k, "BRDG"), key seed: the Brownian increments are untouched.  A crossing needs U < p and U >= 2^-33, so p is only
// evaluated (exp) and U only drawn where the exponent is at most 23 > 33 ln 2: whether a draw happens changes no result.
// p is evaluated in double from the state values in either state precision; the comparisons with lb / rb are the hit
// test's own (state precision), so an unprojected b outside the target is never detected by the next pass.
#define RLSDE_BRIDGE_TAG 0x42524447u /* "BRDG" */
constexpr double RLSDE_BRIDGE_ARG_MAX = 23.0;
// 1 / (sigma^2 dt), correctly rounded: equal to the host's 1.0 / (sigma * sigma * dt) in double
__device__ __forceinline__ double bridge_inv_s2dt(const FwdArgs& A) { return __drcp_rn(__dmul_rn(__dmul_rn(A.sigma_d, A.sigma_d), A.dt_d)); }
template <typename real>
__device__ __forceinline__ void bridge_project(const FwdArgs& A, double inv_s2dt, unsigned long long gt, int k, real a, real& b) {
  constexpr bool F64 = sizeof(real) == 8;
  const bool two = A.hit_rule == RLSDE_HIT_X0_IN_LB_RB;
  const real lb = F64 ? (real)A.lb_d : (real)A.lb_f, rb = F64 ? (real)A.rb_d : (real)A.rb_f;
  const bool a_lo = a < lb, b_lo = b < lb, b_hi = two && b > rb;
  if (!b_lo && !b_hi) return;
  bool cross = a_lo != b_lo;
  if (!cross) {
    const double c = a_lo ? A.lb_d : A.rb_d;
    const double arg = __dmul_rn(__dmul_rn(__dmul_rn(2.0, __dsub_rn(c, (double)a)), __dsub_rn(c, (double)b)), inv_s2dt);
    if (arg <= RLSDE_BRIDGE_ARG_MAX) {
      const Philox4 r = philox4x32_10((uint32_t)gt, (uint32_t)(gt >> 32), (uint32_t)k, RLSDE_BRIDGE_TAG, (uint32_t)A.seed,
                                      (uint32_t)(A.seed >> 32));
      cross = __dmul_rn(__dadd_rn((double)r.x, 0.5), 2.3283064365386963e-10) < exp(-arg);
    }
  }
  if (cross) b = a_lo ? lb : rb;
}

// Cold path of the FIFO: a producer found its slot still holding an unread record (the ring is larger than the number of
// records in flight, so this needs a reader stalled for a whole lap).  Kept out of line: inlined, the spin loop costs the
// rollout kernel ~15 registers.
static __device__ __noinline__ void wait_for_slot(volatile int* seq, int free_mark) {
  while (*seq != free_mark) __nanosleep(64);
}

// A warp without a live lane parks here until the record one of its lanes waits for has been published, or every
// trajectory has completed.  Out of line and with exponential back-off: towards the end of a launch most warps are in
// this state, and a tight poll loop (the whole refill block every 200 ns) took the issue slots the last working warps
// needed (measured: the end of the launch stretched from ~0.4 ms to 2-4 ms).
static __device__ __noinline__ void park_idle_warp(volatile int* seq, int epoch, bool pending,
                                                   const volatile unsigned long long* completed, unsigned long long K) {
  unsigned ns = 128;
  for (;;) {
    const bool wake = (pending && *seq == epoch) || *completed >= K;
    if (__any_sync(0xffffffffu, wake)) return;
    __nanosleep(ns);
    if (ns < 4096) ns <<= 1;
  }
}

template <int D>
struct NoisePlan {
  // passes served by one Philox block (D = 1, 2) or blocks needed per pass (D >= 3)
  static constexpr int SPB = (D == 1) ? 4 : (D == 2 ? 2 : 1);
  static constexpr int BPP = (D <= 2) ? 1 : (D + 3) / 4;
  static constexpr int NZ = 4 * BPP;
};

// policy evaluation of the thread-per-trajectory forward kernel: mlp_forward_mma (mlp_mma.cuh) is compiled where it has
// been measured to win, hidden width 32 at d = 1
constexpr bool fwd_mma_shape(int D, int H) { return D == 1 && H == 32; }
struct MlpMmaNone { int unused; };
template <int D, bool MMA> struct FwdMmaSel { typedef typename std::conditional<MMA, MlpMma<D>, MlpMmaNone>::type type; };

// Register budgets.  Left alone, ptxas settles at 67 registers for d = 1 and at ~250 for the wider shapes (2 blocks per
// SM: two warps per scheduler, every FFMA2 waiting for its LDCU.128), although spill-free allocations exist at 64
// (d = 1: 8 blocks per SM), <= 102 (d = 2..4: 5 blocks) and <= 128 (d = 10: 4 blocks) -- it finds them when asked.
// The tensor-core policy holds a half-tile of fragments (A hi / lo, accumulators, B operands) on top of the pass state:
// 80 registers at 6 blocks per SM, measured best (d = 1, 1e6 trajectories: 21.1 ms against 21.8 / 22.2 ms at 5 / 4).
// At 7 blocks (72 registers) ptxas spills 104 B (float32 state) even with the noise in shared memory.
#ifndef RLSDE_FWD_MMA_MIN_BLOCKS
#define RLSDE_FWD_MMA_MIN_BLOCKS 6
#endif
template <int D, bool MMA>
constexpr int fwd_min_blocks() { return MMA ? RLSDE_FWD_MMA_MIN_BLOCKS : (D == 1 ? 8 : (D <= 4 ? 5 : 4)); }
// CLAMP2 = false (MMA, precise tanh): layer 2 of the policy without the clamp of rsig_group, launched where the host has
// proven it cannot bind (fwd_mma_clamp_bounds)
// BRIDGE: the Brownian-bridge hit test between passes (bridge_project; instantiated at d = 1 only).  A compile-time choice,
// so that the kernels without it keep their register allocation
// RAGGED: checkpoints go to the ragged store (ckpt_slot); no transition stream (path_base shares its field)
template <int D, int H, bool F64, bool FAST, bool MMA, bool CLAMP2 = true, bool BRIDGE = false, bool RAGGED = false>
__global__ void __launch_bounds__(128, fwd_min_blocks<D, MMA>()) rollout_fwd_kernel(const __grid_constant__ MlpConst<D, H> W,
                                                          const __grid_constant__ FwdArgs A,
                                                          const __grid_constant__ typename FwdMmaSel<D, MMA>::type M) {
  typedef typename RealT<F64>::type real;
  constexpr int SPB = NoisePlan<D>::SPB;
  constexpr int BPP = NoisePlan<D>::BPP;
  constexpr int NZ = NoisePlan<D>::NZ;
  constexpr unsigned FULL = 0xffffffffu;
  // MMA: the normals of the current noise block wait in shared memory, one column per thread, instead of in registers,
  // where they cost the tensor-core kernel spills and a select chain per pass
  constexpr bool NOISE_SMEM = MMA && SPB > 1;
  const int lane = threadIdx.x & 31;
  __shared__ float s_noise[NOISE_SMEM ? NZ : 1][128];
  // MMA: the block's copy of the fragment and column tables (mlp_mma.cuh)
  __shared__ uint4 s_mma[MMA ? mlp_mma_smem_words<D>() : 1];
  if constexpr (MMA) {
    for (int i = threadIdx.x; i < mlp_mma_smem_words<D>(); i += blockDim.x) s_mma[i] = reinterpret_cast<const uint4*>(&M)[i];
    __syncthreads();
  }
  const bool inject = (A.flags & RLSDE_F_NOISE_INJECTED) != 0;
  const bool s_exact = (A.flags & RLSDE_F_STOCH_INT_EXACT) != 0;
  const bool store_path = (A.flags & RLSDE_F_STORE_PATH) != 0 && A.path != nullptr;
  const bool want_l2 = (D == 1) && A.policy_opt != nullptr && A.l2 != nullptr;
  const long long lim = inject ? (A.noise_steps < A.n_steps_lim ? A.noise_steps : A.n_steps_lim) : A.n_steps_lim;
  const double inv_s2dt = BRIDGE ? bridge_inv_s2dt(A) : 0.0;
  typedef ContRec<D, F64> Rec;
  // tail strategy: 1 = time slices, 2 = hand-off to the latency kernel, 3 = none, 0 = adaptive launch, not decided yet
  const bool adaptive = A.q_ring != nullptr && A.q_adaptive != 0;
  const bool tracked = A.q_ring != nullptr && (A.q_quantum > 0 || A.q_handoff > 0);
  int mode = adaptive ? 0 : (A.q_ring != nullptr && A.q_quantum > 0 ? 1 : (A.q_ring != nullptr && A.q_handoff > 0 ? 2 : 3));
  Rec* const ring = reinterpret_cast<Rec*>(A.q_ring);
  // live state is kept small (the register budget of 8 blocks per SM is 64): while a lane waits for a record, `traj`
  // holds the record's index; slices end where the pass index is a multiple of the quantum (a power of two)
  const int qmask = A.q_quantum - 1;

  bool alive = false, exhausted = false, pending = false, fin = false, capped = false;
  long long traj = 0;
  int k = 0, ck = 0;
  real x[D];
  real G = 0, S = 0, L2 = 0;
  float z[NOISE_SMEM ? 1 : NZ];
#pragma unroll
  for (int i = 0; i < D; ++i) x[i] = F64 ? (real)A.x0_d[i] : (real)A.x0_f[i];
#pragma unroll
  for (int i = 0; i < (NOISE_SMEM ? 1 : NZ); ++i) z[i] = 0.f;

  for (unsigned it = 0;; ++it) {
    if ((it & (SPB - 1)) == 0) {
      if (tracked) {
        // (a) report the trajectories that completed since the last boundary
        const unsigned fm = __ballot_sync(FULL, fin);
        if (fm) {
          if (lane == __ffs(fm) - 1) atomicAdd(A.q_ctrl + 2, (unsigned long long)__popc(fm));
          fin = false;
        }
      }
      if (mode == 0) {
        // adaptive launch, tail strategy not decided yet: count the trajectories that ran into the pass budget and, every
        // other boundary, look whether somebody has decided / whether it is time to decide for time slices
        const unsigned cm = __ballot_sync(FULL, capped);
        if (cm) {
          if (lane == __ffs(cm) - 1) atomicAdd(A.q_ctrl + 4, (unsigned long long)__popc(cm));
          capped = false;
        }
        if ((it & (2u * SPB - 1u)) == 0) {
          unsigned long long m = 0;
          if (lane == 0) {
            m = *reinterpret_cast<volatile unsigned long long*>(A.q_ctrl + 5);
            if (m == 0) {
              const unsigned long long n_cap = *reinterpret_cast<volatile unsigned long long*>(A.q_ctrl + 4);
              const unsigned long long n_done = *reinterpret_cast<volatile unsigned long long*>(A.q_ctrl + 2);
              if (n_done >= 4096 && n_cap * 20 >= n_done) {
                const unsigned long long old = atomicCAS(A.q_ctrl + 5, 0ull, 1ull);
                m = old == 0 ? 1 : old;
              }
            }
          }
          mode = (int)__shfl_sync(FULL, m, 0);
        }
      }
      if (mode == 2 && (it & (4u * SPB - 1u)) == 0) {
        // every 4th boundary: is this the tail of the launch?  then leave the live trajectories to the latency kernel
        const unsigned long long claimed = *reinterpret_cast<volatile unsigned long long*>(A.q_ctrl);
        const unsigned long long completed = *reinterpret_cast<volatile unsigned long long*>(A.q_ctrl + 2);
        if (claimed >= (unsigned long long)A.K && (unsigned long long)A.K - completed <= (unsigned long long)A.q_handoff) {
          const unsigned live = __ballot_sync(FULL, alive);
          if (live) {
            unsigned long long base = 0;
            const int leader = __ffs(live) - 1;
            if (lane == leader) base = atomicAdd(A.q_ctrl + 1, (unsigned long long)__popc(live));
            base = __shfl_sync(FULL, base, leader);
            if (alive) {
              Rec* r = ring + (base + __popc(live & ((1u << lane) - 1u)));
              r->traj = traj; r->k = k; r->seq = 1; r->G = G; r->S = S; r->L2 = L2;
#pragma unroll
              for (int i = 0; i < D; ++i) r->x[i] = x[i];
            }
          }
          break;
        }
      }
      if (mode == 1) {
        // (b) slice over: append the trajectory to the FIFO
        const bool expire = alive && k != 0 && (k & qmask) == 0;   // (a resumed lane is past this check: it resumes in (d))
        const unsigned em = __ballot_sync(FULL, expire);
        if (em) {
          unsigned long long base = 0;
          const int leader = __ffs(em) - 1;
          if (lane == leader) base = atomicAdd(A.q_ctrl + 1, (unsigned long long)__popc(em));
          base = __shfl_sync(FULL, base, leader);
          if (expire) {
            const unsigned long long j = base + __popc(em & ((1u << lane) - 1u));
            Rec* r = ring + (long long)(j & (unsigned long long)(A.q_cap - 1));
            const int epoch = (int)(j >> A.q_cap_log2) + 1;
            // at most K records are in flight and the ring is larger, so the slot's previous record (item j - cap) was
            // claimed long ago; wait for its reader all the same
            volatile int* seq = &r->seq;
            const int free_mark = epoch == 1 ? 0 : 1 - epoch;
            if (*seq != free_mark) wait_for_slot(seq, free_mark);
            r->traj = traj; r->k = k; r->G = G; r->S = S; r->L2 = L2;
#pragma unroll
            for (int i = 0; i < D; ++i) r->x[i] = x[i];
            __threadfence();
            *seq = epoch;
            alive = false;
          }
        }
      }
      // (c) idle lanes claim the next item: a fresh trajectory, or the index of a continuation record to wait for
      const unsigned need = __ballot_sync(FULL, !alive && !exhausted && !pending);
      if (need) {
        unsigned long long base = 0;
        const int leader = __ffs(need) - 1;
        if (lane == leader) base = atomicAdd(A.counter, (unsigned long long)__popc(need));
        base = __shfl_sync(FULL, base, leader);
        if (!alive && !exhausted && !pending) {
          const long long idx = (long long)base + __popc(need & ((1u << lane) - 1u));
          if (idx < A.K) {
            traj = idx; k = 0; ck = 0; alive = true;
            G = 0; S = 0; L2 = 0;
#pragma unroll
            for (int i = 0; i < D; ++i) x[i] = F64 ? (real)A.x0_d[i] : (real)A.x0_f[i];
          } else {
            // no fresh work left.  An undecided adaptive launch decides now: nothing ran into the budget, so the tail
            // is a few long trajectories -> hand-off (unless another warp has just chosen time slices)
            if (mode == 0) {
              const unsigned long long old = atomicCAS(A.q_ctrl + 5, 0ull, 2ull);
              mode = old == 0 ? 2 : (int)old;
            }
            if (mode == 1) { pending = true; traj = idx - A.K; }
            else exhausted = true;
          }
        }
      }
      // the tail strategy is a property of the launch (one global decision): lanes that have just learnt it in (c) tell
      // the rest of the warp, so that `mode` stays warp-uniform (the blocks above use full-mask collectives)
      if (adaptive) mode = (int)__reduce_max_sync(FULL, (unsigned)mode);
      // (d) lanes waiting for a record look at their slot; the other lanes of the warp are not held up
      if (pending) {
        Rec* r = ring + (traj & (A.q_cap - 1));
        const int epoch = (int)(traj >> A.q_cap_log2) + 1;
        volatile int* seq = &r->seq;
        if (*seq == epoch) {
          __threadfence();
          const volatile Rec* v = r;
          traj = v->traj; k = v->k; G = v->G; S = v->S; L2 = v->L2;
#pragma unroll
          for (int i = 0; i < D; ++i) x[i] = v->x[i];
          *seq = -epoch;
          alive = true; pending = false;
          const int rem = k % A.ckpt_every;
          ck = rem ? A.ckpt_every - rem : 0;
        } else if (*reinterpret_cast<volatile unsigned long long*>(A.q_ctrl + 2) >= (unsigned long long)A.K) {
          pending = false; exhausted = true;      // every trajectory has completed: no record will ever arrive
        }
      }
      if (!__any_sync(FULL, alive)) {
        if (!__any_sync(FULL, pending)) break;
        park_idle_warp(&(ring + (traj & (A.q_cap - 1)))->seq, (int)(traj >> A.q_cap_log2) + 1, pending, A.q_ctrl + 2,
                       (unsigned long long)A.K);
        it |= (unsigned)(SPB - 1);                  // stay on a boundary: the refill block above takes it from here
        continue;
      }
      if (!inject) {
        const unsigned long long gt = (unsigned long long)(A.traj_offset + traj);
#pragma unroll
        for (int q = 0; q < BPP; ++q) {
          float zz[4];
          noise_block(A.seed, gt, (unsigned)(k / SPB) * BPP + q, A.noise_scale2, zz);
#pragma unroll
          for (int s = 0; s < 4; ++s) {
            if constexpr (NOISE_SMEM) s_noise[4 * q + s][threadIdx.x] = zz[s];
            else z[4 * q + s] = zz[s];
          }
        }
      }
    }

    // ---- policy
    float xf[D], u[D];
#pragma unroll
    for (int i = 0; i < D; ++i) xf[i] = (float)x[i];
    if constexpr (MMA) {
      bool clamp1 = true;
      if constexpr (!FAST) {
        bool in_x1 = true;
#pragma unroll
        for (int i = 0; i < D; ++i) in_x1 = in_x1 && fabsf(xf[i]) <= A.mma_x1_max;
        clamp1 = !__all_sync(FULL, in_x1);
      }
      // two inlined copies of the whole policy, one per value of clamp1: with the branch around layer 1 alone ptxas
      // spilled ~200 B, with the branch here the float32-state kernel has no spill at all
      const float4* s_col = reinterpret_cast<const float4*>(s_mma + MLP_MMA_FRAG_WORDS);
      if (clamp1) mlp_forward_mma<D, FAST, false, CLAMP2>(s_mma, s_col, M.b3, lane, xf, u, true);
      else mlp_forward_mma<D, FAST, false, CLAMP2>(s_mma, s_col, M.b3, lane, xf, u, false);
    }
    else if constexpr (!FAST && RLSDE_FWD_FOLDED) mlp_forward_folded<D, H>(W, xf, u);   // W is a pack_mlp_const_folded image
    else mlp_forward<D, H, FAST>(W, xf, u);

    // ---- this pass's Brownian increments
    float dB[D];
    if (inject) {
      const long long row = (long long)k * A.K_global + (A.traj_offset + traj);
#pragma unroll
      for (int i = 0; i < D; ++i) dB[i] = (alive && k < lim) ? __ldg(A.noise + row * D + i) : 0.f;
    } else {
      const int sub = (int)(it & (SPB - 1));
#pragma unroll
      for (int i = 0; i < D; ++i) {
        if constexpr (NOISE_SMEM) {
          dB[i] = s_noise[sub * D + i][threadIdx.x];
        } else if constexpr (SPB == 1) {
          dB[i] = z[i];
        } else {
          float v = z[i];
#pragma unroll
          for (int s = 1; s < SPB; ++s) v = (sub == s) ? z[s * D + i] : v;
          dB[i] = v;
        }
      }
    }

    // ---- hit test on the current state
    bool hit;
    if (A.hit_rule == RLSDE_HIT_X0_IN_LB_RB) {
      hit = F64 ? ((double)x[0] >= A.lb_d && (double)x[0] <= A.rb_d) : ((float)x[0] >= A.lb_f && (float)x[0] <= A.rb_f);
    } else {
      hit = true;
#pragma unroll
      for (int i = 0; i < D; ++i) hit = hit && (F64 ? ((double)x[i] >= A.lb_d) : ((float)x[i] >= A.lb_f));
    }

    // ---- stochastic integral, running cost, l2 error
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
      // idx = floor((clip(x) - lo) / h)   environments.py:318-321;  |u - u_opt|^2 dt  approximate_methods.py:610-615
      double xc = (double)x[0];
      xc = xc < A.grid_lo ? A.grid_lo : (xc > A.grid_hi ? A.grid_hi : xc);
      long long gi = (long long)floor((xc - A.grid_lo) / A.grid_h);
      gi = gi < 0 ? 0 : (gi >= A.n_grid ? A.n_grid - 1 : gi);
      const float uo = alive ? __ldg(A.policy_opt + gi) : 0.f;
      const float du = __fsub_rn(u[0], uo);
      L2 = F64 ? (real)__dadd_rn((double)L2, __dmul_rn((double)__fmul_rn(du, du), A.dt_d))
               : (real)__fadd_rn((float)L2, __fmul_rn(__fmul_rn(du, du), A.dt_f));
    }

    if (alive) {
      if (store_path) {
        if (ck == 0) {
          const int ci = A.ckpt_log2 >= 0 ? (k >> A.ckpt_log2) : (k / A.ckpt_every);      // no integer division per pass
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
      // running cost  r = -(1 + 0.5 |u|^2) dt   (environments.py:104-110,121-127; f = 1, g = 0)
      real r;
      {
        const float nn = (D == 1) ? n2 : __fmul_rn(sqrtf(n2), sqrtf(n2));
        if (F64) {
          // numpy: f (float64 ones) + float32(0.5 * norm(a)^2)  -> float64, times python-float dt
          r = (real)(-__dmul_rn(__dadd_rn(1.0, (double)__fmul_rn(0.5f, nn)), A.dt_d));
        } else {
          r = (real)(-__fmul_rn(__fadd_rn(1.0f, __fmul_rn(0.5f, nn)), A.dt_f));
        }
      }
      // Euler-Maruyama:  x + (-gradV(x) + sigma u) dt + sigma dB,  gradV = 4 alpha x (x^2 - 1)
      real xn[D];
#pragma unroll
      for (int i = 0; i < D; ++i) {
        if (F64) {
          const double xi = (double)x[i];
          double g;
          if (D == 1 && k == 0) {
            // numpy 1-D: the first pass sees a float32 state and a python-float alpha -> float32 gradient
            const float xs = (float)xi;
            g = (double)__fmul_rn(__fmul_rn(A.c4a_f[i], xs), __fsub_rn(__fmul_rn(xs, xs), 1.0f));
          } else if (k == 0) {
            // numpy d-D: float64 alpha array, but state**2 - 1 is still float32 on the first pass
            const float xs = (float)xi;
            g = __dmul_rn(__dmul_rn(A.c4a_d[i], xi), (double)__fsub_rn(__fmul_rn(xs, xs), 1.0f));
          } else {
            g = __dmul_rn(__dmul_rn(A.c4a_d[i], xi), __dsub_rn(__dmul_rn(xi, xi), 1.0));
          }
          const double drift = __dmul_rn(__dadd_rn(-g, __dmul_rn(A.sigma_d, (double)u[i])), A.dt_d);
          xn[i] = (real)__dadd_rn(__dadd_rn(xi, drift), __dmul_rn(A.sigma_d, (double)dB[i]));
        } else {
          const float xi = (float)x[i];
          const float g = __fmul_rn(__fmul_rn(A.c4a_f[i], xi), __fsub_rn(__fmul_rn(xi, xi), 1.0f));
          const float drift = __fmul_rn(__fadd_rn(-g, __fmul_rn(A.sigma_f, u[i])), A.dt_f);
          xn[i] = (real)__fadd_rn(__fadd_rn(xi, drift), __fmul_rn(A.sigma_f, dB[i]));
        }
      }
      if (!RAGGED && A.tr_base != nullptr) {
        // (state, action, reward, next_state, done) of this pass, cast to the replay buffer's float32 arrays
        // (replay_buffers.py:23-33,56-68); on the detecting pass the reward is -g(x) = -0 (environments.py:104-110)
        const long long slot = A.tr_base[traj] + k;
#pragma unroll
        for (int i = 0; i < D; ++i) {
          A.tr_state[slot * D + i] = (float)x[i];
          A.tr_action[slot * D + i] = u[i];
          A.tr_next[slot * D + i] = (float)xn[i];
        }
        A.tr_reward[slot] = hit ? -0.0f : (float)r;
        A.tr_done[slot] = hit ? 1 : 0;
      }
      if (hit) {
        const real Sout = s_exact ? S_prev : S;
        if (F64) {
          ((double*)A.G)[traj] = (double)G;
          ((double*)A.S)[traj] = (double)Sout;
          if (A.l2) ((double*)A.l2)[traj] = (double)L2;
          if (A.logw) ((double*)A.logw)[traj] = (double)G - (double)S_prev;
        } else {
          ((float*)A.G)[traj] = (float)G;
          ((float*)A.S)[traj] = (float)Sout;
          if (A.l2) ((float*)A.l2)[traj] = (float)L2;
          if (A.logw) ((float*)A.logw)[traj] = (float)G - (float)S_prev;
        }
        A.T[traj] = k;
        alive = false; fin = true;
      } else {
        if constexpr (BRIDGE) bridge_project(A, inv_s2dt, (unsigned long long)(A.traj_offset + traj), k, x[0], xn[0]);
        G = add_rn(G, r);
#pragma unroll
        for (int i = 0; i < D; ++i) x[i] = xn[i];
        ++k;
        if (k >= lim) {
          // not detected within the pass budget: flagged, never garbage (SURVEY section 5, failure row)
          if (F64) {
            ((double*)A.G)[traj] = (double)G;
            ((double*)A.S)[traj] = (double)S;
            if (A.l2) ((double*)A.l2)[traj] = (double)L2;
            if (A.logw) ((double*)A.logw)[traj] = (double)G - (double)S;
          } else {
            ((float*)A.G)[traj] = (float)G;
            ((float*)A.S)[traj] = (float)S;
            if (A.l2) ((float*)A.l2)[traj] = (float)L2;
            if (A.logw) ((float*)A.logw)[traj] = (float)G - (float)S;
          }
          A.T[traj] = -1;
          alive = false; fin = true; capped = true;
        }
      }
    }
  }
}

// Kernel variant of a forward launch from its flags, for every forward family, as std::bool_constant arguments.  Two
// rules prune what is compiled, and the C ABI refuses the flags they exclude: the Brownian-bridge test is compiled at
// d = 1 only and never with the ragged checkpoint store (with_fwd_bridge: f(BRIDGE)); the ragged store takes the float32
// state only (with_fwd_state: f(F64, FAST)).  with_fwd_variant: f(F64, FAST, BRIDGE).
template <int D, bool RAGGED, class F>
static inline int with_fwd_bridge(unsigned flags, F&& f) {
  return with_flag<D == 1 && !RAGGED>((flags & RLSDE_F_HIT_BRIDGE) != 0, f);
}
template <bool RAGGED, class F>
static inline int with_fwd_state(unsigned flags, F&& f) {
  return with_flag<!RAGGED>((flags & RLSDE_F_STATE_F64) != 0, [&](auto f64) {
    return with_flag((flags & RLSDE_F_TANH_FAST) != 0, [&](auto fast) { return f(f64, fast); });
  });
}
template <int D, bool RAGGED, class F>
static inline int with_fwd_variant(unsigned flags, F&& f) {
  return with_fwd_bridge<D, RAGGED>(flags, [&](auto bridge) {
    return with_fwd_state<RAGGED>(flags, [&](auto f64, auto fast) { return f(f64, fast, bridge); });
  });
}

// host-side launcher for one (D, H) shape; defined in rollout_fwd_inst.cuh.  RAGGED: the ragged checkpoint store (float32
// state only, no Brownian-bridge test: the caller refuses both)
template <int D, int H, bool RAGGED = false>
int launch_rollout_fwd(const float* params_host, const FwdArgs& args, int sm_count, cudaStream_t stream);

// d = 1 rollout under the control table_dev[grid_index(x)] (fwd_tab_d1.cu).  Tables of up to FWD_TAB_SMEM_MAX entries
// (32 KB) are copied to shared memory when a block starts, larger ones are read through the read-only cache.
constexpr long long FWD_TAB_SMEM_MAX = 8192;
int launch_rollout_fwd_table(const float* table_dev, const FwdArgs& args, int sm_count, cudaStream_t stream);

}  // namespace rlsde
