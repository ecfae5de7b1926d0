/*
 * rlsde.h -- C ABI of librlsde_b200.so: the B200 (sm_100a) implementation of the
 * data-parallel hot path of riberaborrell/rl-sde-is.
 *
 * The reference is pure Python and has no FFI layer; its boundary is the Python call
 * surface listed below.  Each entry point here is what a ctypes binding for that call
 * would bind (the binding itself is rl_sde_is_b200/_lib.py; INTEGRATION.md shows the
 * stub a reference maintainer would add).  Citations are into /root/reference/src/rl_sde_is/.
 *
 *   rlsde_rollout_fwd   whole-rollout replacement for the loops of
 *                       sample_loss_vectorized      reinforce_deterministic_core.py:30-93
 *                       test_policy_vectorized      approximate_methods.py:577-648
 *                       estimate_fht_vectorized     approximate_methods.py:650-695
 *                       (which call env.step_torch / env.step once per pass:
 *                        environments.py:139-162,201-226; environments_2d.py:134-153,184-205)
 *   rlsde_rollout_fwd_table  the same rollout at d = 1 under a tabulated control (DP greedy policy, HJB u*)
 *   rlsde_rollout_bwd   eff_loss.backward()         reinforce_deterministic_core.py:240
 *                       (BPTT through every pass; states are never detached, :88)
 *   rlsde_tables        compute_r_table / compute_p_tensor_batch   dynamic_programming.py:3-36
 *                       + state_action_transition_function          environments.py:87-102
 *   rlsde_dp_sweep      the Bellman sweeps of q_table_update_vect / v_table_update_vect / policy_update_vect
 *                       over a device-resident tensor; rlsde_dp_sweep_implicit the same sweep with the
 *                       tensor generated inside it, for grids whose tensor does not fit
 *   rlsde_env_step      env.step / env.step_torch (single pass, API completeness)
 *   rlsde_noise_fill    the Brownian increments env.step* draws (environments.py:145,208),
 *                       from the same counter-based generator the rollout kernels use
 *   rlsde_reduce_stats  np.mean / np.var of the per-trajectory results
 *                       (reinforce_deterministic_core.py:249-253, approximate_methods.py:645-646)
 *
 * Conventions
 *   - plain C types only; every *_dev pointer is a CUDA device pointer owned by the caller;
 *     the library keeps no pointer after a call returns and allocates nothing persistent;
 *   - all work is enqueued on the caller's stream (cudaStream_t passed as void*) and the
 *     calls return without synchronising, unless stated otherwise;
 *   - return value: 0 on success, a negative rlsde_status otherwise; never throws / exits;
 *   - policy parameters are passed as a HOST pointer to one flat float32 buffer in the order
 *     of the reference's state_dict (models.py:4-18): policy.0.weight (H,d) row-major,
 *     policy.0.bias (H), policy.2.weight (H,H), policy.2.bias (H), policy.4.weight (d,H),
 *     policy.4.bias (d).  They travel to the GPU by value as a kernel parameter (constant
 *     bank), which is what lets the GEMV use uniform-register FFMA2 operands.
 */
#ifndef RLSDE_H_
#define RLSDE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RLSDE_VERSION 200       /* 0.2.0: rlsde_rollout_cfg grew the scheduling knobs */
#define RLSDE_MAX_D 16          /* largest state / action dimension */
#define RLSDE_NSTATS 16         /* doubles in a statistics record */

/* status codes */
typedef enum rlsde_status {
  RLSDE_OK = 0,
  RLSDE_ERR_INVALID_ARG = -1,   /* null pointer, negative size, bad flag combination */
  RLSDE_ERR_UNSUPPORTED = -2,   /* (d, hidden width, depth) without a compiled kernel */
  RLSDE_ERR_CUDA = -3,          /* a CUDA runtime call or launch failed (see rlsde_last_cuda_error) */
  RLSDE_ERR_NO_DEVICE = -4,     /* no CUDA device / device is not sm_100 */
  RLSDE_ERR_WORKSPACE = -5      /* workspace too small (see rlsde_workspace_bytes) */
} rlsde_status;

/* hit_rule: how "state is in the target set" is decided */
#define RLSDE_HIT_ALL_GE_LB 0   /* all_i x_i >= lb     is_done_torch environments.py:51-52; d-D: environments_2d.py:56-61 */
#define RLSDE_HIT_X0_IN_LB_RB 1 /* lb <= x_0 <= rb     is_done (numpy, 1-D)  environments.py:48-49 */

/* rollout flags */
#define RLSDE_F_NOISE_INJECTED (1u << 0) /* read increments from noise_dev instead of Philox */
#define RLSDE_F_TANH_FAST (1u << 1)      /* tanh.approx (2^-11 rel. error): statistical parity only */
#define RLSDE_F_STOCH_INT_EXACT (1u << 2)/* drop the extra u(X_k*) dB term of the reference (SURVEY App. A-4) */
#define RLSDE_F_STATE_F64 (1u << 3)      /* numpy-path arithmetic: f64 state and accumulators, f32 policy
                                            (SURVEY App. A-5); G/S/l2/logw outputs are double* */
#define RLSDE_F_STORE_PATH (1u << 4)     /* write X_k checkpoints (needed by rlsde_rollout_bwd) */
#define RLSDE_F_HIT_BRIDGE (1u << 6)     /* d = 1, rlsde_rollout_fwd / rlsde_rollout_fwd_table only: also detect target hits
                                            between passes with a Brownian-bridge crossing test.  After the Euler-Maruyama
                                            update of a pass whose X_k was no hit, with a = X_k, b = X_{k+1} and the target
                                            [lb, rb] (rb = +inf under RLSDE_HIT_ALL_GE_LB): a and b on opposite sides of it
                                            crossed; both below lb (above rb) crossed if U < exp(-2 (c-a)(c-b) / (sigma^2 dt))
                                            with c = lb (rb).  A crossing sets X_{k+1} to that barrier, which the next pass's
                                            hit test detects: T, G, S, logw, l2 keep their definitions and the hit is
                                            credited at t_{k+1}.  U = (r.x + 0.5) 2^-32, r = Philox4x32-10(counter (traj_lo,
                                            traj_hi, k, 0x42524447), key seed) of the global trajectory id, also with
                                            RLSDE_F_NOISE_INJECTED; the Brownian increments are those of the rollout without
                                            the flag.  p is evaluated in double.  exp(G - S_exact) stays the exact likelihood
                                            ratio of the process stopped this way, so every policy estimates the same Psi.
                                            With RLSDE_F_STORE_PATH -> RLSDE_ERR_INVALID_ARG (the reverse pass knows nothing
                                            of the projection); d >= 2 -> RLSDE_ERR_UNSUPPORTED (no closed form for the
                                            orthant); rlsde_rollout_transitions, rlsde_env_step and the training entry points
                                            refuse it (RLSDE_ERR_INVALID_ARG) */
#define RLSDE_F_KERNEL_THREAD (1u << 8)   /* force the throughput kernels (one trajectory per thread) */
#define RLSDE_F_KERNEL_WARP (1u << 9)     /* force the latency kernels (one trajectory per warp; hidden width 32, and for the
                                            reverse pass ckpt_every == 1).  Default: chosen from K (small batches -> warp) */
#define RLSDE_F_KERNEL_TENSOR (1u << 10)  /* force the tile kernel with the hidden-hidden layer on the tensor cores (tcgen05; one
                                            thread per trajectory, 128-trajectory tiles).  Default: large batches with a bounded pass budget */
#define RLSDE_F_GRAD_F32 (1u << 5)       /* rlsde_env_step with RLSDE_F_STATE_F64: the caller's state array was float32.  numpy then
                                            evaluates grad V in float32 in the 1-D env (python-float alpha), and state**2 - 1 in
                                            float32 in the d-D env (float64 alpha array)  (SURVEY App. A-5) */

/* environment: overdamped Langevin dX = (-grad V + sigma u) dt + sigma dW,
   V(x) = sum_i alpha_i (x_i^2 - 1)^2   (environments.py:42-46, environments_2d.py:44-54) */
typedef struct rlsde_env {
  int32_t d;                    /* state = action dimension, 1..RLSDE_MAX_D */
  int32_t hit_rule;             /* RLSDE_HIT_* */
  double alpha[RLSDE_MAX_D];
  double sigma;                 /* sqrt(2 / beta) */
  double dt;
  double lb, rb;                /* target set bounds (1, 2) */
  double x0[RLSDE_MAX_D];       /* initial state (-1, ..., -1) */
} rlsde_env;

/* policy: a = W3 tanh(W2 tanh(W1 x + b1) + b2) + b3   (models.py:4-18, n_layers = 3) */
typedef struct rlsde_mlp {
  int32_t d_in;                 /* = env.d */
  int32_t d_hidden;             /* H */
  int32_t d_out;                /* = env.d */
  int32_t n_hidden;             /* number of hidden (tanh) layers; 2 is what the reference builds */
} rlsde_mlp;

typedef struct rlsde_rollout_cfg {
  int64_t K;                    /* trajectories handled by this call */
  int64_t traj_offset;          /* global id of local trajectory 0 (sharding: SURVEY 8e) */
  int64_t K_global;             /* trajectories over all shards (row stride of injected noise) */
  uint64_t seed;                /* Philox key */
  int64_t n_steps_lim;          /* a trajectory not detected within this many passes is "unfinished" */
  int64_t noise_steps;          /* passes available in noise_dev (RLSDE_F_NOISE_INJECTED) */
  uint32_t flags;               /* RLSDE_F_* */
  int32_t ckpt_every;           /* RLSDE_F_STORE_PATH: keep X_k for k % ckpt_every == 0 (>= 1) */
  int64_t ckpt_stride;          /* checkpoints reserved per trajectory (>= ceil(n_steps_lim / ckpt_every)) */
  /* optional lookup table for the l2 error of test_policy_vectorized (approximate_methods.py:610-615),
     d == 1 only: idx = floor((clip(x, grid_lo, grid_hi) - grid_lo) / grid_h)  (environments.py:318-321) */
  int64_t n_grid;
  double grid_lo, grid_hi, grid_h;
  /* scheduling knobs (tuning / tests only; 0 = automatic everywhere, so a zero-initialised struct is the default).
     They change the schedule, never a per-trajectory result (tested bit for bit).  The library itself reads no
     environment variables; the Python binding maps RLSDE_FWD_QUANTUM / RLSDE_FWD_HANDOFF / RLSDE_BWD_WARP_SHARE /
     RLSDE_FWD_BLOCKS_PER_SM onto these fields. */
  int32_t fwd_quantum;          /* thread-per-trajectory forward kernel: n > 0 = time slices of n passes, -1 = run to
                                   completion (+ tail hand-off), 0 = adaptive */
  int32_t fwd_blocks_per_sm;    /* n > 0: cap on resident blocks per SM of the forward kernel */
  int64_t fwd_handoff;          /* live trajectories at which the tail goes to the warp-per-trajectory kernel
                                   (-1 = never, 0 = automatic) */
  int64_t bwd_warp_share;       /* longest trajectories the reverse pass gives to the warp-per-trajectory kernel
                                   (-1 = none, 0 = automatic) */
  int32_t bwd_kernel;           /* thread-per-trajectory reverse pass, hidden width 32: 0 or 1 = tensor-core kernel
                                   (mma.sync, float16 x 3 split); any other value is refused (RLSDE_ERR_UNSUPPORTED) */
  int32_t wide_kernel;          /* forward rollout (hidden width 64 / 128 / 256) and reverse pass (128 / 256): 0 = automatic (tcgen05
                                   kernels for batches of at least 512 trajectories at width 256, 64 x SMs below; the reverse pass also needs a
                                   workspace of rlsde_workspace_bytes_bwd), 1 = tcgen05 kernels, 2 = CUDA-core tile kernels */
  int32_t fwd_policy;           /* policy evaluation of the thread-per-trajectory forward kernel and of the kernel that
                                   continues its tail: 0 = automatic (tensor cores at d = 1, hidden width 32), 1 = 32 x 32
                                   layer on the tensor cores (mma.sync, float16 x 3 split; d = 1, hidden width 32 only),
                                   2 = CUDA cores (FFMA2).  Results differ between 1 and 2 by rounding. */
} rlsde_rollout_cfg;

/* layout of a statistics record (double[RLSDE_NSTATS]); sums are over the K local trajectories,
   "finished" means detected within n_steps_lim */
enum {
  RLSDE_ST_N = 0,               /* K */
  RLSDE_ST_N_UNFINISHED = 1,
  RLSDE_ST_SUM_G = 2,           /* finished only: sum of return_fht */
  RLSDE_ST_SUM_G2 = 3,
  RLSDE_ST_SUM_T = 4,           /* finished only: sum of hit index k* (numpy convention; torch's time_steps = k*+1) */
  RLSDE_ST_SUM_T2 = 5,
  RLSDE_ST_SUM_S = 6,
  RLSDE_ST_SUM_L2 = 7,
  RLSDE_ST_SUM_W = 8,           /* sum of exp(logw): importance-sampling estimator numerator (SURVEY App. C) */
  RLSDE_ST_SUM_W2 = 9,
  RLSDE_ST_SUM_LOSS = 10,       /* sum of -G - G*S    (eff_loss numerator, reinforce_deterministic_core.py:91) */
  RLSDE_ST_USEFUL_STEPS = 11,   /* sum of passes executed: k*+1 if finished else n_steps_lim (SURVEY 8d metric) */
  RLSDE_ST_MAX_T = 12
};

int rlsde_version(void);
const char* rlsde_strerror(int status);
/* text of the last CUDA error seen by this thread's calls ("" if none) */
const char* rlsde_last_cuda_error(void);
/* kernels this library has launched in this process so far (diagnostics: bench.py's gpu_launches) */
long long rlsde_launch_count(void);
/* SM count and compute capability of the current device */
int rlsde_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor);
/* 1 if a fused kernel is compiled for this policy shape */
int rlsde_supported(int32_t d, int32_t d_hidden, int32_t n_hidden);
/* number of policy parameters P = dH+H + H^2+H + Hd+d */
int64_t rlsde_param_count(const rlsde_mlp* mlp);
/* bytes of scratch the rollout / backward / reduction kernels need for K trajectories */
size_t rlsde_workspace_bytes(int64_t K);
/* the same for a workspace that is also handed to rlsde_rollout_bwd with a policy of this shape: at hidden width 128 / 256
 * the tcgen05 reverse pass keeps its operand-exchange ring and float64 partials there (about 80 MB on a 148-SM device);
 * with the smaller rlsde_workspace_bytes(K) buffer the call falls back to the CUDA-core tile kernel */
size_t rlsde_workspace_bytes_bwd(int64_t K, int32_t d, int32_t d_hidden);

/*
 * Forward rollout of K trajectories (one launch for the whole rollout, not one per pass).
 * Per trajectory, with X_0 = x0, u_j = policy(X_j), k* = first j with X_j in the target set
 * (tested on the CURRENT state, SURVEY App. A-1):
 *   G    = sum_{j<k*} -(1 + |u_j|^2 / 2) dt                   return_fht
 *   S    = sum_{j<=k*} u_j . dB_{j+1}   (j<k* with RLSDE_F_STOCH_INT_EXACT)   stoch_int_fht
 *   T    = k*   (int32; -1 if not detected within n_steps_lim passes)
 *   l2   = sum_{j<=k*} |u_j - policy_opt[idx(X_j)]|^2 dt       (optional)
 *   logw = G - sum_{j<k*} u_j . dB_{j+1}                       log importance weight (optional)
 * Outputs are float* (double* with RLSDE_F_STATE_F64) of length K; T is int32.
 * noise_dev: float[noise_steps][K_global][d] (pass-major, the order the reference draws them).
 * path_dev:  float[K][ckpt_stride][d] checkpoints X_{c*ckpt_every}, or NULL.
 * stats_dev: double[RLSDE_NSTATS], filled by a deterministic reduction after the rollout, or NULL.
 */
int rlsde_rollout_fwd(const rlsde_env* env, const rlsde_mlp* mlp, const float* params_host,
                      const rlsde_rollout_cfg* cfg, const float* noise_dev, const float* policy_opt_dev,
                      void* G_dev, void* S_dev, int32_t* T_dev, void* l2_dev, void* logw_dev,
                      float* path_dev, double* stats_dev, void* workspace_dev, size_t workspace_bytes,
                      void* stream);

/*
 * Forward rollout at d = 1 under a tabulated control instead of an MLP:  u_j = u_table[idx(X_j)],
 *   idx(x) = floor((clip(x, grid_lo, grid_hi) - grid_lo) / grid_h), clamped to [0, n_grid - 1],
 * evaluated on the state in state precision (float32, or float64 with RLSDE_F_STATE_F64) -- the lookup of the l2 error.
 * u_table_dev: float[cfg->n_grid]; policy_opt_dev (optional, for l2) lives on the same grid.  Everything else is
 * rlsde_rollout_fwd's: outputs, statistics record, RLSDE_F_NOISE_INJECTED / STOCH_INT_EXACT / STATE_F64 and the hit
 * rule; tanh and kernel-family flags do not apply, RLSDE_F_STORE_PATH is refused (a table has no gradient).
 * Errors: env->d != 1 -> RLSDE_ERR_UNSUPPORTED; u_table_dev NULL, n_grid < 1 or grid_h <= 0 -> RLSDE_ERR_INVALID_ARG;
 * a workspace smaller than rlsde_workspace_bytes(0) -> RLSDE_ERR_WORKSPACE.
 */
int rlsde_rollout_fwd_table(const rlsde_env* env, const float* u_table_dev, const rlsde_rollout_cfg* cfg,
                            const float* noise_dev, const float* policy_opt_dev, void* G_dev, void* S_dev, int32_t* T_dev,
                            void* l2_dev, void* logw_dev, double* stats_dev, void* workspace_dev, size_t workspace_bytes,
                            void* stream);

/*
 * Forward rollout that also streams every transition out (replay-buffer sampler, SURVEY 8f-4):
 * sample_trajectories_buffer_vectorized approximate_methods.py:513-545 + ReplayBuffer.store_vectorized
 * replay_buffers.py:56-68.  For trajectory t and each pass k it executes (k = 0 .. k*, the detecting pass included;
 * k = 0 .. n_steps_lim-1 if never detected) the tuple lands at slot  slot_base_dev[t] + k :
 *   states[slot][d]  = X_k            actions[slot][d] = policy(X_k)
 *   rewards[slot]    = -(1 + |u|^2/2) dt, or -0 on the detecting pass (environments.py:104-110, 152-155)
 *   next_states[slot][d] = X_{k+1} (the Euler-Maruyama pass is evaluated on the detecting pass too, as env.step does)
 *   done[slot]       = X_k in the target set
 * all cast to float32 / uint8 the way the reference's float32 buffer arrays cast them.  The number of passes of a
 * trajectory is only known after a rollout: call rlsde_rollout_fwd first with the same cfg (the counter-based noise
 * makes the second rollout identical), build slot_base as the exclusive prefix sum of (T >= 0 ? T + 1 : n_steps_lim),
 * then call this.  Slots are trajectory-major; the reference's pass-major order is a stable sort by k.
 * G/S/T/stats as in rlsde_rollout_fwd.  RLSDE_F_STORE_PATH is not accepted.
 */
int rlsde_rollout_transitions(const rlsde_env* env, const rlsde_mlp* mlp, const float* params_host,
                              const rlsde_rollout_cfg* cfg, const float* noise_dev, const int64_t* slot_base_dev,
                              float* states_dev, float* actions_dev, float* rewards_dev, float* next_states_dev,
                              uint8_t* done_dev, void* G_dev, void* S_dev, int32_t* T_dev, double* stats_dev,
                              void* workspace_dev, size_t workspace_bytes, void* stream);

/*
 * Reverse (adjoint) pass: gradient of  L = loss_scale * sum_k ( -G_k - sg(G_k) S_k )  w.r.t. the
 * policy parameters, through the whole rollout (what eff_loss.backward() computes,
 * reinforce_deterministic_core.py:91,240; recursion in SURVEY App. C).  Needs the G/T outputs
 * and the checkpoints of a forward call made with RLSDE_F_STORE_PATH and the same cfg.
 * grad_dev: float[P] in state_dict order, overwritten.  Unfinished trajectories contribute 0.
 * order_dev: optional int64[K] permutation of the local trajectory ids giving the processing order; passing the
 * ids sorted by decreasing T balances the lock-step lanes (trajectories are dealt round-robin in this order).  The
 * result does not depend on it beyond fp32 summation order; NULL = identity.
 */
int rlsde_rollout_bwd(const rlsde_env* env, const rlsde_mlp* mlp, const float* params_host,
                      const rlsde_rollout_cfg* cfg, const float* noise_dev, const float* G_dev,
                      const int32_t* T_dev, const float* path_dev, const int64_t* order_dev, double loss_scale,
                      float* grad_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

/*
 * Reverse pass of any loss over the returns and stochastic integrals: the gradient
 *     grad = loss_scale * sum_k [T_k >= 0] ( cG_k dG_k/dtheta + cS_k dS_k/dtheta )
 * with per-trajectory coefficients coef_G_dev / coef_S_dev (float[K], indexed by local trajectory id), S = S_ref, or
 * S_exact under RLSDE_F_STOCH_INT_EXACT.  The derivative is the pathwise one along the sampled path with the hit passes
 * held fixed, as in rlsde_rollout_bwd; only the adjoint input of pass j changes:
 *     a_j = -cG_k [j<k*] u_j dt + cS_k [j<=k*, or j<k* with RLSDE_F_STOCH_INT_EXACT] dB_{j+1} + sigma dt lambda_{j+1}
 * rlsde_rollout_bwd is the case cG = -1, cS = -G, and with those coefficients this call returns its gradient bit for bit.
 * For a loss f(G, S) pass cG = df/dG, cS = df/dS (e.g. from autograd over G and S).  Kernel selection, order_dev,
 * traj_offset / K_global, bwd_warp_share, the workspace (rlsde_workspace_bytes_bwd at hidden widths 64..256) and every
 * refusal are those of rlsde_rollout_bwd; a NULL coefficient pointer is RLSDE_ERR_INVALID_ARG.
 */
int rlsde_rollout_bwd_weighted(const rlsde_env* env, const rlsde_mlp* mlp, const float* params_host,
                               const rlsde_rollout_cfg* cfg, const float* noise_dev,
                               const float* coef_G_dev, const float* coef_S_dev, const int32_t* T_dev,
                               const float* path_dev, const int64_t* order_dev, double loss_scale,
                               float* grad_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

/*
 * The ragged checkpoint store: memory in proportion to the passes the trajectories run, not to the pass budget.  With
 * C = cfg->ckpt_every (1 .. 32), the checkpoints of trajectory t are X_{cC} for c = 0 .. floor(T_t / C), stored as
 * float[d] rows path_dev[(path_base_dev[t] + c) * d ...]; path_base_dev is int64[K + 1], nondecreasing, and trajectory t
 * owns rows [path_base_dev[t], path_base_dev[t + 1]).  A trajectory with T = -1 is given 0 rows.  The lengths are only
 * known after a rollout: run one first with the same cfg (the counter-based noise makes the second rollout identical;
 * the same entry point with a base of K + 1 zeros stores nothing and runs the same kernels), form the base as the
 * exclusive prefix sum of (T >= 0 ? T / C + 1 : 0) with the total in entry K, then call rlsde_rollout_fwd_ragged.
 *
 * rlsde_rollout_fwd_ragged: rlsde_rollout_fwd with RLSDE_F_STORE_PATH implied and cfg->ckpt_stride not read; flags,
 * kernel selection, outputs and the statistics record are rlsde_rollout_fwd's.  A checkpoint outside a trajectory's rows
 * is not written.  rlsde_rollout_bwd_ragged: rlsde_rollout_bwd_weighted over the ragged store (same semantics, kernel
 * selection, workspace and refusals; with coefficients (-1, -G) it returns rlsde_rollout_bwd's gradient); a trajectory
 * whose rows do not hold checkpoints 0 .. floor(T_t / C) contributes 0, so nothing outside its rows is read.
 * Refusals, before any device work: RLSDE_F_HIT_BRIDGE, ckpt_every outside 1 .. 32 (rlsde_rollout_fwd_ragged), a NULL
 * path_base_dev or path_dev -> RLSDE_ERR_INVALID_ARG; RLSDE_F_STATE_F64 -> RLSDE_ERR_UNSUPPORTED.
 */
int rlsde_rollout_fwd_ragged(const rlsde_env* env, const rlsde_mlp* mlp, const float* params_host,
                             const rlsde_rollout_cfg* cfg, const float* noise_dev, const int64_t* path_base_dev,
                             void* G_dev, void* S_dev, int32_t* T_dev, float* path_dev, double* stats_dev,
                             void* workspace_dev, size_t workspace_bytes, void* stream);
int rlsde_rollout_bwd_ragged(const rlsde_env* env, const rlsde_mlp* mlp, const float* params_host,
                             const rlsde_rollout_cfg* cfg, const float* noise_dev, const float* coef_G_dev,
                             const float* coef_S_dev, const int32_t* T_dev, const int64_t* path_base_dev,
                             const float* path_dev, const int64_t* order_dev, double loss_scale, float* grad_dev,
                             void* workspace_dev, size_t workspace_bytes, void* stream);

/*
 * One REINFORCE iteration with everything resident on the device (reinforce_deterministic_core.py:232-243:
 * zero_grad -> sample_loss_vectorized -> backward -> Adam step), for the latency-bound small-batch regime
 * (K <= 16 x SMs, hidden width 32; RLSDE_ERR_UNSUPPORTED otherwise): the policy is read from theta_dev (float[P],
 * state_dict order), the forward rollout, the statistics reduction, the reverse pass and the Adam update are enqueued
 * back to back and nothing is read back, so consecutive iterations need no host round trip.
 *   theta_dev, adam_m_dev, adam_v_dev: float[P], updated in place (torch.optim.Adam semantics, amsgrad / weight decay off);
 *   step_t: 1-based Adam step (bias corrections);  cfg: RLSDE_F_STORE_PATH with ckpt_every == 1, float32 state;
 *   G/S/T/stats/grad: this iteration's per-trajectory results, statistics record and gradient of
 *   mean_k(-G_k - sg(G_k) S_k) -- e.g. rows of a device-side log the caller reads once at the end.
 * A trajectory that does not reach the target set within n_steps_lim contributes nothing to the gradient and is
 * counted in stats[RLSDE_ST_N_UNFINISHED]; such a batch does NOT update theta / m / v (the Adam kernel looks at the
 * count on the device), and the caller sees it when it reads the log.
 */
int rlsde_reinforce_step(const rlsde_env* env, const rlsde_mlp* mlp, float* theta_dev, float* adam_m_dev, float* adam_v_dev,
                         const rlsde_rollout_cfg* cfg, const float* noise_dev, double lr, double beta1, double beta2,
                         double eps, int64_t step_t, float* G_dev, float* S_dev, int32_t* T_dev, float* path_dev,
                         double* stats_dev, float* grad_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

/*
 * The same iteration split in two for data-parallel training (SURVEY 8e: trajectories sharded over the GPUs of a box,
 * ONE exchange per iteration).  rlsde_reinforce_rollout runs this rank's shard (cfg.K of cfg.K_global trajectories,
 * gradient scaled by 1 / K_global) and leaves the row  [grad as P doubles | statistics record]  in packed_dev
 * (double[P + RLSDE_NSTATS]).  The caller all-gathers the rows of all ranks (one collective, e.g. ncclAllGather through
 * torch.distributed, enqueued on the same stream) and hands the n_ranks rows to rlsde_reinforce_apply, which adds them
 * in rank order -- every rank forms bit-identical sums -- writes the global gradient / statistics (optional outputs)
 * and takes the Adam step, unless some rank reported an unfinished trajectory.
 */
int rlsde_reinforce_rollout(const rlsde_env* env, const rlsde_mlp* mlp, const float* theta_dev, const rlsde_rollout_cfg* cfg,
                            const float* noise_dev, float* G_dev, float* S_dev, int32_t* T_dev, float* path_dev,
                            double* stats_dev, float* grad_dev, double* packed_dev, void* workspace_dev,
                            size_t workspace_bytes, void* stream);
int rlsde_reinforce_apply(const rlsde_mlp* mlp, float* theta_dev, float* adam_m_dev, float* adam_v_dev,
                          const double* packed_all_dev, int32_t n_ranks, double lr, double beta1, double beta2, double eps,
                          int64_t step_t, float* grad_out_dev, double* stats_out_dev, void* stream);

/* Deterministic fp64 reduction of per-trajectory outputs into a statistics record. */
int rlsde_reduce_stats(int64_t K, int64_t n_steps_lim, uint32_t flags, const void* G_dev, const void* S_dev,
                       const int32_t* T_dev, const void* l2_dev, const void* logw_dev, double* stats_dev,
                       void* workspace_dev, size_t workspace_bytes, void* stream);

/*
 * Tabular transition tensor and reward table (dynamic_programming.py:3-36):
 *   P[s', s, a]  (C order, action innermost)  for s' in [sprime_begin, sprime_end): the slab
 *                P_dev points at has (sprime_end - sprime_begin) * Ns * Na doubles;
 *   R[s, a]      Ns * Na doubles (written when R_dev != NULL).
 * For s outside the target set: Phi((x_s'+h-mu)/sd) - Phi((x_s'-h-mu)/sd) with the two tails
 * folded into rows 0 and Ns-1; for s in the target set: 1/|TS| if s' in TS else 0.
 * h_half is the bin half-width (the reference passes h_state / 2, dynamic_programming.py:34).
 * state_grid_uniform != 0: the caller asserts that the state grid is equally spaced (to ~1e-14) with spacing
 * state_grid_step = (x_{Ns-1} - x_0) / (Ns - 1) (a host value: the recurrence constants derived from it travel as a
 * kernel parameter); cells no wider than 0.2 sd are then integrated by Gauss-Legendre quadrature with a density
 * recurrence along s' (|error| < 1e-13) instead of two erf/erfc evaluations per cell.  0 always takes the erf/erfc path.
 */
int rlsde_tables(const double* state_grid_dev, int64_t Ns, const double* action_grid_dev, int64_t Na,
                 const uint8_t* in_ts_dev, int64_t n_ts, double alpha, double sigma, double dt, double h_half,
                 double lb, double rb, int64_t sprime_begin, int64_t sprime_end, double* P_dev, double* R_dev,
                 int32_t state_grid_uniform, double state_grid_step, void* stream);

/* column sums over s' of a P slab, accumulated into colsum_dev[Ns*Na] (check_p_tensor, tabular_dp_tables.py:15-17) */
int rlsde_tables_colsum(const double* P_dev, int64_t n_sprime, int64_t Ns, int64_t Na, double* colsum_dev,
                        void* stream);

/*
 * Bellman sweep over a device-resident transition tensor (SURVEY 8f-1; the contraction inside q_table_update_vect
 * tabular_dp_qvalue_iteration.py:35-43, v_table_update_vect tabular_dp_value_iteration.py:41-52 and policy_update_vect
 * tabular_dp_policy_iteration.py:37-49):
 *   values[s, a] = R[s, a] + (1 - in_ts[s]) * gamma * sum_{s'} P[s', s, a] * v[s']
 * P_dev: double[Ns][Ns][Na] as written by rlsde_tables; v_dev: double[Ns]; values_dev: double[Ns][Na].
 * scratch_dev: rlsde_dp_scratch_bytes(Ns, Na) bytes.  HBM-read bound: 8 Ns^2 Na bytes per sweep.
 */
size_t rlsde_dp_scratch_bytes(int64_t Ns, int64_t Na);
int rlsde_dp_sweep(const double* P_dev, int64_t Ns, int64_t Na, const double* R_dev, const uint8_t* in_ts_dev,
                   const double* v_dev, double gamma, double* values_dev, void* scratch_dev, size_t scratch_bytes,
                   void* stream);
/*
 * The same sweep without the tensor: P[s', s, a] is generated inside the sweep, exactly as rlsde_tables defines it
 * (same arguments, same choice between the erf/erfc and the quadrature path), and contracted at once.  Memory is
 * O(Ns Na) whatever the grid, so grids whose tensor (8 Ns^2 Na bytes) does not fit on the device can be swept.  Cells
 * lying entirely beyond 9 sd of a column's mean are skipped: at most 2^-60 of each column's mass.  Deterministic and
 * bitwise repeatable; bound by the FP64 pipe, not by memory.  Columns of target-set states are R[s, a].
 * state_grid_dev: double[Ns], increasing; action_grid_dev: double[Na]; in_ts_dev: uint8[Ns]; R_dev, values_dev:
 * double[Ns][Na]; v_dev: double[Ns].
 * Refused before any device work (RLSDE_ERR_INVALID_ARG): a NULL pointer, Ns < 1 or Na < 1, sigma, dt or h_half not
 * positive, state_grid_uniform != 0 with state_grid_step not positive.
 */
int rlsde_dp_sweep_implicit(const double* state_grid_dev, int64_t Ns, const double* action_grid_dev, int64_t Na,
                            const uint8_t* in_ts_dev, double alpha, double sigma, double dt, double h_half,
                            int32_t state_grid_uniform, double state_grid_step, const double* R_dev, const double* v_dev,
                            double gamma, double* values_dev, void* stream);
/* vmax[s] = max_a values[s, a] and argmax[s] = first maximiser (np.max / np.argmax, axis 1); either output may be NULL */
int rlsde_dp_rowmax(const double* values_dev, int64_t Ns, int64_t Na, double* vmax_dev, int64_t* argmax_dev, void* stream);

/* reward_type for rlsde_env_step */
#define RLSDE_REWARD_STATE_ACTION 0            /* done and r on the current state   environments.py:152-155 */
#define RLSDE_REWARD_STATE_ACTION_NEXT_STATE 1 /* done on the next state            environments.py:157-160 */

/*
 * One Euler-Maruyama pass for K states (env.step / env.step_torch).  state/next_state/reward are
 * float* (double* with RLSDE_F_STATE_F64: numpy promotion rules, SURVEY App. A-5).  dbt_in_dev == NULL
 * draws the increments from Philox(seed, traj_offset + k, pass_index); they are returned in dbt_out_dev.
 */
int rlsde_env_step(const rlsde_env* env, int64_t K, const void* state_dev, const float* action_dev,
                   const float* dbt_in_dev, uint64_t seed, int64_t traj_offset, int64_t pass_index,
                   uint32_t flags, int32_t reward_type, void* next_state_dev, void* reward_dev,
                   uint8_t* done_dev, float* dbt_out_dev, void* stream);

/* increments dB[p][k][i] = sqrt(dt) * N(0,1) for passes [pass_begin, pass_begin+n_pass), trajectories
   [traj_offset, traj_offset+K): exactly what the rollout kernels generate in-kernel for that seed */
int rlsde_noise_fill(uint64_t seed, int64_t traj_offset, int64_t K, int32_t d, int64_t pass_begin, int64_t n_pass,
                     double dt, float* out_dev, void* stream);

/* host only: the bounds behind the clamp-free precise tanh of the d = 1, hidden width 32 tensor-core forward policy, from
   its folded, pre-scaled image (params_host: state_dict order).  out[0]: an upper bound on every layer-2 pre-activation
   (the clamp-free layer 2 is used when it is <= 30); out[1]: every layer-1 pre-activation is <= 30 while |x| <= out[1]
   (negative: for no x) */
int rlsde_fwd_mma_clamp_bounds(const float* params_host, double* out);

#ifdef __cplusplus
}
#endif
#endif /* RLSDE_H_ */
