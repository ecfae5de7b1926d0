// C ABI of librlsde_b200.so (declared in include/rlsde.h): argument checking, host-side
// precomputation of the environment constants the way torch / numpy round them, dispatch on the
// policy shape, and stream-ordered launches.  No torch types, no exceptions, no environment variables, no
// global mutable state except the thread-local text of the last CUDA error and the launch counter.
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../../include/rlsde.h"
#include "aux_kernels.cuh"
#include "rollout_bwd.cuh"
#include "rollout_bwd_mma.cuh"
#include "rollout_warp.cuh"
#include "rollout_wide.cuh"
#include "rollout_umma_bwd.cuh"
#include "rollout_umma.cuh"

namespace rlsde {

static thread_local char g_last_cuda_error[256] = "";
static std::atomic<long long> g_kernel_launches{0};
void note_kernel_launches(int n) { g_kernel_launches.fetch_add(n, std::memory_order_relaxed); }

// Second stream for the reverse pass: the warp-per-trajectory kernel walks the longest trajectories of a large batch
// while the thread-per-trajectory kernel works on the bulk (fork / join with events, so the caller's stream stays the
// only one it has to think about; the pattern is legal inside CUDA graph capture).  One per host thread, created on first
// use, never destroyed: the one piece of state the library keeps besides the last-error text.
struct AuxStream {
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
  int device = -1;
  bool get() {
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return false;
    if (stream != nullptr && dev == device) return true;
    if (stream != nullptr) { cudaStreamDestroy(stream); cudaEventDestroy(fork); cudaEventDestroy(join); stream = nullptr; }
    if (cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking) != cudaSuccess) { stream = nullptr; return false; }
    if (cudaEventCreateWithFlags(&fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&join, cudaEventDisableTiming) != cudaSuccess) { cudaStreamDestroy(stream); stream = nullptr; return false; }
    device = dev;
    return true;
  }
};
static thread_local AuxStream g_aux;

static int cuda_fail(cudaError_t e, const char* where) {
  snprintf(g_last_cuda_error, sizeof(g_last_cuda_error), "%s: %s", where, cudaGetErrorString(e));
  return RLSDE_ERR_CUDA;
}

// The policy shapes (d, H) with compiled fused kernels, the one list: with_shape calls f(Shape<D, H>{}) for a compiled shape
// and returns RLSDE_ERR_UNSUPPORTED for any other.  Hidden width 32: the fully unrolled register / constant-bank kernels
// (rollout_fwd.cuh, rollout_bwd*.cuh, rollout_warp.cuh).  Hidden widths 64 / 128 / 256 (the reference's reinforce()
// default is 256): the tile kernels of rollout_wide.cuh, for the state dimensions the reference has environments for.
// The predicates say which kernel families a shape has; the callers test them with if constexpr, so that no launcher is
// referenced for a shape that has none.
template <int D_, int H_>
struct Shape {
  static constexpr int D = D_, H = H_;
  static constexpr bool narrow = H == 32;          // K1, K1w, K2m, K2w and the H = 32 tcgen05 forward (K1u)
  static constexpr bool wide = H >= 64;            // K1x, K2x
  static constexpr bool umma_fwd_wide = H >= 64;   // the tcgen05 forward at H >= 64 (K1u)
  static constexpr bool umma_bwd = H >= 128;       // the tcgen05 reverse pass (K2u)
};

template <class F>
static int with_shape(int d, int H, F&& f) {
#define X(D_, H_) \
  if (d == D_ && H == H_) return f(Shape<D_, H_>{});
  X(1, 32) X(2, 32) X(3, 32) X(4, 32) X(10, 32) X(1, 64) X(1, 128) X(1, 256) X(2, 64) X(2, 128) X(2, 256)
#undef X
  return RLSDE_ERR_UNSUPPORTED;
}

// smallest batch the tcgen05 tile kernels take automatically.  They advance 128-trajectory tiles at ~13 us (forward) /
// ~23 us (reverse) per pass at H = 256 whatever the batch, the CUDA-core tile kernels 16-trajectory tiles at ~15 / ~40 us:
// measured at H = 256, K = 1 000: forward 13.2 against 14.9 ms, reverse 34.9 against 61.8 ms (K = 4 000: 13.2 / 22.4 and 35.7 /
// 68.4).  At H = 128 the CUDA-core kernels are as fast up to a few thousand trajectories (K = 1 000: 4.7 against 6.3 ms).
static long long umma_min_k(int H, int sm) { return H >= 256 ? 4 * UMMA_M : (long long)sm * UMMA_M / 2; }

static bool shape_supported(int d, int H, int n_hidden) {
  return n_hidden == 2 && with_shape(d, H, [](auto) { return RLSDE_OK; }) == RLSDE_OK;
}

// kernel family for a call: latency kernels (warp per trajectory) for small batches, throughput kernels otherwise
static bool use_warp_kernels(const FwdArgs& A, int H, int sm_count, bool needs_all_states) {
  if (H != WARP_H) return false;
  if (needs_all_states && A.ckpt_every != 1) return false;
  if (A.flags & RLSDE_F_KERNEL_THREAD) return false;
  if (A.flags & RLSDE_F_KERNEL_WARP) return true;
  return A.K <= warp_path_max_k(sm_count);
}

static int device_sm_count(int* sm_count) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) { cuda_fail(e, "cudaGetDevice"); return RLSDE_ERR_NO_DEVICE; }
  int n = 0;
  e = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  if (e != cudaSuccess) { cuda_fail(e, "cudaDeviceGetAttribute"); return RLSDE_ERR_NO_DEVICE; }
  *sm_count = n;
  return RLSDE_OK;
}

static int check_env_mlp(const rlsde_env* env, const rlsde_mlp* mlp) {
  if (!env || !mlp) return RLSDE_ERR_INVALID_ARG;
  if (env->d < 1 || env->d > RLSDE_MAX_D) return RLSDE_ERR_INVALID_ARG;
  if (mlp->d_in != env->d || mlp->d_out != env->d) return RLSDE_ERR_INVALID_ARG;
  if (!(env->dt > 0) || !(env->sigma > 0)) return RLSDE_ERR_INVALID_ARG;
  if (env->hit_rule != RLSDE_HIT_ALL_GE_LB && env->hit_rule != RLSDE_HIT_X0_IN_LB_RB) return RLSDE_ERR_INVALID_ARG;
  if (!shape_supported(env->d, mlp->d_hidden, mlp->n_hidden)) return RLSDE_ERR_UNSUPPORTED;
  return RLSDE_OK;
}

// the environment constants FwdArgs and StepArgs share, rounded the way the reference rounds them: torch multiplies the
// f32 state by the python scalar 4*alpha cast to f32; sigma_tensor / dt_tensor are float32 (environments.py:19,23).  The
// caller has zeroed A.
template <class Args>
static void fill_env_consts(const rlsde_env* env, Args& A) {
  for (int i = 0; i < env->d; ++i) { A.c4a_d[i] = 4.0 * env->alpha[i]; A.c4a_f[i] = (float)(4.0 * env->alpha[i]); }
  A.sigma_d = env->sigma; A.sigma_f = (float)env->sigma;
  A.dt_d = env->dt; A.dt_f = (float)env->dt;
  A.lb_d = env->lb; A.rb_d = env->rb; A.lb_f = (float)env->lb; A.rb_f = (float)env->rb;
  A.noise_scale2 = (float)(-2.0 * env->dt * 0.6931471805599453);
  A.hit_rule = env->hit_rule;
}

// passes an undetected trajectory executes: the budget, or the injected noise if that is shorter
static long long passes_run(const FwdArgs& A) {
  return (A.flags & RLSDE_F_NOISE_INJECTED) && A.noise_steps < A.n_steps_lim ? A.noise_steps : A.n_steps_lim;
}

// ragged: the checkpoints go to the ragged store (rlsde_rollout_fwd_ragged / rlsde_rollout_bwd_ragged), whose size the
// caller has fitted to the trajectories: cfg->ckpt_stride is not read
static int fill_cfg(const rlsde_rollout_cfg* cfg, FwdArgs& A, bool ragged) {
  if (!cfg || cfg->K < 0 || cfg->n_steps_lim < 1 || cfg->n_steps_lim > 2000000000LL) return RLSDE_ERR_INVALID_ARG;
  if (cfg->traj_offset < 0) return RLSDE_ERR_INVALID_ARG;
  if ((cfg->flags & RLSDE_F_NOISE_INJECTED) && cfg->noise_steps < 1) return RLSDE_ERR_INVALID_ARG;
  // injected noise is indexed [pass][traj_offset + k] with row stride K_global: the shard must lie inside the global batch
  if ((cfg->flags & RLSDE_F_NOISE_INJECTED) && cfg->traj_offset + cfg->K > (cfg->K_global > 0 ? cfg->K_global : cfg->K))
    return RLSDE_ERR_INVALID_ARG;
  A.K = cfg->K; A.traj_offset = cfg->traj_offset;
  A.K_global = cfg->K_global > 0 ? cfg->K_global : cfg->K;
  A.seed = cfg->seed; A.n_steps_lim = cfg->n_steps_lim; A.noise_steps = cfg->noise_steps;
  A.flags = cfg->flags; A.ckpt_every = cfg->ckpt_every > 0 ? cfg->ckpt_every : 1; A.ckpt_stride = cfg->ckpt_stride;
  if ((cfg->flags & RLSDE_F_STORE_PATH) && !ragged) {
    // the kernels write path[(traj * ckpt_stride + k / ckpt_every) * d] for every pass k they execute
    if (cfg->ckpt_every < 1 || cfg->ckpt_stride < (passes_run(A) + cfg->ckpt_every - 1) / cfg->ckpt_every) return RLSDE_ERR_INVALID_ARG;
  }
  A.ckpt_log2 = -1;
  for (int b = 0; b < 31; ++b)
    if (A.ckpt_every == (1 << b)) A.ckpt_log2 = b;
  A.n_grid = cfg->n_grid; A.grid_lo = cfg->grid_lo; A.grid_hi = cfg->grid_hi; A.grid_h = cfg->grid_h;
  A.blocks_per_sm_cap = cfg->fwd_blocks_per_sm > 0 ? cfg->fwd_blocks_per_sm : 0;
  if (cfg->fwd_policy < 0 || cfg->fwd_policy > 2) return RLSDE_ERR_INVALID_ARG;
  return RLSDE_OK;
}

// the arguments every rollout and reverse pass starts from: the environment and the cfg; the ragged store implies
// RLSDE_F_STORE_PATH
static int make_args(const rlsde_env* env, const rlsde_rollout_cfg* cfg, FwdArgs& A, bool ragged = false) {
  memset(&A, 0, sizeof(A));
  fill_env_consts(env, A);
  for (int i = 0; i < env->d; ++i) {
    A.x0_d[i] = (double)(float)env->x0[i];     // state_init is float32 (environments.py:30)
    A.x0_f[i] = (float)env->x0[i];
  }
  const int rc = fill_cfg(cfg, A, ragged);
  if (rc == RLSDE_OK && ragged) A.flags |= RLSDE_F_STORE_PATH;
  return rc;
}

// Workspace layout, in order: counters (u64: items claimed, records queued, trajectories completed); statistics partials;
// device copy of the packed policy (device-resident training step); reverse-pass partials; device image of a wide policy
// (rollout_wide.cuh); float16 hi / lo image of W2 for the tcgen05 kernels (H = 256).  Then, to the end of the buffer, the
// ring of continuation records of the time-sliced forward rollout (one record per trajectory + one per lane:
// rlsde_workspace_bytes(K) sizes it for the largest record), or the tcgen05 reverse pass's exchange ring and float64
// partials (rlsde_workspace_bytes_bwd).
constexpr size_t WS_COUNTER_BYTES = 1024;
constexpr size_t WS_STATS_BYTES = (size_t)STATS_BLOCKS * RLSDE_NSTATS * sizeof(double);
constexpr size_t WS_POLICY_BYTES = 16384;
constexpr size_t WS_WIDE_BYTES = (WIDE_PARAM_BYTES_MAX + 255) & ~(size_t)255;
constexpr size_t WS_UMMA_BYTES = 256 * 256 * 4;
constexpr long long WS_MAX_LANES = 148LL * 16 * 128;                          // lanes of the largest forward grid
constexpr size_t WS_CONT_REC_BYTES = 16 + 8 * (RLSDE_MAX_D + 3);              // >= sizeof(ContRec<D, F64>) for every D
static_assert(sizeof(MlpConst<RLSDE_MAX_D, WARP_H>) <= WS_POLICY_BYTES, "raise WS_POLICY_BYTES");

struct Workspace {
  static constexpr size_t o_stats = WS_COUNTER_BYTES;
  static constexpr size_t o_policy = o_stats + WS_STATS_BYTES;     // also the least a forward rollout takes
  static constexpr size_t o_bwd = o_policy + WS_POLICY_BYTES;
  static size_t o_wide() { return o_bwd + bwd_workspace_bytes(); }
  static size_t o_umma() { return o_wide() + WS_WIDE_BYTES; }
  static size_t fixed_bytes() { return o_umma() + WS_UMMA_BYTES; }

  char* base;
  unsigned long long* counters() const { return (unsigned long long*)base; }
  double* stats() const { return (double*)(base + o_stats); }
  void* policy() const { return base + o_policy; }
  float* bwd_partial() const { return (float*)(base + o_bwd); }
  float* wide_params() const { return (float*)(base + o_wide()); }
  uint8_t* umma_image() const { return (uint8_t*)base + o_umma(); }
  uint8_t* tail() const { return (uint8_t*)base + fixed_bytes(); }
};

static int launch_status(int lrc, const char* what) { return lrc != 0 ? cuda_fail((cudaError_t)lrc, what) : RLSDE_OK; }

// the device's SM count, and the work counters cleared on the stream
static int begin_launch(const Workspace& ws, cudaStream_t stream, int& sm) {
  const int rc = device_sm_count(&sm);
  if (rc != RLSDE_OK) return rc;
  const cudaError_t e = cudaMemsetAsync(ws.base, 0, WS_COUNTER_BYTES, stream);
  return e != cudaSuccess ? cuda_fail(e, "cudaMemsetAsync(workspace)") : RLSDE_OK;
}

// the statistics record of a rollout (stats_dev may be null: none)
static int reduce_stats(const FwdArgs& A, double* stats_dev, const Workspace& ws, cudaStream_t stream) {
  if (!stats_dev) return RLSDE_OK;
  return launch_status(launch_reduce_stats(A.K, passes_run(A), (A.flags & RLSDE_F_STATE_F64) != 0, A.G, A.S, A.T, A.l2, A.logw,
                                           stats_dev, ws.stats(), stream), "reduce_stats launch");
}

}  // namespace rlsde

using namespace rlsde;

extern "C" {

int rlsde_version(void) { return RLSDE_VERSION; }

const char* rlsde_strerror(int status) {
  switch (status) {
    case RLSDE_OK: return "ok";
    case RLSDE_ERR_INVALID_ARG: return "invalid argument";
    case RLSDE_ERR_UNSUPPORTED: return "no fused kernel compiled for this policy shape (d, hidden width, depth)";
    case RLSDE_ERR_CUDA: return "CUDA error (see rlsde_last_cuda_error)";
    case RLSDE_ERR_NO_DEVICE: return "no usable CUDA device";
    case RLSDE_ERR_WORKSPACE: return "workspace too small (see rlsde_workspace_bytes)";
    default: return "unknown status";
  }
}

const char* rlsde_last_cuda_error(void) { return g_last_cuda_error; }

long long rlsde_launch_count(void) { return g_kernel_launches.load(std::memory_order_relaxed); }

int rlsde_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) { cuda_fail(e, "cudaGetDevice"); return RLSDE_ERR_NO_DEVICE; }
  int n = 0, ma = 0, mi = 0;
  if ((e = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess ||
      (e = cudaDeviceGetAttribute(&ma, cudaDevAttrComputeCapabilityMajor, dev)) != cudaSuccess ||
      (e = cudaDeviceGetAttribute(&mi, cudaDevAttrComputeCapabilityMinor, dev)) != cudaSuccess) {
    cuda_fail(e, "cudaDeviceGetAttribute");
    return RLSDE_ERR_NO_DEVICE;
  }
  if (sm_count) *sm_count = n;
  if (cc_major) *cc_major = ma;
  if (cc_minor) *cc_minor = mi;
  return RLSDE_OK;
}

int rlsde_supported(int32_t d, int32_t d_hidden, int32_t n_hidden) { return shape_supported(d, d_hidden, n_hidden) ? 1 : 0; }

int64_t rlsde_param_count(const rlsde_mlp* mlp) {
  if (!mlp) return -1;
  const int64_t d = mlp->d_in, H = mlp->d_hidden, o = mlp->d_out;
  return d * H + H + (int64_t)(mlp->n_hidden - 1) * (H * H + H) + H * o + o;
}

size_t rlsde_workspace_bytes(int64_t K) {
  const long long k = K > 0 ? K : 0;
  long long cap = 1;
  while (cap < k + WS_MAX_LANES) cap <<= 1;             // the ring's capacity is a power of two
  return Workspace::fixed_bytes() + (size_t)cap * WS_CONT_REC_BYTES;
}

// the reverse pass of a wide policy on the tensor cores (rollout_umma_bwd.cuh) keeps its scratch behind the fixed part
size_t rlsde_workspace_bytes_bwd(int64_t K, int32_t d, int32_t d_hidden) {
  size_t n = rlsde_workspace_bytes(K);
  with_shape(d, d_hidden, [&](auto s) {
    using S = decltype(s);
    int sm = 0;
    if constexpr (S::umma_bwd) {
      if (device_sm_count(&sm) == RLSDE_OK) {
        const size_t need = Workspace::fixed_bytes() + bwd_umma_scratch_bytes<S::D, S::H>(sm);
        if (need > n) n = need;
      }
    }
    return RLSDE_OK;
  });
  return n;
}

// transition-stream outputs of a forward rollout (all null = none)
struct TransitionOut {
  const long long* base;
  float* state;
  float* action;
  float* reward;
  float* next_state;
  unsigned char* done;
};

// RAGGED: rlsde_rollout_fwd_ragged (checkpoints into the ragged store at path_base; no transition stream)
extern "C++" {
template <bool RAGGED>
static int rollout_fwd_impl(const rlsde_env* env, const rlsde_mlp* mlp, const float* params_host,
                            const rlsde_rollout_cfg* cfg, const float* noise_dev, const float* policy_opt_dev,
                            void* G_dev, void* S_dev, int32_t* T_dev, void* l2_dev, void* logw_dev, float* path_dev,
                            double* stats_dev, const TransitionOut& tr, const long long* path_base, void* workspace_dev,
                            size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  int rc = check_env_mlp(env, mlp);
  if (rc != RLSDE_OK) return rc;
  if (!params_host || !G_dev || !S_dev || !T_dev || !workspace_dev) return RLSDE_ERR_INVALID_ARG;
  if (workspace_bytes < Workspace::o_policy) return RLSDE_ERR_WORKSPACE;
  FwdArgs A;
  if ((rc = make_args(env, cfg, A, RAGGED)) != RLSDE_OK) return rc;
  if (RAGGED) {
    // the store exists for the reverse pass, so it takes that pass's conditions: a float32 state, no projection (below)
    // and at most BWD_MAX_SEG passes per checkpoint
    if (!path_base || !path_dev || tr.base) return RLSDE_ERR_INVALID_ARG;
    if (cfg->ckpt_every < 1 || cfg->ckpt_every > BWD_MAX_SEG) return RLSDE_ERR_INVALID_ARG;
    if (A.flags & RLSDE_F_HIT_BRIDGE) return RLSDE_ERR_INVALID_ARG;
    if (A.flags & RLSDE_F_STATE_F64) return RLSDE_ERR_UNSUPPORTED;
  }
  if ((A.flags & RLSDE_F_NOISE_INJECTED) && !noise_dev) return RLSDE_ERR_INVALID_ARG;
  if ((A.flags & RLSDE_F_STORE_PATH) && !path_dev) return RLSDE_ERR_INVALID_ARG;
  if (policy_opt_dev && (cfg->n_grid < 1 || !(cfg->grid_h > 0) || env->d != 1)) return RLSDE_ERR_INVALID_ARG;
  if (A.flags & RLSDE_F_HIT_BRIDGE) {
    // the reverse pass recomputes states from checkpoints and knows nothing of the projection; the transition stream
    // records the unprojected pass
    if ((A.flags & RLSDE_F_STORE_PATH) || tr.base) return RLSDE_ERR_INVALID_ARG;
    if (env->d != 1) return RLSDE_ERR_UNSUPPORTED;        // the target all_i x_i >= lb is an orthant: no closed form
  }
  A.noise = noise_dev; A.policy_opt = policy_opt_dev;
  A.G = G_dev; A.S = S_dev; A.T = T_dev; A.l2 = l2_dev; A.logw = logw_dev; A.path = path_dev;
  A.tr_base = tr.base; A.tr_state = tr.state; A.tr_action = tr.action; A.tr_reward = tr.reward;
  A.tr_next = tr.next_state; A.tr_done = tr.done;
  if (RAGGED) A.path_base = path_base;                  // shares tr_base's field: the ragged kernels have no stream
  if (tr.base) A.flags = (A.flags & ~RLSDE_F_KERNEL_WARP) | RLSDE_F_KERNEL_THREAD;   // the stream lives in the throughput kernel
  const Workspace ws{(char*)workspace_dev};
  A.counter = ws.counters();
  A.q_ctrl = ws.counters();
  if (workspace_bytes > Workspace::fixed_bytes()) {     // ring of continuation records: whatever lies behind the fixed part
    A.q_ring = ws.tail();
    A.q_cap = (long long)(workspace_bytes - Workspace::fixed_bytes());   // bytes; the launcher turns it into a record count
  }
  if (A.K == 0) return RLSDE_OK;
  int sm = 0;
  if ((rc = begin_launch(ws, stream, sm)) != RLSDE_OK) return rc;
  rc = with_shape(env->d, mlp->d_hidden, [&](auto shape) -> int {
    using S = decltype(shape);
    if constexpr (S::wide) {
      // wide policies: one kernel family (tiles of trajectories per block), no transition stream, no time slices
      if (tr.base) return RLSDE_ERR_UNSUPPORTED;
      if (workspace_bytes < Workspace::fixed_bytes()) return RLSDE_ERR_WORKSPACE;
      // hidden width 64 / 128 / 256 with enough trajectories (umma_min_k: four 128-row tiles at H = 256, half the SMs
      // below): the tcgen05 kernel (rollout_umma.cuh; weights resident at width 64, streamed above); otherwise the
      // CUDA-core tile kernel (rollout_wide.cuh).  cfg.wide_kernel: 1 forces tcgen05, 2 forces the CUDA-core kernel.
      if constexpr (S::umma_fwd_wide) {
        if (cfg->wide_kernel == 1 || (cfg->wide_kernel == 0 && A.K >= umma_min_k(S::H, sm)))
          return launch_status(launch_rollout_fwd_umma<S::D, S::H, RAGGED>(params_host, ws.wide_params(), ws.umma_image(), A, sm,
                                                                           stream), "rollout_fwd (wide) launch");
      }
      return launch_status(launch_rollout_fwd_wide<S::D, S::H, RAGGED>(params_host, ws.wide_params(), A, sm, stream),
                           "rollout_fwd (wide) launch");
    } else {
      const bool warp_path = use_warp_kernels(A, S::H, sm, (A.flags & RLSDE_F_STORE_PATH) != 0);
      // ---- policy arithmetic of the thread-per-trajectory kernel and of the kernel that continues its tail (mlp_mma.cuh
      // or FFMA2).  A function of (d, H, cfg.fwd_policy) only: the replay sampler launches it twice, with and without the
      // transition stream, and needs the same hit passes from both launches.
      if (cfg->fwd_policy == 1 && !fwd_mma_shape(S::D, S::H)) return RLSDE_ERR_UNSUPPORTED;
      A.policy_mma = fwd_mma_shape(S::D, S::H) && cfg->fwd_policy != 2 ? 1 : 0;
      // ---- hidden width 32 on the tensor cores (rollout_umma.cuh with resident weights: tiles of 128 trajectories, one
      // thread per trajectory, lane refill).  The per-pass work of a warp drops from ~1 290 to ~860 instructions; like K1
      // it ends up bound by the MUFU pipe (71 % busy with the two-MUFU tanh: profiles/r02/ncu_rollout_fwd_umma_h32_v1.txt).
      // Measured at 1e6 trajectories, budget 1 000 passes (tools/bench_fwd_kernels.py): d = 1 precise tanh 27.5 ms against
      // K1's 25.1 ms, fast tanh 20.6 against 21.5; d = 2: 54.5 % of the FP32 roofline against 52 %; d = 4: 58.1 % against
      // 53.4 %; d = 10: 50.9 % against 44.9 %.  It has no breadth-first schedule, so its launch ends with a tail of
      // (longest trajectory) x (~1 us per pass).  At d = 1 the thread-per-trajectory kernel with its 32 x 32 layer on
      // mma.sync (mlp_mma.cuh) beats it in both tanh modes: 21.1 / 15.4 ms against 27.4 / 20.6 ms (profiles/r03).
      // Automatic where it wins: d >= 2, large batches, a bounded pass budget -- and never when the caller pins a kernel
      // family, a schedule or the policy arithmetic of the thread-per-trajectory kernel.
      const long long passes = passes_run(A);
      const bool forced = (A.flags & RLSDE_F_KERNEL_TENSOR) != 0;
      const bool pinned = (A.flags & (RLSDE_F_KERNEL_THREAD | RLSDE_F_KERNEL_WARP)) != 0 || cfg->fwd_quantum != 0 ||
                          cfg->fwd_handoff != 0 || cfg->fwd_policy != 0;
      const bool automatic = !pinned && !warp_path && A.K >= (long long)sm * UMMA_M * 2 && passes <= 4096 && S::D >= 2;
      if (!tr.base && (forced || automatic)) {
        if (workspace_bytes < Workspace::fixed_bytes()) return RLSDE_ERR_WORKSPACE;
        return launch_status(launch_rollout_fwd_umma<S::D, S::H, RAGGED>(params_host, ws.wide_params(), ws.umma_image(), A, sm,
                                                                         stream), "rollout_fwd (tensor) launch");
      }
      // ---- schedule of the thread-per-trajectory kernel (rollout_fwd.cuh).  Two ways to deal with the tail of a launch:
      //  * time slices (FIFO of continuation records, breadth-first): right when many trajectories run into the pass
      //    budget -- the bench workload, 24 % of them: 24.5 ms against 27.8 ms; passes per slice = 1/128 of the budget,
      //    between 8 and 128 (24.3 / 24.5 / 24.9 / 25.4 / 27.8 ms at 4 / 8 / 16 / 32 / 128) -- but 3-13 % slower in
      //    steady state;
      //  * run to completion and hand the last live trajectories to the warp-per-trajectory kernel (RESUME mode, K1's
      //    arithmetic, ~5x faster on a lone trajectory): right when the tail is a few very long trajectories (metastable
      //    configuration 5.68 -> 4.14 s, training forward 21.5 -> 13.9 ms, d = 2 test rollouts 16.6 -> 14.5 ms).
      // Which one applies depends on the length distribution, which the launch only learns as it goes: it starts running
      // to completion and switches to time slices as soon as 5 % of the completed trajectories have run into the budget
      // (q_adaptive).  RLSDE_FWD_QUANTUM forces one or the other (0 = run to completion + hand-off, n = n-pass slices).
      long long quantum = passes / 128 > 128 ? 128 : (passes / 128 < 8 ? 8 : passes / 128);
      const bool can_hand_off = !tr.base;                   // the latency kernel has no transition stream
      A.q_adaptive = can_hand_off ? 1 : 0;
      if (!can_hand_off && passes > 4096) quantum = 0;
      if (cfg->fwd_quantum != 0) { quantum = cfg->fwd_quantum > 0 ? cfg->fwd_quantum : 0; A.q_adaptive = 0; }
      if (quantum > 0) {                                    // a power of two, at least one noise block (4 passes)
        long long q2 = 4;
        while (q2 < quantum && q2 < (1LL << 30)) q2 <<= 1;
        quantum = q2;
      }
      A.q_quantum = (int)quantum;
      A.q_handoff = (can_hand_off && (quantum == 0 || A.q_adaptive)) ? 4LL * warp_path_max_k(sm) : 0;
      if (cfg->fwd_handoff != 0) {
        if (A.q_handoff > 0) A.q_handoff = cfg->fwd_handoff;
        if (A.q_handoff <= 0) { A.q_handoff = 0; A.q_adaptive = 0; }
      }
      const int lrc = warp_path ? launch_rollout_fwd_warp<S::D, RAGGED>(params_host, nullptr, A, sm, stream)
                                : launch_rollout_fwd<S::D, S::H, RAGGED>(params_host, A, sm, stream);
      if (lrc != 0) return cuda_fail((cudaError_t)lrc, "rollout_fwd launch");
      // the trajectories K1 left in the ring (none if it ran without one): one warp each, K1's arithmetic
      if (!warp_path && A.q_handoff > 0 && (A.q_quantum == 0 || A.q_adaptive) && A.q_ring != nullptr)
        return launch_status(launch_rollout_fwd_warp_resume<S::D, RAGGED>(params_host, A, sm, stream), "rollout_fwd resume launch");
      return RLSDE_OK;
    }
  });
  if (rc != RLSDE_OK) return rc;
  return reduce_stats(A, stats_dev, ws, stream);
}
}  // extern "C++"

int rlsde_rollout_fwd(const rlsde_env* env, const rlsde_mlp* mlp, const float* params_host,
                      const rlsde_rollout_cfg* cfg, const float* noise_dev, const float* policy_opt_dev,
                      void* G_dev, void* S_dev, int32_t* T_dev, void* l2_dev, void* logw_dev, float* path_dev,
                      double* stats_dev, void* workspace_dev, size_t workspace_bytes, void* stream_) {
  const TransitionOut none = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  return rollout_fwd_impl<false>(env, mlp, params_host, cfg, noise_dev, policy_opt_dev, G_dev, S_dev, T_dev, l2_dev, logw_dev,
                                 path_dev, stats_dev, none, nullptr, workspace_dev, workspace_bytes, stream_);
}

int rlsde_rollout_fwd_ragged(const rlsde_env* env, const rlsde_mlp* mlp, const float* params_host,
                             const rlsde_rollout_cfg* cfg, const float* noise_dev, const int64_t* path_base_dev,
                             void* G_dev, void* S_dev, int32_t* T_dev, float* path_dev, double* stats_dev,
                             void* workspace_dev, size_t workspace_bytes, void* stream_) {
  const TransitionOut none = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  return rollout_fwd_impl<true>(env, mlp, params_host, cfg, noise_dev, nullptr, G_dev, S_dev, T_dev, nullptr, nullptr, path_dev,
                                stats_dev, none, (const long long*)path_base_dev, workspace_dev, workspace_bytes, stream_);
}

int rlsde_rollout_fwd_table(const rlsde_env* env, const float* u_table_dev, const rlsde_rollout_cfg* cfg,
                            const float* noise_dev, const float* policy_opt_dev, void* G_dev, void* S_dev, int32_t* T_dev,
                            void* l2_dev, void* logw_dev, double* stats_dev, void* workspace_dev, size_t workspace_bytes,
                            void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!env || !cfg) return RLSDE_ERR_INVALID_ARG;
  if (env->d != 1) return RLSDE_ERR_UNSUPPORTED;                 // tables, DP sweeps and the HJB solution are 1-D
  if (!(env->dt > 0) || !(env->sigma > 0)) return RLSDE_ERR_INVALID_ARG;
  if (env->hit_rule != RLSDE_HIT_ALL_GE_LB && env->hit_rule != RLSDE_HIT_X0_IN_LB_RB) return RLSDE_ERR_INVALID_ARG;
  if (!u_table_dev || cfg->n_grid < 1 || !(cfg->grid_h > 0)) return RLSDE_ERR_INVALID_ARG;
  if (!G_dev || !S_dev || !T_dev || !workspace_dev) return RLSDE_ERR_INVALID_ARG;
  if (workspace_bytes < Workspace::o_policy) return RLSDE_ERR_WORKSPACE;
  FwdArgs A;
  int rc = make_args(env, cfg, A);
  if (rc != RLSDE_OK) return rc;
  if (A.flags & RLSDE_F_STORE_PATH) return RLSDE_ERR_INVALID_ARG;                 // no reverse pass through a table
  if ((A.flags & RLSDE_F_NOISE_INJECTED) && !noise_dev) return RLSDE_ERR_INVALID_ARG;
  // kernel-family and tanh flags do not apply
  A.flags &= RLSDE_F_NOISE_INJECTED | RLSDE_F_STOCH_INT_EXACT | RLSDE_F_STATE_F64 | RLSDE_F_HIT_BRIDGE;
  A.noise = noise_dev; A.policy_opt = policy_opt_dev;
  A.G = G_dev; A.S = S_dev; A.T = T_dev; A.l2 = l2_dev; A.logw = logw_dev;
  const Workspace ws{(char*)workspace_dev};
  A.counter = ws.counters();
  if (A.K == 0) return RLSDE_OK;
  int sm = 0;
  if ((rc = begin_launch(ws, stream, sm)) != RLSDE_OK) return rc;
  if ((rc = launch_status(launch_rollout_fwd_table(u_table_dev, A, sm, stream), "rollout_fwd_table launch")) != RLSDE_OK) return rc;
  return reduce_stats(A, stats_dev, ws, stream);
}

int rlsde_rollout_transitions(const rlsde_env* env, const rlsde_mlp* mlp, const float* params_host,
                              const rlsde_rollout_cfg* cfg, const float* noise_dev, const int64_t* slot_base_dev,
                              float* states_dev, float* actions_dev, float* rewards_dev, float* next_states_dev,
                              uint8_t* done_dev, void* G_dev, void* S_dev, int32_t* T_dev, double* stats_dev,
                              void* workspace_dev, size_t workspace_bytes, void* stream_) {
  if (!slot_base_dev || !states_dev || !actions_dev || !rewards_dev || !next_states_dev || !done_dev) return RLSDE_ERR_INVALID_ARG;
  if (cfg && (cfg->flags & RLSDE_F_STORE_PATH)) return RLSDE_ERR_INVALID_ARG;
  const TransitionOut tr = {(const long long*)slot_base_dev, states_dev, actions_dev, rewards_dev, next_states_dev, done_dev};
  return rollout_fwd_impl<false>(env, mlp, params_host, cfg, noise_dev, nullptr, G_dev, S_dev, T_dev, nullptr, nullptr, nullptr,
                                 stats_dev, tr, nullptr, workspace_dev, workspace_bytes, stream_);
}

// WEIGHTED = false: rlsde_rollout_bwd (cS_dev = G, cG_dev unused); true: rlsde_rollout_bwd_weighted.  The weighted kernels
// read cS from FwdArgs::G and cG from FwdArgs::S (rollout_bwd.cuh, the comment above em_step_f32).
// RAGGED (with WEIGHTED only): rlsde_rollout_bwd_ragged, the checkpoints come from the ragged store at path_base.
extern "C++" {
template <bool WEIGHTED, bool RAGGED = false>
static int rollout_bwd_impl(const rlsde_env* env, const rlsde_mlp* mlp, const float* params_host, const rlsde_rollout_cfg* cfg,
                            const float* noise_dev, const float* cS_dev, const float* cG_dev, const int32_t* T_dev,
                            const float* path_dev, const int64_t* order_dev, double loss_scale, float* grad_dev,
                            void* workspace_dev, size_t workspace_bytes, void* stream_, const long long* path_base = nullptr) {
  static_assert(WEIGHTED || !RAGGED, "the ragged reverse pass is the weighted one");
  cudaStream_t stream = (cudaStream_t)stream_;
  int rc = check_env_mlp(env, mlp);
  if (rc != RLSDE_OK) return rc;
  if (!params_host || !cS_dev || !T_dev || !path_dev || !grad_dev || !workspace_dev) return RLSDE_ERR_INVALID_ARG;
  if (WEIGHTED && !cG_dev) return RLSDE_ERR_INVALID_ARG;
  if (workspace_bytes < Workspace::fixed_bytes()) return RLSDE_ERR_WORKSPACE;
  FwdArgs A;
  if ((rc = make_args(env, cfg, A, RAGGED)) != RLSDE_OK) return rc;
  if (RAGGED && !path_base) return RLSDE_ERR_INVALID_ARG;
  if (A.flags & RLSDE_F_HIT_BRIDGE) return RLSDE_ERR_INVALID_ARG;   // no reverse pass through the projection
  if (A.flags & RLSDE_F_STATE_F64) return RLSDE_ERR_UNSUPPORTED;   // the reference differentiates the f32 torch path only
  if (!(A.flags & RLSDE_F_STORE_PATH)) return RLSDE_ERR_INVALID_ARG;
  if (A.ckpt_every > BWD_MAX_SEG) return RLSDE_ERR_INVALID_ARG;        // the reverse pass recomputes at most 32 passes per checkpoint
  if (cfg->bwd_kernel != 0 && cfg->bwd_kernel != 1) return RLSDE_ERR_UNSUPPORTED;   // the tensor-core kernel is the only one
  if ((A.flags & RLSDE_F_NOISE_INJECTED) && !noise_dev) return RLSDE_ERR_INVALID_ARG;
  A.noise = noise_dev;
  A.G = (void*)cS_dev; A.T = (int*)T_dev; A.path = (float*)path_dev;
  if (WEIGHTED) A.S = (void*)cG_dev;
  A.order = (const long long*)order_dev;
  if (RAGGED) A.path_base = path_base;
  const Workspace ws{(char*)workspace_dev};
  A.counter = ws.counters();
  int sm = 0;
  if ((rc = begin_launch(ws, stream, sm)) != RLSDE_OK) return rc;
  float* partial = ws.bwd_partial();
  return with_shape(env->d, mlp->d_hidden, [&](auto shape) -> int {
    using S = decltype(shape);
    if constexpr (S::wide) {
      if (A.ckpt_every != 1) return RLSDE_ERR_UNSUPPORTED;        // the wide reverse kernel reads every state from the path
      // hidden width 128 / 256 with enough trajectories (umma_min_k): the tcgen05 kernel (rollout_umma_bwd.cuh), given a
      // workspace from rlsde_workspace_bytes_bwd; cfg.wide_kernel as in the forward rollout
      if constexpr (S::umma_bwd) {
        const size_t umma_need = Workspace::fixed_bytes() + bwd_umma_scratch_bytes<S::D, S::H>(sm);
        if (cfg->wide_kernel == 1 && workspace_bytes < umma_need) return RLSDE_ERR_WORKSPACE;
        if (workspace_bytes >= umma_need && (cfg->wide_kernel == 1 || (cfg->wide_kernel == 0 && A.K >= umma_min_k(S::H, sm))))
          return launch_status(launch_rollout_bwd_umma<S::D, S::H, WEIGHTED, RAGGED>(
                                   params_host, ws.wide_params(), ws.umma_image(), A, (float)loss_scale, grad_dev, ws.tail(),
                                   workspace_bytes - Workspace::fixed_bytes(), sm, stream),
                               "rollout_bwd (tcgen05) launch");
      }
      return launch_status(launch_rollout_bwd_wide<S::D, S::H, WEIGHTED, RAGGED>(params_host, ws.wide_params(), A, (float)loss_scale,
                                                                                  grad_dev, partial, bwd_partial_main_bytes(), sm, stream),
                           "rollout_bwd (wide) launch");
    } else {
      const bool warp_path = use_warp_kernels(A, S::H, sm, true);
      // Large batches with a length-sorted order: the reverse pass of a trajectory is sequential, and a thread-per-
      // trajectory kernel walks a lone trajectory slowly (~12 us per pass for the CUDA-core kernel K2 this split was made
      // for) -- the longest few thousand trajectories, not the total work, set its run time (K = 4e5, longest 3 900 passes:
      // 47 ms for ~28 ms of throughput work).  They go to the warp-per-trajectory kernel instead (~0.5 us per pass), the bulk
      // to the tensor-core kernel; the two gradients are added in a fixed order.  The split depends on the sorted lengths
      // only, so the result is deterministic.
      long long n_long = 0;
      if (!warp_path && order_dev && A.ckpt_every == 1 && A.K > (long long)sm * 128) {
        // measured (K = 4e5, d = 1): 46.2 / 36.7 / 36.7 / 37.5 / 41.9 ms at 0 / 2 368 / 4 736 / 9 472 / 25 000 long trajectories
        n_long = A.K / 16 < warp_path_max_k(sm) ? A.K / 16 : warp_path_max_k(sm);
        if (cfg->bwd_warp_share != 0) n_long = cfg->bwd_warp_share < A.K ? cfg->bwd_warp_share : A.K;
        if (n_long < 0) n_long = 0;
      }
      FwdArgs Abulk = A;
      float* partial_aux = (float*)((char*)partial + bwd_partial_main_bytes());
      cudaEvent_t join = nullptr;
      int lrc = -1;                                         // an empty batch without long trajectories fails as a launch
      if (n_long > 0) {
        FwdArgs Along = A;
        Along.K = n_long;
        Abulk.order = A.order + n_long;
        Abulk.K = A.K - n_long;
        Abulk.grad_accumulate = 1;
        // the long trajectories run concurrently with the bulk on the second stream, and the bulk's reduction waits for
        // them; without a second stream they run first, on the caller's stream
        cudaStream_t s_long = stream;
        cudaError_t e;
        if (Abulk.K > 0 && g_aux.get()) {
          if ((e = cudaEventRecord(g_aux.fork, stream)) != cudaSuccess) return cuda_fail(e, "cudaEventRecord(fork)");
          if ((e = cudaStreamWaitEvent(g_aux.stream, g_aux.fork, 0)) != cudaSuccess) return cuda_fail(e, "cudaStreamWaitEvent(fork)");
          s_long = g_aux.stream;
        }
        lrc = launch_rollout_bwd_warp<S::D, WEIGHTED, RAGGED>(params_host, nullptr, Along, (float)loss_scale, grad_dev, partial_aux,
                                                              sm, s_long);
        if (lrc != 0) return cuda_fail((cudaError_t)lrc, "rollout_bwd (long trajectories) launch");
        if (s_long != stream) {
          if ((e = cudaEventRecord(g_aux.join, s_long)) != cudaSuccess) return cuda_fail(e, "cudaEventRecord(join)");
          join = g_aux.join;
        }
      }
      // thread-per-trajectory family, hidden width 32: the tensor-core kernel (rollout_bwd_mma.cuh; state dimensions above
      // 4: the d-sized products -- layer 1, head, dW1, dW3, dX -- run as padded 16-wide tiles on the tensor cores as well)
      if (Abulk.K > 0)
        lrc = warp_path ? launch_rollout_bwd_warp<S::D, WEIGHTED, RAGGED>(params_host, nullptr, Abulk, (float)loss_scale, grad_dev,
                                                                           partial, sm, stream)
                        : launch_rollout_bwd_mma<S::D, WEIGHTED, RAGGED>(params_host, Abulk, (float)loss_scale, grad_dev, partial,
                                                                         sm, stream, join);
      return launch_status(lrc, "rollout_bwd launch");
    }
  });
}
}  // extern "C++"

int rlsde_rollout_bwd(const rlsde_env* env, const rlsde_mlp* mlp, const float* params_host,
                      const rlsde_rollout_cfg* cfg, const float* noise_dev, const float* G_dev, const int32_t* T_dev,
                      const float* path_dev, const int64_t* order_dev, double loss_scale, float* grad_dev,
                      void* workspace_dev, size_t workspace_bytes, void* stream_) {
  return rollout_bwd_impl<false>(env, mlp, params_host, cfg, noise_dev, G_dev, nullptr, T_dev, path_dev, order_dev, loss_scale,
                                 grad_dev, workspace_dev, workspace_bytes, stream_);
}

int rlsde_rollout_bwd_weighted(const rlsde_env* env, const rlsde_mlp* mlp, const float* params_host,
                               const rlsde_rollout_cfg* cfg, const float* noise_dev, const float* coef_G_dev,
                               const float* coef_S_dev, const int32_t* T_dev, const float* path_dev, const int64_t* order_dev,
                               double loss_scale, float* grad_dev, void* workspace_dev, size_t workspace_bytes, void* stream_) {
  return rollout_bwd_impl<true>(env, mlp, params_host, cfg, noise_dev, coef_S_dev, coef_G_dev, T_dev, path_dev, order_dev, loss_scale,
                                grad_dev, workspace_dev, workspace_bytes, stream_);
}

int rlsde_rollout_bwd_ragged(const rlsde_env* env, const rlsde_mlp* mlp, const float* params_host,
                             const rlsde_rollout_cfg* cfg, const float* noise_dev, const float* coef_G_dev,
                             const float* coef_S_dev, const int32_t* T_dev, const int64_t* path_base_dev, const float* path_dev,
                             const int64_t* order_dev, double loss_scale, float* grad_dev, void* workspace_dev,
                             size_t workspace_bytes, void* stream_) {
  return rollout_bwd_impl<true, true>(env, mlp, params_host, cfg, noise_dev, coef_S_dev, coef_G_dev, T_dev, path_dev, order_dev,
                                      loss_scale, grad_dev, workspace_dev, workspace_bytes, stream_,
                                      (const long long*)path_base_dev);
}

// rollout + statistics + reverse pass of one device-resident REINFORCE iteration (everything but the parameter update)
static int reinforce_rollout_impl(const rlsde_env* env, const rlsde_mlp* mlp, const float* theta_dev, const rlsde_rollout_cfg* cfg,
                                  const float* noise_dev, float* G_dev, float* S_dev, int32_t* T_dev, float* path_dev,
                                  double* stats_dev, float* grad_dev, void* workspace_dev, size_t workspace_bytes,
                                  cudaStream_t stream) {
  int rc = check_env_mlp(env, mlp);
  if (rc != RLSDE_OK) return rc;
  if (!theta_dev || !G_dev || !S_dev || !T_dev || !path_dev || !stats_dev || !grad_dev || !workspace_dev) return RLSDE_ERR_INVALID_ARG;
  if (workspace_bytes < Workspace::fixed_bytes()) return RLSDE_ERR_WORKSPACE;
  FwdArgs A;
  if ((rc = make_args(env, cfg, A)) != RLSDE_OK) return rc;
  if ((A.flags & (RLSDE_F_STATE_F64 | RLSDE_F_HIT_BRIDGE)) || !(A.flags & RLSDE_F_STORE_PATH) || A.ckpt_every != 1)
    return RLSDE_ERR_INVALID_ARG;
  if ((A.flags & RLSDE_F_NOISE_INJECTED) && !noise_dev) return RLSDE_ERR_INVALID_ARG;
  if (A.K < 1) return RLSDE_ERR_INVALID_ARG;
  int sm = 0;
  if ((rc = device_sm_count(&sm)) != RLSDE_OK) return rc;
  // the device-resident step exists for the latency-bound regime only: warp-per-trajectory kernels
  if (mlp->d_hidden != WARP_H || A.K > warp_path_max_k(sm) || (A.flags & RLSDE_F_KERNEL_THREAD)) return RLSDE_ERR_UNSUPPORTED;
  A.noise = noise_dev;
  A.G = G_dev; A.S = S_dev; A.T = T_dev; A.path = path_dev;
  const Workspace ws{(char*)workspace_dev};
  A.counter = ws.counters();
  A.q_ctrl = ws.counters();
  const bool fast = (A.flags & RLSDE_F_TANH_FAST) != 0;
  const float scale = (float)(1.0 / (double)A.K_global);       // the loss is the mean over ALL shards' trajectories
  return with_shape(env->d, mlp->d_hidden, [&](auto shape) -> int {
    using S = decltype(shape);
    int lrc = -1;
    if constexpr (S::narrow) {
      lrc = launch_pack_mlp_const_dev<S::D>(theta_dev, ws.policy(), fast, stream);
      if (lrc == 0) lrc = launch_rollout_fwd_warp<S::D>(nullptr, ws.policy(), A, sm, stream);
      if (lrc == 0) lrc = launch_reduce_stats(A.K, passes_run(A), false, G_dev, S_dev, T_dev, nullptr, nullptr, stats_dev, ws.stats(),
                                              stream);
      if (lrc == 0) lrc = launch_rollout_bwd_warp<S::D>(nullptr, ws.policy(), A, scale, grad_dev, ws.bwd_partial(), sm, stream);
    }
    return launch_status(lrc, "reinforce rollout launch");
  });
}

int rlsde_reinforce_step(const rlsde_env* env, const rlsde_mlp* mlp, float* theta_dev, float* adam_m_dev, float* adam_v_dev,
                         const rlsde_rollout_cfg* cfg, const float* noise_dev, double lr, double beta1, double beta2,
                         double eps, int64_t step_t, float* G_dev, float* S_dev, int32_t* T_dev, float* path_dev,
                         double* stats_dev, float* grad_dev, void* workspace_dev, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!adam_m_dev || !adam_v_dev || step_t < 1) return RLSDE_ERR_INVALID_ARG;
  const int rc = reinforce_rollout_impl(env, mlp, theta_dev, cfg, noise_dev, G_dev, S_dev, T_dev, path_dev, stats_dev, grad_dev,
                                        workspace_dev, workspace_bytes, stream);
  if (rc != RLSDE_OK) return rc;
  const int P = (int)rlsde_param_count(mlp);
  const int lrc = launch_adam_step(P, 0, grad_dev, stats_dev, nullptr, theta_dev, adam_m_dev, adam_v_dev, lr, beta1, beta2, eps,
                                   step_t, nullptr, nullptr, stream);
  if (lrc != 0) return cuda_fail((cudaError_t)lrc, "adam_step launch");
  return RLSDE_OK;
}

int rlsde_reinforce_rollout(const rlsde_env* env, const rlsde_mlp* mlp, const float* theta_dev, const rlsde_rollout_cfg* cfg,
                            const float* noise_dev, float* G_dev, float* S_dev, int32_t* T_dev, float* path_dev,
                            double* stats_dev, float* grad_dev, double* packed_dev, void* workspace_dev, size_t workspace_bytes,
                            void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!packed_dev) return RLSDE_ERR_INVALID_ARG;
  const int rc = reinforce_rollout_impl(env, mlp, theta_dev, cfg, noise_dev, G_dev, S_dev, T_dev, path_dev, stats_dev, grad_dev,
                                        workspace_dev, workspace_bytes, stream);
  if (rc != RLSDE_OK) return rc;
  const int lrc = launch_pack_grad_stats((int)rlsde_param_count(mlp), grad_dev, stats_dev, packed_dev, stream);
  if (lrc != 0) return cuda_fail((cudaError_t)lrc, "pack_grad_stats launch");
  return RLSDE_OK;
}

int rlsde_reinforce_apply(const rlsde_mlp* mlp, float* theta_dev, float* adam_m_dev, float* adam_v_dev,
                          const double* packed_all_dev, int32_t n_ranks, double lr, double beta1, double beta2, double eps,
                          int64_t step_t, float* grad_out_dev, double* stats_out_dev, void* stream_) {
  if (!mlp || !theta_dev || !adam_m_dev || !adam_v_dev || !packed_all_dev || n_ranks < 1 || step_t < 1) return RLSDE_ERR_INVALID_ARG;
  const int64_t P = rlsde_param_count(mlp);
  if (P < 1) return RLSDE_ERR_INVALID_ARG;
  const int lrc = launch_adam_step((int)P, n_ranks, nullptr, nullptr, packed_all_dev, theta_dev, adam_m_dev, adam_v_dev, lr, beta1,
                                   beta2, eps, step_t, grad_out_dev, stats_out_dev, (cudaStream_t)stream_);
  if (lrc != 0) return cuda_fail((cudaError_t)lrc, "adam_step launch");
  return RLSDE_OK;
}

int rlsde_reduce_stats(int64_t K, int64_t n_steps_lim, uint32_t flags, const void* G_dev, const void* S_dev,
                       const int32_t* T_dev, const void* l2_dev, const void* logw_dev, double* stats_dev,
                       void* workspace_dev, size_t workspace_bytes, void* stream_) {
  if (K < 0 || !G_dev || !S_dev || !T_dev || !stats_dev || !workspace_dev) return RLSDE_ERR_INVALID_ARG;
  if (workspace_bytes < Workspace::o_policy) return RLSDE_ERR_WORKSPACE;
  const Workspace ws{(char*)workspace_dev};
  const int lrc = launch_reduce_stats(K, n_steps_lim, (flags & RLSDE_F_STATE_F64) != 0, G_dev, S_dev, T_dev, l2_dev, logw_dev,
                                      stats_dev, ws.stats(), (cudaStream_t)stream_);
  if (lrc != 0) return cuda_fail((cudaError_t)lrc, "reduce_stats launch");
  return RLSDE_OK;
}

int rlsde_tables(const double* state_grid_dev, int64_t Ns, const double* action_grid_dev, int64_t Na,
                 const uint8_t* in_ts_dev, int64_t n_ts, double alpha, double sigma, double dt, double h_half,
                 double lb, double rb, int64_t sprime_begin, int64_t sprime_end, double* P_dev, double* R_dev,
                 int32_t state_grid_uniform, double state_grid_step, void* stream_) {
  if (!state_grid_dev || !action_grid_dev || !in_ts_dev || Ns < 1 || Na < 1 || Ns > 65535) return RLSDE_ERR_INVALID_ARG;
  if (sprime_begin < 0 || sprime_end > Ns || sprime_begin > sprime_end) return RLSDE_ERR_INVALID_ARG;
  if (!(dt > 0) || !(sigma > 0) || !(h_half > 0)) return RLSDE_ERR_INVALID_ARG;
  if (!P_dev && !R_dev) return RLSDE_ERR_INVALID_ARG;
  const int lrc = launch_tables(state_grid_dev, Ns, action_grid_dev, Na, in_ts_dev, n_ts, alpha, sigma, dt, h_half, lb, rb,
                                sprime_begin, sprime_end, P_dev, R_dev, state_grid_uniform, state_grid_step, (cudaStream_t)stream_);
  if (lrc != 0) return cuda_fail((cudaError_t)lrc, "tables launch");
  return RLSDE_OK;
}

int rlsde_tables_colsum(const double* P_dev, int64_t n_sprime, int64_t Ns, int64_t Na, double* colsum_dev, void* stream_) {
  if (!P_dev || !colsum_dev || n_sprime < 0 || Ns < 1 || Na < 1) return RLSDE_ERR_INVALID_ARG;
  const int lrc = launch_tables_colsum(P_dev, n_sprime, Ns, Na, colsum_dev, (cudaStream_t)stream_);
  if (lrc != 0) return cuda_fail((cudaError_t)lrc, "tables_colsum launch");
  return RLSDE_OK;
}

size_t rlsde_dp_scratch_bytes(int64_t Ns, int64_t Na) { return (Ns > 0 && Na > 0) ? dp_sweep_scratch_bytes(Ns, Na) : 0; }

int rlsde_dp_sweep(const double* P_dev, int64_t Ns, int64_t Na, const double* R_dev, const uint8_t* in_ts_dev,
                   const double* v_dev, double gamma, double* values_dev, void* scratch_dev, size_t scratch_bytes,
                   void* stream_) {
  if (!P_dev || !R_dev || !in_ts_dev || !v_dev || !values_dev || !scratch_dev || Ns < 1 || Na < 1) return RLSDE_ERR_INVALID_ARG;
  if (scratch_bytes < dp_sweep_scratch_bytes(Ns, Na)) return RLSDE_ERR_WORKSPACE;
  const int lrc = launch_dp_sweep(P_dev, Ns, Na, R_dev, in_ts_dev, v_dev, gamma, values_dev, (double*)scratch_dev, (cudaStream_t)stream_);
  if (lrc != 0) return cuda_fail((cudaError_t)lrc, "dp_sweep launch");
  return RLSDE_OK;
}

int rlsde_dp_sweep_implicit(const double* state_grid_dev, int64_t Ns, const double* action_grid_dev, int64_t Na,
                            const uint8_t* in_ts_dev, double alpha, double sigma, double dt, double h_half,
                            int32_t state_grid_uniform, double state_grid_step, const double* R_dev, const double* v_dev,
                            double gamma, double* values_dev, void* stream_) {
  if (!state_grid_dev || !action_grid_dev || !in_ts_dev || !R_dev || !v_dev || !values_dev) return RLSDE_ERR_INVALID_ARG;
  if (Ns < 1 || Na < 1) return RLSDE_ERR_INVALID_ARG;
  if (Na > INT32_MAX || Ns > INT32_MAX / ((Na + IMPLICIT_THREADS - 1) / IMPLICIT_THREADS)) return RLSDE_ERR_INVALID_ARG;  // one block per (s, action tile)
  if (!(sigma > 0) || !(dt > 0) || !(h_half > 0)) return RLSDE_ERR_INVALID_ARG;
  if (state_grid_uniform && !(state_grid_step > 0)) return RLSDE_ERR_INVALID_ARG;
  const int lrc = launch_dp_sweep_implicit(state_grid_dev, Ns, action_grid_dev, Na, in_ts_dev, alpha, sigma, dt, h_half,
                                           state_grid_uniform, state_grid_step, R_dev, v_dev, gamma, values_dev,
                                           (cudaStream_t)stream_);
  if (lrc != 0) return cuda_fail((cudaError_t)lrc, "dp_sweep_implicit launch");
  return RLSDE_OK;
}

int rlsde_dp_rowmax(const double* values_dev, int64_t Ns, int64_t Na, double* vmax_dev, int64_t* argmax_dev, void* stream_) {
  if (!values_dev || Ns < 1 || Na < 1 || (!vmax_dev && !argmax_dev)) return RLSDE_ERR_INVALID_ARG;
  const int lrc = launch_dp_rowmax(values_dev, Ns, Na, vmax_dev, (long long*)argmax_dev, (cudaStream_t)stream_);
  if (lrc != 0) return cuda_fail((cudaError_t)lrc, "dp_rowmax launch");
  return RLSDE_OK;
}

int rlsde_env_step(const rlsde_env* env, int64_t K, const void* state_dev, const float* action_dev,
                   const float* dbt_in_dev, uint64_t seed, int64_t traj_offset, int64_t pass_index, uint32_t flags,
                   int32_t reward_type, void* next_state_dev, void* reward_dev, uint8_t* done_dev, float* dbt_out_dev,
                   void* stream_) {
  if (!env || env->d < 1 || env->d > RLSDE_MAX_D || K < 0) return RLSDE_ERR_INVALID_ARG;
  if (!state_dev || !action_dev || !next_state_dev || !reward_dev || !done_dev) return RLSDE_ERR_INVALID_ARG;
  if (reward_type != RLSDE_REWARD_STATE_ACTION && reward_type != RLSDE_REWARD_STATE_ACTION_NEXT_STATE) return RLSDE_ERR_INVALID_ARG;
  if (flags & RLSDE_F_HIT_BRIDGE) return RLSDE_ERR_INVALID_ARG;      // a single pass has no next pass to detect a crossing
  StepArgs A;
  memset(&A, 0, sizeof(A));
  fill_env_consts(env, A);
  A.grad_f32 = (flags & RLSDE_F_GRAD_F32) ? 1 : 0;
  A.d = env->d; A.reward_type = reward_type;
  A.K = K; A.traj_offset = traj_offset; A.pass_index = pass_index; A.seed = seed;
  A.state = state_dev; A.action = action_dev; A.dbt_in = dbt_in_dev;
  A.next_state = next_state_dev; A.reward = reward_dev; A.done = done_dev; A.dbt_out = dbt_out_dev;
  const int lrc = launch_env_step(A, (flags & RLSDE_F_STATE_F64) != 0, (cudaStream_t)stream_);
  if (lrc != 0) return cuda_fail((cudaError_t)lrc, "env_step launch");
  return RLSDE_OK;
}

int rlsde_noise_fill(uint64_t seed, int64_t traj_offset, int64_t K, int32_t d, int64_t pass_begin, int64_t n_pass,
                     double dt, float* out_dev, void* stream_) {
  if (K < 0 || n_pass < 0 || d < 1 || d > RLSDE_MAX_D || !out_dev || !(dt > 0)) return RLSDE_ERR_INVALID_ARG;
  const int lrc = launch_noise_fill(seed, traj_offset, K, d, pass_begin, n_pass, dt, out_dev, (cudaStream_t)stream_);
  if (lrc != 0) return cuda_fail((cudaError_t)lrc, "noise_fill launch");
  return RLSDE_OK;
}

int rlsde_fwd_mma_clamp_bounds(const float* params_host, double* out) {
  if (!params_host || !out) return RLSDE_ERR_INVALID_ARG;
  MlpConst<1, 32> W;
  pack_mlp_const_folded<1, 32>(params_host, W);
  fwd_mma_clamp_bounds<1, 32>(W, out[0], out[1]);
  return RLSDE_OK;
}

}  // extern "C"
