// Forward rollout at d = 1 under a tabulated control: u_k = table[grid_index(x_k)], the cell lookup of the l2 error.
// A lean kernel on K1's per-pass arithmetic (TrajOwner::pass, traj_owner.cuh: noise, hit rules, accumulators, budget,
// outputs) with one trajectory per thread and lane refill from the work counter after every pass; the statistics record
// is the shared reduction.  It is a separate kernel rather than a policy choice inside K1 because templating K1 on the
// policy changed the SASS of every existing K1 instantiation.  A pass costs a quarter of a Philox block and its Box-Muller
// transform, the Euler-Maruyama arithmetic and one shared-memory load for the policy.  Tails are run to completion: a
// table pass is a few dozen instructions, so the last long trajectory costs little (profiles/r06).
#include "traj_owner.cuh"

namespace rlsde {

// SMEM: the block copies the table to shared memory first (n_grid <= FWD_TAB_SMEM_MAX); otherwise it reads it with __ldg
// BRIDGE: the Brownian-bridge hit test between passes (TrajOwner::pass)
template <bool F64, bool SMEM, bool BRIDGE = false>
__global__ void __launch_bounds__(128, 8) rollout_fwd_tab_kernel(const __grid_constant__ FwdArgs A, const float* __restrict__ table) {
  constexpr unsigned FULL = 0xffffffffu;
  extern __shared__ float s_tab[];
  if constexpr (SMEM) {
    for (long long i = threadIdx.x; i < A.n_grid; i += blockDim.x) s_tab[i] = __ldg(table + i);
    __syncthreads();
  }
  const int lane = threadIdx.x & 31;
  const bool inject = (A.flags & RLSDE_F_NOISE_INJECTED) != 0;
  const long long lim = inject ? (A.noise_steps < A.n_steps_lim ? A.noise_steps : A.n_steps_lim) : A.n_steps_lim;
  TrajOwner<1, F64, BRIDGE> o;
  o.init(A);
  for (;;) {
    const bool idle = !o.alive && !o.exhausted;
    const unsigned need = __ballot_sync(FULL, idle);
    if (need) {
      unsigned long long base = 0;
      const int leader = __ffs(need) - 1;
      if (lane == leader) base = atomicAdd(A.counter, (unsigned long long)__popc(need));
      base = __shfl_sync(FULL, base, leader);
      if (idle) {
        const long long idx = (long long)base + __popc(need & ((1u << lane) - 1u));
        if (idx < A.K) o.start(A, idx);
        else o.exhausted = true;
      }
    }
    if (!__any_sync(FULL, o.alive)) break;
    if (o.alive) {
      const long long gi = grid_index(A, (double)o.x[0]);
      const float u[1] = {SMEM ? s_tab[gi] : __ldg(table + gi)};
      o.pass(A, u, lim);
    }
  }
}

template <bool F64, bool SMEM, bool BRIDGE>
static int launch_tab_variant(const float* table, const FwdArgs& args, int sm_count, cudaStream_t stream) {
  auto kern = rollout_fwd_tab_kernel<F64, SMEM, BRIDGE>;
  const size_t smem = SMEM ? (size_t)args.n_grid * sizeof(float) : 0;
  int block;
  const long long grid = persistent_grid(kern, args.K, sm_count, smem, 0, block);
  kern<<<(unsigned)grid, block, smem, stream>>>(args, table);
  note_kernel_launches(1);
  return (int)cudaGetLastError();
}

int launch_rollout_fwd_table(const float* table, const FwdArgs& args, int sm_count, cudaStream_t stream) {
  return with_fwd_variant<1, false>(args.flags, [&](auto f64, auto, auto bridge) {
    return with_flag(args.n_grid <= FWD_TAB_SMEM_MAX, [&](auto smem) {
      return launch_tab_variant<f64, smem, bridge>(table, args, sm_count, stream);
    });
  });
}

}  // namespace rlsde
