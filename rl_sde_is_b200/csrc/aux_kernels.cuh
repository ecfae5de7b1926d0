// Declarations of the small kernels' launchers (aux_kernels.cu) and of the table builder (tables.cu).
#pragma once
#include "rollout_fwd.cuh"

namespace rlsde {

constexpr int STATS_BLOCKS = 256;

struct StepArgs {
  float c4a_f[RLSDE_MAX_D];
  double c4a_d[RLSDE_MAX_D];
  float sigma_f, dt_f;
  double sigma_d, dt_d, lb_d, rb_d;
  float noise_scale2;
  int d, hit_rule, reward_type, grad_f32;
  float lb_f, rb_f;
  long long K, traj_offset, pass_index;
  unsigned long long seed;
  const void* state;
  const float* action;
  const float* dbt_in;
  void* next_state;
  void* reward;
  unsigned char* done;
  float* dbt_out;
};

int launch_reduce_stats(long long K, long long n_steps_lim, bool f64, const void* G, const void* S, const int* T,
                        const void* l2, const void* logw, double* stats, double* partial, cudaStream_t stream);
int launch_adam_step(int P, int n_ranks, const float* grad, const double* stats, const double* packed, float* theta, float* m,
                     float* v, double lr, double beta1, double beta2, double eps, long long step_t, float* grad_out,
                     double* stats_out, cudaStream_t stream);
int launch_pack_grad_stats(int P, const float* grad, const double* stats, double* packed, cudaStream_t stream);
int launch_noise_fill(unsigned long long seed, long long traj_offset, long long K, int d, long long pass_begin,
                      long long n_pass, double dt, float* out, cudaStream_t stream);
int launch_env_step(const StepArgs& A, bool f64, cudaStream_t stream);

int launch_tables(const double* state_grid, long long Ns, const double* action_grid, long long Na,
                  const unsigned char* in_ts, long long n_ts, double alpha, double sigma, double dt, double h_half,
                  double lb, double rb, long long sprime_begin, long long sprime_end, double* P, double* R,
                  int uniform_grid, double grid_step, cudaStream_t stream);
int launch_tables_colsum(const double* P, long long n_sprime, long long Ns, long long Na, double* colsum,
                         cudaStream_t stream);

int launch_dp_sweep(const double* P, long long Ns, long long Na, const double* R, const unsigned char* in_ts,
                    const double* v, double gamma, double* values, double* scratch, cudaStream_t stream);
size_t dp_sweep_scratch_bytes(long long Ns, long long Na);
int launch_dp_sweep_implicit(const double* sgrid, long long Ns, const double* agrid, long long Na,
                             const unsigned char* in_ts, double alpha, double sigma, double dt, double h_half,
                             int uniform_grid, double grid_step, const double* R, const double* v, double gamma,
                             double* values, cudaStream_t stream);
constexpr int IMPLICIT_THREADS = 128;            // actions per block of the tensor-free sweep
int launch_dp_rowmax(const double* values, long long Ns, long long Na, double* vmax, long long* arg, cudaStream_t stream);

}  // namespace rlsde
