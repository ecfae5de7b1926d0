"""rl_sde_is_b200 -- the data-parallel hot path of riberaborrell/rl-sde-is on B200 (sm_100a).

Module names mirror the reference package ``rl_sde_is`` for the functions on the hot path:

    environments                  DoubleWellStoppingTime1D / 2D / ND  (env.step, env.step_torch, grids)
    models                        mlp, DeterministicPolicy
    reinforce_deterministic_core  sample_loss_vectorized, sample_returns_vectorized, reinforce
    approximate_methods           test_policy_vectorized, estimate_fht_vectorized, is_estimate
    dynamic_programming           compute_r_table, compute_p_tensor_batch
    tabular_dp_tables             check_p_tensor, dynamic_programming_tables
    rollout / distributed / _lib  device-level API, sharding, ctypes binding of include/rlsde.h

Everything computes in hand-written CUDA kernels behind a C ABI (librlsde_b200.so); there is no CPU
fallback: calls raise if the library is not built or no CUDA device is present.
"""
__version__ = "0.1.0"
