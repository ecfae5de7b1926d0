#!/usr/bin/env python
"""Throughput of the d = 1 rollout under a tabulated control (rlsde_rollout_fwd_table): one JSON line per table.

    python tools/bench_tabular.py [--K 1000000] [--n-steps-lim 1000] [--reps 20] [--warmup 5]

The workload is bench.py config 2's (beta = 1, dt = 0.005, x0 = -1, 1e6 trajectories, budget 1 000 passes, importance
weights with the exact stochastic integral, float32 state) with the MLP replaced by a table on the h = 0.01 grid:
  u_star     the HJB control u* (hjb_1d.HJBSolution1D.policy_opt_table)
  dp_greedy  env.action_space_h[greedy_action_idx] of 1 500 q-value-iteration sweeps on the h = 0.01 tables
  zero       u = 0
Metric: useful trajectory-steps/s (passes up to and including the detecting one, or the budget), timed with CUDA events around `reps` launches after at least half a second of warm-up.
Writes nothing.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return q
    except Exception as e:                  # the numbers still stand; say why the card description is missing
        return f"unavailable ({e})"


def tables(env_h):
    from rl_sde_is_b200.dynamic_programming import compute_p_tensor_batch, compute_r_table
    from rl_sde_is_b200.hjb_1d import HJBSolution1D
    from rl_sde_is_b200.tabular_dp_sweeps import DeviceTables, qvalue_iteration
    import torch
    out = {"u_star": HJBSolution1D(env_h).policy_opt_table(env_h)}
    env_h.set_action_space_bounds(); env_h.discretize_action_space(0.01)
    np.random.seed(0)
    T = DeviceTables(env_h, compute_r_table(env_h, device_out=True), compute_p_tensor_batch(env_h, device_out=True))
    res = qvalue_iteration(env_h, gamma=1.0, n_iterations=1500, r_table=None, p_tensor=T)
    out["dp_greedy"] = env_h.action_space_h[res["greedy_action_idx"]]
    del T
    torch.cuda.empty_cache()
    out["zero"] = np.zeros(env_h.n_states)
    return {k: np.asarray(v, dtype=np.float32).reshape(-1) for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--K", type=int, default=1_000_000)
    ap.add_argument("--n-steps-lim", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    a = ap.parse_args()
    import torch
    from rl_sde_is_b200 import _lib as L, rollout as R
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D
    env = DoubleWellStoppingTime1D(beta=1.0, alpha=1.0, dt=0.005)
    env.discretize_state_space(0.01)
    env_c = R.env_struct(env, L.HIT_X0_IN_LB_RB)
    grid = (env.state_space_low, env.state_space_high, env.h_state)
    card = gpu_info()
    for name, tab in tables(env).items():
        tab_dev = torch.as_tensor(tab, device="cuda")
        run = lambda seed: R.rollout_forward_table(env_c, tab_dev, a.K, grid=grid, seed=seed, n_steps_lim=a.n_steps_lim,
                                                   stoch_int="exact", want_logw=True)
        # warm up for at least `warmup` launches and half a second, so that clocks have settled before the timed window
        t0, i = time.perf_counter(), 0
        while i < a.warmup or time.perf_counter() - t0 < 0.5:
            run(1000 + i)
            torch.cuda.synchronize()
            i += 1
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        outs = []
        start.record()
        for i in range(a.reps):
            outs.append(run(i))
        stop.record()
        torch.cuda.synchronize()
        ms = start.elapsed_time(stop) / a.reps
        useful = float(np.mean([o.stats[L.ST_USEFUL_STEPS] for o in outs]))
        s = R.summarize(outs[-1].stats)
        print(json.dumps({"table": name, "K": a.K, "n_steps_lim": a.n_steps_lim, "n_grid": int(tab.size),
                          "ms_per_launch": round(ms, 4), "useful_steps": useful,
                          "useful_steps_per_s": useful / (ms * 1e-3), "n_unfinished": s["n_unfinished"],
                          "is_mean": s.get("is_mean"), "is_rel_error": s.get("is_rel_error"), "gpu": card}), flush=True)


if __name__ == "__main__":
    main()
