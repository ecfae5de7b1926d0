#!/usr/bin/env python
"""Cost of the Brownian-bridge hit test (RLSDE_F_HIT_BRIDGE): the same launch with the test on and off, alternating in
one process, one JSON line per (workload, bridge) and round.

    python tools/bench_bridge.py [--K 1000000] [--n-steps-lim 1000] [--reps 10] [--rounds 3]

Workloads (beta = 1, dt = 0.005, x0 = -1, target [1, 2], exact stochastic integral, importance weights):
  mlp_f32 / mlp_f64  bench.py config 2: the seed-1 MLP 1-32-32-1, 1e6 trajectories, budget 1 000 passes, float32 / float64
                     state (the dispatcher's choice of kernel and schedule)
  u_star             the HJB control u* tabulated on the h = 0.01 grid (rlsde_rollout_fwd_table), same budget
Metric: ms per launch (CUDA events around `reps` launches after warm-up) and useful trajectory-steps/s; the cost of the
bridge per useful trajectory-step is (t_on / steps_on - t_off / steps_off).  `draw_fraction`: passes on which the test
drew a uniform, counted by the float64 bridge replay (tests/test_bridge_hit.py) of the first 2 000 trajectories on the
same increments -- the kernels count nothing.  The card's name, power limit and clock are read in the same call.
Writes nothing.
"""
import argparse
import importlib.util
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
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:
        return f"unavailable ({e})"


def _replay_module():
    spec = importlib.util.spec_from_file_location("_bridge_replay", os.path.join(ROOT, "tests", "test_bridge_hit.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--K", type=int, default=1_000_000)
    ap.add_argument("--n-steps-lim", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--replay-K", type=int, default=2000)
    a = ap.parse_args()
    import torch
    from bench import WORKLOAD, make_policy
    from rl_sde_is_b200 import _lib as L, rollout as R
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D
    from rl_sde_is_b200.hjb_1d import HJBSolution1D
    env = DoubleWellStoppingTime1D(beta=1.0, alpha=1.0, dt=0.005)
    env.discretize_state_space(0.01)
    env_c = R.env_struct(env, L.HIT_X0_IN_LB_RB)
    grid = (env.state_space_low, env.state_space_high, env.h_state)
    model = make_policy(WORKLOAD["policy_seed"])
    params = R.flat_parameters(model).detach().numpy()
    state_dict = {k: v.detach().numpy().copy() for k, v in model.state_dict().items()}
    u_star = np.asarray(HJBSolution1D(env).policy_opt_table(env), dtype=np.float32).reshape(-1)
    tab_dev = torch.as_tensor(u_star, device="cuda")
    lim = a.n_steps_lim
    mlp_c = L.make_mlp(1, 32)
    work = {
        "mlp_f32": lambda seed, b: R.rollout_forward(env_c, mlp_c, params, a.K, seed=seed, n_steps_lim=lim, stoch_int="exact",
                                                     want_logw=True, bridge=b),
        "mlp_f64": lambda seed, b: R.rollout_forward(env_c, mlp_c, params, a.K, seed=seed, n_steps_lim=lim, stoch_int="exact",
                                                     want_logw=True, state_f64=True, bridge=b),
        "u_star": lambda seed, b: R.rollout_forward_table(env_c, tab_dev, a.K, grid=grid, seed=seed, n_steps_lim=lim,
                                                          stoch_int="exact", want_logw=True, bridge=b),
    }
    card = gpu_info()
    # passes that drew a uniform, from the float64 replay on the kernels' increments (seed 0, first replay_K trajectories)
    rp = _replay_module()
    noise = R.noise_fill(0, a.replay_K, 1, lim, env.dt).cpu().numpy()
    draws = {}
    for name, pol in (("mlp", rp.mlp_policy(state_dict, f32_input=True)), ("u_star", rp.table_policy(u_star, grid))):
        r = rp.bridge_replay(pol, noise, seed=0, device="cuda")
        draws[name] = (r["n_draws"], r["n_passes"])
    for name, run in work.items():
        for b in (False, True):
            for i in range(3):
                run(100 + i, b)
        torch.cuda.synchronize()
    for rnd in range(a.rounds):
        for name, run in work.items():
            for b in (False, True):
                t0 = time.perf_counter()
                while time.perf_counter() - t0 < 0.3:
                    run(900, b)
                    torch.cuda.synchronize()
                start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                outs = []
                start.record()
                for i in range(a.reps):
                    outs.append(run(i, b))
                stop.record()
                torch.cuda.synchronize()
                ms = start.elapsed_time(stop) / a.reps
                useful = float(np.mean([o.stats[L.ST_USEFUL_STEPS] for o in outs]))
                s = R.summarize(outs[0].stats)
                nd, npass = draws["u_star" if name == "u_star" else "mlp"]
                print(json.dumps({"workload": name, "bridge": b, "round": rnd, "K": a.K, "n_steps_lim": lim,
                                  "ms_per_launch": round(ms, 4), "useful_steps": useful,
                                  "ns_per_useful_step": ms * 1e6 / useful, "useful_steps_per_s": useful / (ms * 1e-3),
                                  "n_unfinished": s["n_unfinished"], "is_mean": s.get("is_mean"),
                                  "is_rel_error": s.get("is_rel_error"), "mean_T": s.get("mean_T"),
                                  "draw_fraction_replay": nd / max(npass, 1) if b else None, "gpu": card}), flush=True)


if __name__ == "__main__":
    main()
