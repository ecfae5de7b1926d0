#!/usr/bin/env python
"""Cost of the weighted reverse pass: rlsde_rollout_bwd and rlsde_rollout_bwd_weighted (cG = -1, cS = -G, the same
gradient) alternating in one process on one forward rollout, one JSON line per shape.

    python tools/bench_bwd_weighted.py [--reps 5] [--rounds 3]

Shapes (beta = 1, alpha = 1, dt = 0.005, x0 = -1, target [1, 2], seeded MLP with head bias 2 (d = 1) / 3 (d = 10),
budget 2 000 passes, Philox noise, precise tanh, reference integral, length-sorted order):
  d1_h32   d = 1,  H = 32,  K = 4e5: K2m with the longest trajectories split onto the warp kernel (bwd_warp_share auto)
  d10_h32  d = 10, H = 32,  K = 1e6: K2m
  d1_h256  d = 1,  H = 256, K = 6e4: K2u
Metric: ms per call (CUDA events around `reps` calls after one warm-up call of each), the median over `rounds` rounds
in which the two entry points alternate, and their ratio.  The card's name, power limit and clock are read in the same
call.  Writes nothing.
"""
import argparse
import json
import os
import subprocess
import sys

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


SHAPES = [("d1_h32", 1, 32, 400_000), ("d10_h32", 10, 32, 1_000_000), ("d1_h256", 1, 256, 60_000)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--n-steps-lim", type=int, default=2000)
    args = ap.parse_args()
    import torch
    import torch.nn as nn
    from rl_sde_is_b200 import _lib as L, rollout as R
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D, DoubleWellStoppingTimeND
    from rl_sde_is_b200.models import DeterministicPolicy

    info = gpu_info()
    for name, d, H, K in SHAPES:
        env = DoubleWellStoppingTime1D(beta=1.0, alpha=1.0, dt=0.005) if d == 1 else DoubleWellStoppingTimeND(d, beta=1.0, alpha=1.0, dt=0.005)
        torch.manual_seed(1)
        m = DeterministicPolicy(d, d, [H, H], nn.Tanh())
        m.policy[4].bias.data.fill_(2.0 if d == 1 else 3.0)
        flat = R.flat_parameters(m).detach().numpy()
        env_c, mlp_c = R.env_struct(env, L.HIT_ALL_GE_LB), L.make_mlp(d, H)
        fwd = R.rollout_forward(env_c, mlp_c, flat, K, seed=7, n_steps_lim=args.n_steps_lim, store_path=True, want_logw=False)
        done = float((fwd.T >= 0).float().mean())
        coef = (torch.full_like(fwd.G, -1.0), (-fwd.G).contiguous())
        calls = {"bwd": lambda: R.rollout_backward(env_c, mlp_c, flat, fwd, 1.0 / K),
                 "weighted": lambda: R.rollout_backward(env_c, mlp_c, flat, fwd, 1.0 / K, coef=coef)}
        grads = {k: f() for k, f in calls.items()}
        torch.cuda.synchronize()
        ms = {k: [] for k in calls}
        for _ in range(args.rounds):
            for k, f in calls.items():
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record()
                for _ in range(args.reps):
                    f()
                t1.record()
                torch.cuda.synchronize()
                ms[k].append(t0.elapsed_time(t1) / args.reps)
        med = {k: float(np.median(v)) for k, v in ms.items()}
        print(json.dumps({"shape": name, "d": d, "H": H, "K": K, "n_steps_lim": args.n_steps_lim, "finished": done,
                          "ms_bwd": med["bwd"], "ms_weighted": med["weighted"], "ratio": med["weighted"] / med["bwd"],
                          "ms_rounds": ms, "bitwise_equal": bool(torch.equal(grads["bwd"], grads["weighted"])), "gpu": info}),
              flush=True)


if __name__ == "__main__":
    main()
