#!/usr/bin/env python
"""Forward test rollout (config 2 workload: 1-D, H = 32, n_steps_lim 1000) through the kernel families, CUDA events.
    python tools/bench_fwd_kernels.py [--K 1000000] [--d 1] [--lim 1000] [--f64] [--tanh precise] [--policy ffma,mma]
                                      [--blocks-per-sm 0]
--policy runs the thread-per-trajectory kernel ("thread") once per policy arithmetic (cfg.fwd_policy); the tensor-core
kernel ("tensor") is timed once."""
import argparse, json, os, sys
import numpy as np, torch, torch.nn as nn
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rl_sde_is_b200 import _lib as L, rollout as R
from rl_sde_is_b200.environments import DoubleWellStoppingTime1D, DoubleWellStoppingTimeND
from rl_sde_is_b200.models import DeterministicPolicy
ap = argparse.ArgumentParser()
ap.add_argument("--K", type=int, default=1000000); ap.add_argument("--d", type=int, default=1); ap.add_argument("--lim", type=int, default=1000)
ap.add_argument("--f64", action="store_true"); ap.add_argument("--tanh", default="precise"); ap.add_argument("--bias", type=float, default=None)
ap.add_argument("--kernels", default="thread,tensor")
ap.add_argument("--policy", default="auto", help="comma-separated fwd_policy values for the thread kernel: auto, ffma, mma")
ap.add_argument("--blocks-per-sm", type=int, default=0, help="cap on resident blocks per SM of the thread kernel (0 = occupancy)")
a = ap.parse_args()
d = a.d
env = DoubleWellStoppingTime1D(beta=1.0, alpha=1.0, dt=0.005) if d == 1 else DoubleWellStoppingTimeND(d, beta=1.0, alpha=1.0, dt=0.005)
np.random.seed(1); torch.manual_seed(1)
m = DeterministicPolicy(d, d, [32, 32], nn.Tanh())
if a.bias is not None or d > 1:
    m.policy[4].bias.data.fill_(a.bias if a.bias is not None else 3.0)
params = R.flat_parameters(m).detach().numpy()
env_c, mlp_c = R.env_struct(env, L.HIT_X0_IN_LB_RB if d == 1 else L.HIT_ALL_GE_LB), L.make_mlp(d, 32)
F = 2 * (2 * d * 32 + 1024) + 14 * d + 4
runs = [(k, p) for k in a.kernels.split(",") for p in (a.policy.split(",") if k == "thread" else ["auto"])]
for kern, pol in runs:
    tuning = {"fwd_policy": pol, "fwd_blocks_per_sm": a.blocks_per_sm or None}
    ts = []
    for it in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = R.rollout_forward(env_c, mlp_c, params, a.K, seed=it, n_steps_lim=a.lim, stoch_int="exact", state_f64=a.f64, tanh=a.tanh, kernel=kern,
                                tuning=tuning)
        e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    u = float(out.stats[L.ST_USEFUL_STEPS]); ms = float(np.median(ts[2:]))
    s = R.summarize(out.stats)
    print(json.dumps({"kernel": kern, "policy": pol, "blocks_per_sm": a.blocks_per_sm, "d": d, "K": a.K, "f64": a.f64, "tanh": a.tanh, "ms": ms, "steps_per_s": u / ms * 1e3, "fp32_frac": u / ms * 1e3 * F / 74.45e12,
                      "mean_return": s.get("mean_return"), "is_mean": s.get("is_mean"), "n_unfinished": s["n_unfinished"], "mean_hit": s.get("mean_hit_index")}))
