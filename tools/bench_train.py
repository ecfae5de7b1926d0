#!/usr/bin/env python
"""Large-batch REINFORCE loss + gradient timing (K1 with state checkpoints + the reverse pass), CUDA events.
    python tools/bench_train.py [--d 1] [--K 400000] [--lim 4000] [--ckpt 1] [--reps 3]"""
import argparse, json, os, sys
import numpy as np, torch, torch.nn as nn
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rl_sde_is_b200 import _lib as L, rollout as R
from rl_sde_is_b200.environments import DoubleWellStoppingTime1D, DoubleWellStoppingTimeND
from rl_sde_is_b200.models import DeterministicPolicy

ap = argparse.ArgumentParser()
ap.add_argument("--d", type=int, default=1); ap.add_argument("--K", type=int, default=400000)
ap.add_argument("--lim", type=int, default=4000); ap.add_argument("--ckpt", type=int, default=1)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--bias", type=float, default=None)
a = ap.parse_args()
d = a.d
env = DoubleWellStoppingTime1D(beta=1.0, alpha=1.0, dt=0.005) if d == 1 else DoubleWellStoppingTimeND(d, beta=1.0, alpha=1.0, dt=0.005)
torch.manual_seed(1)
m = DeterministicPolicy(d, d, [32, 32], nn.Tanh())
m.policy[4].bias.data.fill_(a.bias if a.bias is not None else (0.5 if d == 1 else 3.0))
params = R.flat_parameters(m).detach().numpy()
env_c, mlp_c = R.env_struct(env, L.HIT_ALL_GE_LB), L.make_mlp(d, 32)
for it in range(a.reps):
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    e[0].record()
    fo = R.rollout_forward(env_c, mlp_c, params, a.K, seed=it, n_steps_lim=a.lim, store_path=True, ckpt_every=a.ckpt, want_logw=False)
    e[1].record()
    g = R.rollout_backward(env_c, mlp_c, params, fo, 1.0 / a.K)
    e[2].record()
    torch.cuda.synchronize()
u = float(fo.stats[L.ST_USEFUL_STEPS])
f_ms, b_ms = e[0].elapsed_time(e[1]), e[1].elapsed_time(e[2])
F = 3 * 2 * (2 * d * 32 + 1024) + 24 * d + 4
print(json.dumps({"d": d, "K": a.K, "ckpt": a.ckpt, "useful_steps": u, "fwd_ms": f_ms, "bwd_ms": b_ms,
                  "bwd_steps_per_s": u / b_ms * 1e3, "train_steps_per_s": u / (f_ms + b_ms) * 1e3,
                  "fp32_frac_train": u / (f_ms + b_ms) * 1e3 * F / 74.45e12, "grad_norm": float(g.norm())}))
