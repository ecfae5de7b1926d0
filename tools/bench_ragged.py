#!/usr/bin/env python
"""Loss plus gradient (rollout_loss_and_grad) on the dense and on the ragged checkpoint store: time and peak device memory.

    python tools/bench_ragged.py [--reps 3] [--out FILE.jsonl]

Where both stores fit, the two routes alternate on one policy and seed: the ragged route costs one more forward rollout
and one host synchronisation, and needs memory for the passes run instead of the pass budget.  Where the dense store
does not fit (the default budget of 10**6 passes at H = 256, and a metastable beta = 4 batch), the ragged route alone.
One JSON line per measurement."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rl_sde_is_b200 import _lib as L, rollout as R                                   # noqa: E402
from rl_sde_is_b200.environments import DoubleWellStoppingTime1D, DoubleWellStoppingTime2D  # noqa: E402
from rl_sde_is_b200.models import DeterministicPolicy                              # noqa: E402

# (name, d, H, K, n_steps_lim, beta, both routes)
CASES = [
    ("d1_h32_K4e5_lim2000", 1, 32, 400_000, 2000, 1.0, True),
    ("d1_h256_K6e4_lim20000", 1, 256, 60_000, 20_000, 1.0, True),
    ("d10_h32_K1e6_lim2000", 10, 32, 1_000_000, 2000, 1.0, True),
    ("d1_h256_K6e4_default_budget", 1, 256, 60_000, 10**6, 1.0, False),
    ("d1_h32_K1e5_beta4_default_budget", 1, 32, 100_000, 10**6, 4.0, False),
]


def env_for(d, beta):
    if d == 1:
        return DoubleWellStoppingTime1D(beta=beta, alpha=1.0, dt=0.005)
    if d == 2:
        return DoubleWellStoppingTime2D(beta=beta, alpha=1.0, dt=0.005)
    from rl_sde_is_b200.environments import DoubleWellStoppingTimeND
    return DoubleWellStoppingTimeND(d=d, beta=beta, alpha=1.0, dt=0.005)


def run(env_c, mlp_c, flat, K, lim, ckpt, seed):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    t0 = time.perf_counter()
    stats, grad, G, T = R.rollout_loss_and_grad(env_c, mlp_c, flat, K, seed=seed, n_steps_lim=lim, ckpt_every=ckpt)
    dt = time.perf_counter() - t0                      # the call ends in a device-to-host copy of its results
    peak = torch.cuda.max_memory_allocated() - base
    return dt, peak, stats, grad, T


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cases", default="")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    out = open(a.out, "a") if a.out else None
    props = torch.cuda.get_device_properties(0)
    for name, d, H, K, lim, beta, both in CASES:
        if a.cases and name not in a.cases.split(","):
            continue
        env = env_for(d, beta)
        torch.manual_seed(0)
        model = DeterministicPolicy(d, d, [H, H], torch.nn.Tanh())
        if d > 1:       # a drift towards the orthant target, which an untrained policy at d = 10 almost never reaches
            with torch.no_grad():
                R.policy_linears(model)[2].bias.fill_(1.5)
        env_c, mlp_c = R.env_struct(env, L.HIT_ALL_GE_LB), L.make_mlp(d, H)
        flat = R.flat_parameters(model).detach().numpy()
        dense_c = R.choose_path_store(K, d, lim, hidden=H)
        routes = [("ragged", None)] + ([("dense", dense_c)] if both and dense_c is not None else [])
        for r, ck in routes:                           # warm-up: module loads, workspace, allocator
            run(env_c, mlp_c, flat, K, lim, ck, 1)
        grads = {}
        for rep in range(a.reps):
            for r, ck in routes:
                dt, peak, stats, grad, T = run(env_c, mlp_c, flat, K, lim, ck, 2 + rep)
                grads[r] = grad
                s = R.summarize(stats)
                if ck is None:          # the spacing the ragged route picked, from the same hit indices
                    T = T.astype(np.int64)[T >= 0]
                    sp = R.RAGGED_SPACINGS if H == 32 else R.RAGGED_SPACINGS[:1]
                    ck_r = R.choose_ragged_ckpt_every([int((T // c + 1).sum()) for c in sp], d, hidden=H)
                rec = dict(case=name, route=r, ckpt_every=ck if ck is not None else ck_r, rep=rep, seconds=dt,
                           peak_bytes=int(peak), d=d, H=H, K=K, n_steps_lim=lim, beta=beta, mean_hit_index=s.get("mean_hit_index"), max_hit_index=s["max_hit_index"],
                           n_unfinished=s["n_unfinished"], gpu=props.name)
                print(json.dumps(rec), flush=True)
                if out:
                    out.write(json.dumps(rec) + "\n")
            if len(grads) == 2:     # bit for bit where both routes ran at the same spacing (the reverse kernels scale per segment)
                print(json.dumps(dict(case=name, rep=rep, grads_equal=bool(np.array_equal(grads["ragged"], grads["dense"])))),
                      flush=True)


if __name__ == "__main__":
    main()
