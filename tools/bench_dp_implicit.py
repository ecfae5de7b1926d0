"""Per-sweep time of the Bellman sweep over the resident tensor (K6, rlsde_dp_sweep) against the tensor-free sweep (K6i,
rlsde_dp_sweep_implicit), and the wall time of q-value iteration on either route.  One JSON line per measurement.

    python tools/bench_dp_implicit.py [--rounds 7] [--reps 50] [--iters 1500]

Timing: CUDA events around `reps` back-to-back launches of one route, after warm-up; the two routes alternate within each
of `rounds` rounds, and the median, min and max per-sweep times over the rounds are reported (the spread).  Both routes
are called through the C ABI with preallocated buffers, so no Python work sits between launches.  The dense tensor
(0.77 GB and 5.1 GB here) is larger than the 126 MB L2: each dense sweep streams it from HBM.  The implicit sweep reads
O(Ns) bytes and is bound by the FP64 pipe; its share of the FP64 rate is credited as
    FP64_PER_ENTRY x (entries visited) / time / (148 SMs x 64 FP64 lanes x max SM clock),
with the entries visited computed on the host from the kernel's band rule (warp unions, idle lanes not counted)."""
import argparse, json, os, subprocess, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rl_sde_is_b200 import _lib as L
from rl_sde_is_b200.dynamic_programming import compute_p_tensor_batch
from rl_sde_is_b200.environments import DoubleWellStoppingTime1D
from rl_sde_is_b200.rollout import _ptr
from rl_sde_is_b200.tabular_dp_sweeps import DeviceTables, ImplicitTables, qvalue_iteration

# FP64 instructions per visited entry in the inner loop of dp_sweep_implicit_kernel<true> (SASS, cuobjdump -sass):
# DADD (ya + yb), DMUL (phi * .), DFMA (acc), DMUL x 2 (phi, r), DADD + DFMA (a node), DADD + DFMA (b node)
FP64_PER_ENTRY = 9
BAND_Z, THREADS = 9.0, 128


def hardware():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clock = (x.strip() for x in q.split(","))
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return {"gpu": name, "power_limit_W": float(power), "max_sm_clock_MHz": float(clock), "sms": sms}


def make_env(hs, ha, beta=1.0, dt=0.005):
    env = DoubleWellStoppingTime1D(beta=beta, alpha=1.0, dt=dt)
    env.set_action_space_bounds(); env.discretize_state_space(hs); env.discretize_action_space(ha)
    return env


def entries_visited(env):
    """Sum over the columns of non-target states of the rows their warp walks (the kernel's band rule)."""
    x, a = np.asarray(env.state_space_h, np.float64), np.asarray(env.action_space_h, np.float64)
    h, sd = env.h_state / 2.0, env.sigma * np.sqrt(env.dt)
    inner = x[1:] - h
    Na, total = a.size, 0
    for s in np.flatnonzero(~env.is_in_ts):
        xs = x[s]
        mu = xs + (-(4.0 * env.alpha * xs * (xs * xs - 1.0)) + env.sigma * a) * env.dt
        lo = np.searchsorted(inner, mu - BAND_Z * sd, side="left")
        hi = np.searchsorted(inner, mu + BAND_Z * sd, side="right")
        for w in range(0, Na, 32):                                   # a warp: 32 consecutive actions of one state
            n = min(32, Na - w)
            total += n * (hi[w:w + n].max() - lo[w:w + n].min() + 1)
    return int(total)


def dense_call(T, v, out, gamma):
    lib, st = L.load(), torch.cuda.current_stream().cuda_stream
    args = (_ptr(T.P), T.Ns, T.Na, _ptr(T.R), _ptr(T.in_ts), _ptr(v), gamma, _ptr(out), _ptr(T.scratch), T.scratch.numel(), st)
    return lambda: lib.rlsde_dp_sweep(*args)


def implicit_call(T, v, out, gamma):
    lib, st = L.load(), torch.cuda.current_stream().cuda_stream
    args = (_ptr(T.sgrid), T.Ns, _ptr(T.agrid), T.Na, _ptr(T.in_ts), *T.consts, T.uniform, T.step, _ptr(T.R), _ptr(v), gamma,
            _ptr(out), st)
    return lambda: lib.rlsde_dp_sweep_implicit(*args)


def time_ms(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()                                             # keeps the stream busy while the first timed launch is enqueued
    a.record()
    for _ in range(reps):
        rc = fn()
    b.record(); torch.cuda.synchronize()
    assert rc == 0, rc
    return a.elapsed_time(b) / reps


def stats(ts):
    return {"median_ms": float(np.median(ts)), "min_ms": float(np.min(ts)), "max_ms": float(np.max(ts)), "all_ms": ts}


def emit(rec):
    print(json.dumps(rec), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--iters", type=int, default=1500)
    args = ap.parse_args()
    hw = hardware()
    emit({"what": "hardware", **hw})
    fp64_rate = hw["sms"] * 64 * hw["max_sm_clock_MHz"] * 1e6
    cases = [("config 3 (h_s = h_a = 0.01)", dict(hs=0.01, ha=0.01), True),
             ("config 5 env (beta = 4, dt = 0.001), h_s = 0.005, h_a = 0.01", dict(hs=0.005, ha=0.01, beta=4.0, dt=0.001), True),
             ("h_s = 0.001, h_a = 0.01", dict(hs=0.001, ha=0.01), False),
             ("h_s = h_a = 0.001", dict(hs=0.001, ha=0.001), False)]
    gamma = 1.0
    for name, kw, with_dense in cases:
        env = make_env(**kw)
        I = ImplicitTables(env)
        v = torch.as_tensor(-3.0 * np.random.default_rng(0).random(env.n_states), device="cuda")
        out_i = torch.empty((I.Ns, I.Na), dtype=torch.float64, device="cuda")
        fns = {"implicit": implicit_call(I, v, out_i, gamma)}
        D = None
        if with_dense:
            D = DeviceTables(env, I.R, compute_p_tensor_batch(env, device_out=True))
            out_d = torch.empty_like(out_i)
            fns["dense"] = dense_call(D, v, out_d, gamma)
        reps = max(3, args.reps if I.Ns * I.Na < 5e6 else args.reps // 10)
        for fn in fns.values():                      # warm-up: module load, occupancy queries
            time_ms(fn, 2)
        ts = {k: [] for k in fns}
        for _ in range(args.rounds):
            for k, fn in fns.items():
                ts[k].append(time_ms(fn, reps))
        entries = entries_visited(env)
        rec = {"what": "per-sweep time", "grid": name, "Ns": I.Ns, "Na": I.Na, "reps_per_round": reps,
               "rounds": args.rounds, "path": "quadrature" if (I.uniform and env.h_state / (env.sigma * np.sqrt(env.dt)) <= 0.2)
               else "erf", "implicit": stats(ts["implicit"]), "entries_visited": entries,
               "entries_per_column": entries / float((~env.is_in_ts).sum() * I.Na),
               "dense_tensor_GB": 8.0 * I.Ns * I.Ns * I.Na / 1e9}
        t = rec["implicit"]["median_ms"] * 1e-3
        rec["implicit"]["entries_per_s"] = entries / t
        if rec["path"] == "quadrature":
            rec["implicit"]["fp64_share"] = FP64_PER_ENTRY * entries / t / fp64_rate
        if D is not None:
            rec["dense"] = stats(ts["dense"])
            rec["dense"]["GBps"] = 8.0 * I.Ns * I.Ns * I.Na / (rec["dense"]["median_ms"] * 1e-3) / 1e9
            rec["speedup_median"] = rec["dense"]["median_ms"] / rec["implicit"]["median_ms"]
            rec["max_abs_diff"] = float((out_i - out_d).abs().max())
        emit(rec)
        if kw in (dict(hs=0.01, ha=0.01), dict(hs=0.001, ha=0.01)):
            routes = {"implicit": I} if D is None else {"dense": D, "implicit": I}
            walls = {}
            for rname, T in routes.items():
                np.random.seed(0)
                torch.cuda.synchronize(); t0 = time.perf_counter()
                res = qvalue_iteration(env, gamma=1.0, n_iterations=args.iters, p_tensor=T)
                torch.cuda.synchronize(); walls[rname] = time.perf_counter() - t0
                walls[rname + "_v_init"] = float(res["v_table"][env.state_init_idx[0]])
            emit({"what": f"qvalue_iteration wall time, {args.iters} sweeps (host clock, ends in a synchronise)", "grid": name,
                  **{k: v for k, v in walls.items()}})
        del D, I
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
