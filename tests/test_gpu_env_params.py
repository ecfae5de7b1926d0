"""Every rollout and reverse-pass kernel against the float64 reference away from the default environment.

The kernels read alpha and x0 per coordinate, sigma, dt, lb and rb from the rlsde_env they are given (capi.cu fill_env,
and the single-pass packer of rlsde_env_step).  With the default environment -- alpha = 1 and x0 = -1 in every coordinate,
beta = 1, target [1, 2] -- a kernel that read coordinate 0's alpha or x0 for every coordinate, swapped lb and rb, or took
sigma from elsewhere would pass every other test.  Here every forward family (FWD_CASES of test_gpu_fp64_reference.py),
the table kernel, the Brownian-bridge hit test, every reverse family (BWD_CASES), the single pass and the transition
stream run in

    E_d (d >= 2): alpha_i cycling through 0.5, 1.5, 0.75, 2; x0_i through -1.25, -0.75, -1.5, -1; beta = 2 (sigma = 1),
                  dt = 0.004, lb = 0.75;
    E_1 (d = 1):  alpha = 0.5, beta = 0.5 (sigma = 2), dt = 0.002, target [0.75, 1.5], from x0 = -1.25 and from x0 = 1.75,
                  above rb, so that the rb side of the hit test decides.

4 alpha, x0 and sigma are exact in float32, so the kernels' float32 images and the reference's values coincide.  Each case
also replays the reference in the nearest wrong environments (alpha_0 or x0_0 broadcast to every coordinate, the sigma
of beta = 1) and asserts that the kernel falls outside the same tolerances there.  Swapped barriers need no replay: from
x0 = 1.75 a kernel that tested x >= rb and x <= lb would stop no trajectory, which the comparisons' own hit-pass checks
(and their share of finished trajectories) reject.  The tolerances are
those of test_gpu_fp64_reference.py, test_gpu_tabular_policy.py and test_gpu_bridge_hit.py where they hold in these
environments with a margin of 2 or more; the others are replaced below, each beside the largest value measured."""
import importlib.util
import json
import os

import numpy as np
import pytest
import torch

from oracle import reference_semantics as ref

pytestmark = pytest.mark.gpu


def _load(name):
    """a test module of this directory, loaded by path: tests/ is not a package"""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), name + ".py")
    spec = importlib.util.spec_from_file_location("_" + name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


FP = _load("test_gpu_fp64_reference")
BR = _load("test_gpu_bridge_hit")
TAB, BRIDGE = BR.TAB, BR.CPU             # test_gpu_tabular_policy, test_bridge_hit


@pytest.fixture(autouse=True)
def _no_schedule_overrides(monkeypatch):
    for name in ("FWD_QUANTUM", "FWD_HANDOFF", "BWD_WARP_SHARE", "FWD_BLOCKS_PER_SM", "BWD_KERNEL", "WIDE_KERNEL", "FWD_POLICY"):
        monkeypatch.delenv("RLSDE_" + name, raising=False)


def _mods():
    from rl_sde_is_b200 import _lib as L, rollout as R
    return L, R


def _cycle(values, d):
    return [values[i % len(values)] for i in range(d)]


def env_d(d):
    return dict(alpha=_cycle((0.5, 1.5, 0.75, 2.0), d), beta=2.0, dt=0.004, x0=_cycle((-1.25, -0.75, -1.5, -1.0), d),
                lb=0.75, rb=2.0)


E_1 = dict(alpha=0.5, beta=0.5, dt=0.002, x0=-1.25, lb=0.75, rb=1.5)
E_1_ABOVE = dict(E_1, x0=1.75)
ENVS = {"E_d": env_d, "E_1": lambda d: E_1, "E_1_above": lambda d: E_1_ABOVE}


def _wrong_envs(d, env):
    """the nearest wrong environments: what a kernel that misread one field of rlsde_env would compute"""
    w = {"sigma of beta = 1": dict(env, beta=1.0)}
    if d > 1:
        w["alpha_0 everywhere"] = dict(env, alpha=env["alpha"][0])
        w["x0_0 everywhere"] = dict(env, x0=env["x0"][0])
    return w


# Largest |error| / bound(C = 1) over every case of this file (both modes), measured on an NVIDIA B200 (1000 W power limit,
# max SM clock 1965 MHz), against the constants of test_gpu_fp64_reference.py (float32 state / float64 state):
#   G       0.055 / 0.0056 (C_G 2 / 0.3)         S   0.15 / 0.082 (C_S 2 / 0.3)      logw 0.25 / 0.056 (C_S 2 / 0.3)
#   l2      0.017 (C_L2 12)                       state path and float64-state l2: below, the default constants' margin
#   is under 2 here.  The wrong environments put the kernel outside these bounds on every finished trajectory.
C_ENV = {"path": (6.0, 1.0),      # 2.72 (K1 d = 10, E_d) / 0.49 (K1 d = 10, E_d): 2.2x / 2.0x
         "l2": (12.0, 0.015)}     # 0.017 / 0.0070 (K1, E_1 above rb): 700x / 2.1x
# max |g_kernel - g_f64| / max |g_f64|: GRAD_TOL of test_gpu_fp64_reference.py holds with a margin of 2 or more for K2m
# (3.0e-6, d = 10, ckpt 8), K2w (7.1e-7, d = 10) and the split (2.2e-7); not for the wide policies:
GRAD_TOL_ENV = {"K2x": 4e-6,      # 1.6e-6 (d = 1, H = 256, E_1), 2.5x
                "K2u": 4e-6}      # 1.8e-6 (d = 1, H = 256, E_1), 2.3x
# Share of trajectories within the float32-state tolerance of test_gpu_bridge_hit.py (1e-4 of 1 + |value|): 99.5 % there;
# under the table in E_1 0.992 (8 of 1 024 trajectories outside: paths that parted at a cell edge of the table, whose
# control jumps there; 2.5x more passes than at dt = 0.005 give 2.5x more edges to part at).  Every MLP family: 1.0.
BRIDGE_SHARE_TABLE_F32 = 0.98


def _output_wrong_envs(spec):
    """_wrong_envs for the kernels that store no path (table, bridge), which are told from a wrong environment by G, logw
    and hit decisions.  From above rb most trajectories stop within a few dozen passes, too few for the sigma of beta = 1
    to move G or logw beyond the tolerance on 90 % of them (measured 50 to 72 %; on [1.5, 2] u* of the default environment
    is 0, so G there depends on the hit pass alone); sigma is told apart from x0 = -1.25, where it moves every trajectory."""
    return {} if spec["x0"] > spec["rb"] else _wrong_envs(1, spec)


def _record(test, case, **values):
    """Measured ratios, one JSON line per case, appended to the file named by RLSDE_RATIO_LOG (if set)."""
    path = os.environ.get("RLSDE_RATIO_LOG")
    if path:
        with open(path, "a") as fh:
            fh.write(json.dumps(dict(test=test, case=case, **values)) + "\n")


def _ref_rule(L, rule):
    return ref.HIT_X0_IN_LB_RB if rule == L.HIT_X0_IN_LB_RB else ref.HIT_ALL_GE_LB


# ------------------------------------------------------------------------------ forward families
FWD_CASES = ([(f, d, H, "E_d") for f, d, H in FP.FWD_CASES if d > 1]
             + [(f, d, H, e) for f, d, H in FP.FWD_CASES if d == 1 for e in ("E_1", "E_1_above")])
HORIZON = 64          # passes the wrong-environment replays run (every trajectory, whether or not it stops earlier)


def _env_discriminates(out, params, family, d, H, f64, rule, env, lim=2000, K=128):
    """The kernel's path (or its hit pass) lies outside the tolerance of the reference replayed in each wrong environment on
    more than 90 % of the finished trajectories.  The replays are teacher-forced on the kernel's hit passes and run the
    first HORIZON passes."""
    L, R = _mods()
    prec = 1 if f64 else 0
    seed = 1000 * d + H
    noise = R.noise_fill(seed, K, d, lim, env["dt"])
    T = out.T.cpu().numpy().astype(np.int64)
    fin = T >= 0
    assert fin.sum() >= 64
    shares = {}
    for name, wrong in _wrong_envs(d, env).items():
        r = FP._reference(d, params, noise, wrong, hit_rule=_ref_rule(L, rule), hit_index=T, n_steps_lim=HORIZON,
                          f32_policy_input=f64, keep_path=True, device="cuda")
        n = np.minimum(np.where(fin, T, lim - 1), r["path"].shape[1] - 1)
        dev, store, _ = FP._path_deviation(out.path, r["path"], n)
        far = dev > store + FP._bound(n, 1.0, C_ENV["path"][prec])
        T_own = r["T_own"].cpu().numpy()
        decided = (T_own != T) & (T < HORIZON)
        shares[name] = float((far | decided)[fin].mean())
    assert all(v > 0.9 for v in shares.values()), (family, d, H, shares)
    return shares


@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("family,d,H,env_name", FWD_CASES)
def test_forward_kernel_matches_float64_reference(family, d, H, env_name, f64):
    """test_gpu_fp64_reference.test_forward_kernel_matches_float64_reference in E_d / E_1: both integral modes, state
    paths, hit passes, G, S, logw, l2 (d = 1) and the statistics record against the float64 reference, the nearest wrong
    answers of _discriminates, and the nearest wrong environments.  From above rb both modes use lb <= x <= rb (under
    all(x >= lb) every trajectory would stop on pass 0)."""
    L, _ = _mods()
    env = ENVS[env_name](d)
    above = d == 1 and env["x0"] > env["rb"]
    rule_exact = L.HIT_X0_IN_LB_RB if d == 1 else L.HIT_ALL_GE_LB
    rule_ref = L.HIT_X0_IN_LB_RB if (d == 1 and (f64 or above)) else L.HIT_ALL_GE_LB
    rx, rr = {}, {}
    out_x, r_x, params = FP._forward_case(family, d, H, f64, "exact", rule_exact, env=env, ratios=rx, tols=C_ENV)
    same_rule = rule_ref == rule_exact
    out_r, r_r, _ = FP._forward_case(family, d, H, f64, "reference", rule_ref, ref_out=r_x if same_rule else None, env=env,
                                     ratios=rr, tols=C_ENV)
    if same_rule:
        assert torch.equal(out_r.G, out_x.G) and torch.equal(out_r.T, out_x.T) and torch.equal(out_r.logw, out_x.logw)
    FP._discriminates(family, d, H, f64, out_r, r_r, out_x, r_x, params, dt=env["dt"])
    shares = _env_discriminates(out_x, params, family, d, H, f64, rule_exact, env)
    _record("forward", [family, d, H, env_name, f64], exact=rx, reference=rr, wrong_env_share=shares)


# ------------------------------------------------------------------------------ the table kernel (K1t)
def _env1(spec, h=0.01):
    """DoubleWellStoppingTime1D of a d = 1 spec, state space discretised with step h"""
    e, _ = FP._env_c(1, 0, spec)
    e.discretize_state_space(h)
    return e


@pytest.mark.parametrize("env_name", ["E_1", "E_1_above"])
@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("stoch_int", ["reference", "exact"])
def test_table_kernel_matches_float64_replay(env_name, f64, stoch_int):
    """rlsde_rollout_fwd_table under u* of the default environment (a smooth control on the h = 0.01 grid) in E_1:
    test_gpu_tabular_policy._fp64_case's comparison with the float64 table replay, then the wrong environments: G or logw
    outside the same bound, or the replay's own hit pass another, on more than 90 % of the finished trajectories."""
    L, R = _mods()
    spec = ENVS[env_name](1)
    env = _env1(spec)
    table = TAB._u_star(TAB._env(0.01))[1]
    K, lim, seed = 512, 4000, 5
    out, r, ok = TAB._fp64_case(table, env, f64, stoch_int, K=K, lim=lim, seed=seed)
    T = out.T.cpu().numpy().astype(np.int64)
    fin = T >= 0
    n = np.where(fin, T, lim - 1).astype(np.float64)
    noise = R.noise_fill(seed, K, 1, lim, env.dt)
    bound = lambda v: TAB.C_OUT[1 if f64 else 0] * (n + 1) * TAB.EPS32 * (1.0 + np.abs(v))
    shares = {}
    for name, wrong in _output_wrong_envs(spec).items():
        rw = TAB.rollout_reference_table(table, TAB._grid(env), noise, hit_index=T, device="cuda", **wrong)
        bad = (rw["T_own"].cpu().numpy() != T)
        for key in ("G", "logw"):
            bad |= np.abs(TAB._np(getattr(out, key)) - TAB._np(rw[key])) > bound(TAB._np(rw[key]))
        shares[name] = float(bad[fin].mean())
    _record("table", [env_name, f64, stoch_int], flip_share=float((~ok).mean()), wrong_env_share=shares)
    assert all(v > 0.9 for v in shares.values()), shares


# ------------------------------------------------------------------------------ the Brownian-bridge hit test
BRIDGE_CASES = [(fam, env_name, f64) for fam in BR.FAMILIES for env_name in ("E_1", "E_1_above") for f64 in (False, True)]


@pytest.mark.parametrize("family,env_name,f64", BRIDGE_CASES)
def test_bridge_against_float64_replay(family, env_name, f64):
    """Every d = 1 family with bridge=True in E_1 against the float64 bridge replay (tests/test_bridge_hit.py) on the
    kernel's increments, teacher-forced on its hit passes, with test_gpu_bridge_hit's tolerances: float32 state with the
    exact integral on in-kernel Philox noise, float64 state with the reference integral on injected noise.  sigma = 2 puts
    4x today's sigma^2 into the crossing exponent; from above rb the crossings at rb decide.  Wrong environment (the sigma
    of beta = 1, from x0 = -1.25): G or logw outside the tolerance, or an own decision of the replay against the forced
    one, on more than 90 % of the finished trajectories."""
    L, R = _mods()
    spec = ENVS[env_name](1)
    stoch_int, inject = ("reference", True) if f64 else ("exact", False)
    K, lim, seed = 1024, 2000, 77
    H, fkw = BR.FAMILIES[family]
    noise = R.noise_fill(seed, K, 1, lim, spec["dt"])
    _, env_c = FP._env_c(1, L.HIT_X0_IN_LB_RB, spec)
    common = dict(seed=seed, n_steps_lim=lim, state_f64=f64, stoch_int=stoch_int, noise=noise if inject else None,
                  bridge=True)
    if family == "table":
        table, grid = TAB._u_star(TAB._env(0.01))[1], (-2.0, 2.0, 0.01)
        out = R.rollout_forward_table(env_c, table, K, grid=grid, **common)
        pol = BRIDGE.table_policy(table, grid)
    else:
        out = R.rollout_forward(env_c, L.make_mlp(1, H), BR._policy(H)[1], K, **common, **fkw)
        pol = BRIDGE.mlp_policy(BR._policy(H)[0], f32_input=True)
    T = out.T.cpu().numpy()
    fin = T >= 0
    assert fin.mean() > 0.9
    nz = noise.cpu().numpy()
    r = BRIDGE.bridge_replay(pol, nz, seed=seed, hit_index=T, device="cuda", **spec)
    knife = r["knife"].cpu().numpy()
    assert (np.isnan(knife) | (knife < (1e-5 if f64 else 1e-3))).all(), (family, np.nanmax(knife))
    assert np.isnan(knife).mean() > 0.99, (family, np.isnan(knife).mean())
    S_key = "S_exact" if stoch_int == "exact" else "S_ref"
    atol = 1e-6 if f64 else 1e-4
    q = {}
    for key, ref_key in (("G", "G"), ("S", S_key), ("logw", "logw")):
        want = r[ref_key].cpu().numpy()
        err = np.abs(getattr(out, key).double().cpu().numpy() - want) / (1.0 + np.abs(want))
        q[key] = float(np.quantile(err, 0.995))
        share = BRIDGE_SHARE_TABLE_F32 if (family == "table" and not f64) else 0.995
        assert (err <= atol).mean() >= share, (family, key, float(err.max()), float((err <= atol).mean()))
    shares = {}
    for name, wrong in _output_wrong_envs(spec).items():
        rw = BRIDGE.bridge_replay(pol, nz, seed=seed, hit_index=T, device="cuda", **wrong)
        bad = ~np.isnan(rw["knife"].cpu().numpy())
        for key in ("G", "logw"):
            want = rw[key].cpu().numpy()
            bad |= np.abs(getattr(out, key).double().cpu().numpy() - want) > atol * (1.0 + np.abs(want))
        shares[name] = float(bad[fin].mean())
    _record("bridge", [family, env_name, f64], q995=q, knife_max=float(np.nan_to_num(knife).max()), wrong_env_share=shares)
    assert all(v > 0.9 for v in shares.values()), (family, shares)


# ------------------------------------------------------------------------------ reverse families
BWD_CASES = ([(f, d, H, c, "E_d") for f, d, H, c in FP.BWD_CASES if d > 1]
             + [(f, d, H, c, "E_1") for f, d, H, c in FP.BWD_CASES if d == 1])
BWD_LIM = {"E_d": 1500, "E_1": 1000}      # budgets in which more than 90 % of the trajectories hit


@pytest.mark.parametrize("family,d,H,ckpt,env_name", BWD_CASES)
def test_reverse_pass_matches_float64_autograd(family, d, H, ckpt, env_name):
    """Every reverse family in both integral modes against float64 autograd in E_d / E_1, within GRAD_TOL of
    test_gpu_fp64_reference.py (GRAD_TOL_ENV for the wide policies); the exact-mode gradient told apart from the
    reference-mode float64 one.  The yardstick is sensitive to each field: float64 autograd of the whole rollout with
    alpha_0 or x0_0 broadcast (d >= 2), or with the sigma of beta = 1 (d = 1), lies more than 10 tol from the kernel's
    gradient.  That a reverse pass whose forward is right and whose adjoint alone misreads alpha (the Hessian term
    c4a_f[k] (3 x^2 - 1)) fails the GRAD_TOL assertion is shown by deliberately wrong builds (profiles/r08)."""
    env = ENVS[env_name](d)
    wrong = {k: v for k, v in _wrong_envs(d, env).items() if (d > 1) != k.startswith("sigma")}
    errs, wrong_mode, wrong_env = FP._grad_case(family, d, H, ckpt, lim=BWD_LIM[env_name], env=env, wrong_envs=wrong)
    tol = GRAD_TOL_ENV.get(family, FP.GRAD_TOL[family])
    _record("reverse", [family, d, H, ckpt, env_name], errs=errs, ratio=max(errs.values()) / tol, wrong_mode=wrong_mode,
            wrong_env=wrong_env)
    assert errs["exact"] <= tol and errs["reference"] <= tol, (family, d, H, ckpt, errs)
    assert wrong_mode > 10 * tol, (family, d, H, ckpt, wrong_mode)
    assert all(v > 10 * tol for v in wrong_env.values()), (family, d, H, ckpt, wrong_env)


@pytest.mark.parametrize("bulk,d", [("K2m", 2), ("K2m", 3)])
def test_reverse_pass_split_between_families(bulk, d):
    """The split of a large batch between the warp reverse kernel (1 000 longest trajectories) and K2m, in E_d at
    d = 2 and 3, both integral modes, against float64 autograd."""
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    env = env_d(d)
    errs, wrong_mode, wrong_env = FP._grad_case(bulk, d, 32, 1, K=128 * n_sm + 200, lim=BWD_LIM["E_d"],
                                                extra_cfg={"bwd_warp_share": 1000}, env=env,
                                                wrong_envs={"alpha_0 everywhere": _wrong_envs(d, env)["alpha_0 everywhere"]})
    tol = FP.GRAD_TOL["split"]
    _record("split", [bulk, d], errs=errs, ratio=max(errs.values()) / tol, wrong_mode=wrong_mode, wrong_env=wrong_env)
    assert errs["exact"] <= tol and errs["reference"] <= tol, errs
    assert wrong_mode > 10 * tol and all(v > 10 * tol for v in wrong_env.values()), (wrong_mode, wrong_env)


# ------------------------------------------------------------------------------ single passes and the transition stream
STEP_ENVS = {"d3": dict(d=3, alpha=[0.5, 1.5, 0.75], beta=0.5, dt=0.004, lb=0.75, rb=2.0),
             "E_1": dict(d=1, alpha=0.5, beta=0.5, dt=0.002, lb=0.75, rb=1.5)}


@pytest.mark.parametrize("name", list(STEP_ENVS))
def test_env_step_per_coordinate(name):
    """rlsde_env_step (its own packer, not fill_env) through env.step / env.step_torch against env_step_numpy /
    env_step_torch given the alpha vector: float32 states into the NumPy path (float64 results, F_GRAD_F32), float64
    states (no F_GRAD_F32), and the torch path (float32); sigma = 2 in both environments, so a packer that dropped sigma
    (or used 1) would fail both.  Next states and done bit for bit; rewards exact at d = 1, and at
    d = 3 within 1e-7 (NumPy path) and 4 float32 ulps (torch path; measured 2.9 ulps): there the kernel squares the norm
    as sqrt(|u|^2)^2, torch's linalg.norm rounds differently.  The reward does not depend on alpha or sigma."""
    s = STEP_ENVS[name]
    d = s["d"]
    env, _ = FP._env_c(d, 0, {k: v for k, v in s.items() if k != "d"})
    rng = np.random.default_rng(d)
    K = 4096
    st32 = rng.uniform(-2.0, 2.0, (K, d)).astype(np.float32)
    st32[: K // 4] = rng.uniform(0.5, 1.8, (K // 4, d)).astype(np.float32)         # a share of states in the target
    act = rng.uniform(-3.0, 3.0, (K, d)).astype(np.float32)
    dbt = (np.sqrt(s["dt"]) * rng.standard_normal((K, d))).astype(np.float32)
    alpha = s["alpha"] if d == 1 else np.asarray(s["alpha"])
    step_kw = {} if d > 1 else dict(reward_type="state-action")
    for states in (st32, st32.astype(np.float64) + rng.uniform(-1e-3, 1e-3, (K, d))):
        nxt, r, done, _ = env.step(states, act, dbt=dbt, **step_kw)
        want_n, want_r, want_d = ref.env_step_numpy(d, alpha, s["beta"], s["dt"], states, act, dbt, lb=s["lb"], rb=s["rb"])
        assert nxt.dtype == np.float64 and np.array_equal(nxt, want_n), (name, states.dtype)
        assert np.array_equal(done, want_d) and 0.05 < done.mean() < 0.95
        if d == 1:
            assert np.array_equal(r, want_r)
        else:
            np.testing.assert_allclose(r, want_r, rtol=1e-7)
    nxt, r, done, _ = env.step_torch(torch.from_numpy(st32), torch.from_numpy(act), dbt=torch.from_numpy(dbt))
    want_n, want_r, want_d = ref.env_step_torch(d, alpha, s["beta"], s["dt"], torch.from_numpy(st32), torch.from_numpy(act),
                                                torch.from_numpy(dbt), lb=s["lb"])
    assert nxt.dtype == torch.float32 and torch.equal(nxt, want_n), name
    assert torch.equal(done, want_d)
    np.testing.assert_allclose(r.numpy(), want_r.numpy(), rtol=0 if d == 1 else 4 * 2.0 ** -23)


def test_transition_stream_per_coordinate():
    """rlsde_rollout_transitions in E_d at d = 2 against transitions_numpy fed the alpha and x0 vectors: the same tuples
    in the reference's pass-major order, done flags exact, float32 values within 1e-5 relative or 1e-5 absolute (the
    kernel's policy sums in another order than torch: states of up to 1 000 passes differ by up to 2.9e-6 where they
    cross zero; alpha_0 broadcast moves them by about 5e-3 per pass)."""
    L, R = _mods()
    env = env_d(2)
    _, env_c = FP._env_c(2, L.HIT_ALL_GE_LB, env)
    _, params, flat = FP._policy(2, 32, 2.5, 404)
    K, n_max = 64, 2000
    noise = R.noise_fill(404, K, 2, n_max, env["dt"])
    tr = R.rollout_transitions(env_c, L.make_mlp(2, 32), flat, K, n_max=n_max, noise=noise, order="reference")
    want = ref.transitions_numpy(2, np.asarray(env["alpha"]), env["beta"], env["dt"], params, noise.cpu().numpy(), n_max,
                                 lb=env["lb"], rb=env["rb"], x0=np.asarray(env["x0"]))
    assert int(tr.done.sum()) == K
    assert np.array_equal(tr.done.cpu().numpy(), want["done"])
    assert np.all(tr.states.cpu().numpy()[:K] == np.asarray(env["x0"], dtype=np.float32))
    for key in ("states", "actions", "rewards", "next_states"):
        np.testing.assert_allclose(getattr(tr, key).cpu().numpy(), want[key], rtol=1e-5, atol=1e-5, err_msg=key)
