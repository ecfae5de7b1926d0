"""The Brownian-bridge hit test between passes (RLSDE_F_HIT_BRIDGE, d = 1) on the GPU.

1. Coupling: with the same seed a bridge rollout and a plain one share every increment, so on every d = 1 family the
   bridge only ends trajectories earlier, and a trajectory it does not end earlier is bit for bit the plain one.
2. Every family against the float64 bridge replay (tests/test_bridge_hit.py) on the kernel's increments, teacher-forced
   on the kernel's hit passes, in both state precisions and integral modes, with Philox and injected noise.
3. Outputs do not depend on the batch size, the traj_offset shard or the schedule of the thread-per-trajectory kernel.
4. Science: with the bridge the IS estimate under u* converges to Psi(-1) at O(dt), u = 0, u* and the DP greedy table
   agree, and the mean first hitting time moves by O(dt) when dt is halved.

Tolerances are written beside the values measured on an NVIDIA B200 (profiles/r07)."""
import importlib.util
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

pytestmark = pytest.mark.gpu

DT = 0.005


def _load(name):
    """a test module of this directory, loaded by path: tests/ is not a package"""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), name + ".py")
    spec = importlib.util.spec_from_file_location("_" + name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


CPU = _load("test_bridge_hit")
TAB = _load("test_gpu_tabular_policy")


@pytest.fixture(autouse=True)
def _no_schedule_overrides(monkeypatch):
    for name in ("FWD_QUANTUM", "FWD_HANDOFF", "BWD_WARP_SHARE", "FWD_BLOCKS_PER_SM", "BWD_KERNEL", "WIDE_KERNEL", "FWD_POLICY"):
        monkeypatch.delenv("RLSDE_" + name, raising=False)


def _mods():
    from rl_sde_is_b200 import _lib as L, rollout as R
    return L, R


def _n_sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


# family -> (hidden width, rollout_forward keywords); "table" is rlsde_rollout_fwd_table under u* on the h = 0.01 grid
FAMILIES = {
    "K1-mma": (32, dict(kernel="thread", tuning={"fwd_policy": "mma", "fwd_handoff": -1})),
    "K1-ffma": (32, dict(kernel="thread", tuning={"fwd_policy": "ffma", "fwd_handoff": -1})),
    "K1w": (32, dict(kernel="warp")),
    "K1u-32": (32, dict(kernel="tensor")),
    "K1x-64": (64, dict(tuning={"wide_kernel": "ffma"})),
    "K1u-64": (64, dict(tuning={"wide_kernel": "umma"})),
    "K1x-128": (128, dict(tuning={"wide_kernel": "ffma"})),
    "K1u-128": (128, dict(tuning={"wide_kernel": "umma"})),
    "K1x-256": (256, dict(tuning={"wide_kernel": "ffma"})),
    "K1u-256": (256, dict(tuning={"wide_kernel": "umma"})),
    "table": (None, {}),
}
_params = {}


def _policy(H):
    if H not in _params:
        from rl_sde_is_b200.models import DeterministicPolicy
        from rl_sde_is_b200 import rollout as R
        torch.manual_seed(7 + H)
        m = DeterministicPolicy(1, 1, [H, H], nn.Tanh())
        m.policy[4].bias.data.fill_(1.0)
        _params[H] = ({k: v.detach().numpy().copy() for k, v in m.state_dict().items()},
                      R.flat_parameters(m).detach().numpy())
    return _params[H]


def _run(family, K, *, bridge, seed=31, lim=3000, f64=False, stoch_int="exact", noise=None, tanh="precise", **kw):
    L, R = _mods()
    H, fkw = FAMILIES[family]
    fkw = dict(fkw)
    if "tuning" in kw:
        fkw["tuning"] = {**fkw.get("tuning", {}), **kw.pop("tuning")}
    if family == "table":
        env = TAB._env(0.01)
        fkw.pop("tuning", None)
        return R.rollout_forward_table(R.env_struct(env, L.HIT_X0_IN_LB_RB), TAB._u_star(env)[1], K, grid=TAB._grid(env),
                                       seed=seed, n_steps_lim=lim, state_f64=f64, stoch_int=stoch_int, noise=noise,
                                       bridge=bridge, **kw)
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D
    env = DoubleWellStoppingTime1D(beta=1.0, alpha=1.0, dt=DT)
    return R.rollout_forward(R.env_struct(env, L.HIT_X0_IN_LB_RB), L.make_mlp(1, H), _policy(H)[1], K, seed=seed,
                             n_steps_lim=lim, state_f64=f64, stoch_int=stoch_int, noise=noise, tanh=tanh, bridge=bridge,
                             **fkw, **kw)


def _K(family):
    return 16 * _n_sm() + 512 if family.startswith("K1-") or family == "K1u-32" else 2048


# ------------------------------------------------------------------------------ 1. coupling
@pytest.mark.parametrize("tanh", ["precise", "fast"])
@pytest.mark.parametrize("family", list(FAMILIES))
def test_bridge_only_ends_trajectories_earlier(family, tanh):
    if family == "table" and tanh == "fast":
        pytest.skip("a table has no tanh")
    K = _K(family)
    on = _run(family, K, bridge=True, tanh=tanh)
    off = _run(family, K, bridge=False, tanh=tanh)
    big = np.iinfo(np.int32).max
    Tb, To = on.T.cpu().numpy(), off.T.cpu().numpy()
    Tb_, To_ = np.where(Tb < 0, big, Tb), np.where(To < 0, big, To)
    assert (Tb_ <= To_).all(), family
    assert (Tb_ < To_).mean() > 0.05, (family, (Tb_ < To_).mean())
    same = torch.as_tensor(Tb == To, device=on.T.device)
    for key in ("G", "S", "logw"):
        assert torch.equal(getattr(on, key)[same], getattr(off, key)[same]), (family, key)


# ------------------------------------------------------------------------------ 2. float64 replay
REPLAY_CASES = [(fam, f64, si, inj) for fam in FAMILIES for f64 in (False, True)
                for si, inj in (("exact", False), ("reference", True))]


@pytest.mark.parametrize("family,f64,stoch_int,inject", REPLAY_CASES)
def test_against_float64_bridge_replay(family, f64, stoch_int, inject):
    """Kernel against the float64 bridge replay on the kernel's own increments (noise_fill for Philox, or the injected
    array), teacher-forced on the kernel's hit passes.  A forced pass is a knife edge: the replay's own decision there
    was within rounding of the other side (|margin| of the grid test, |U - p| of a draw); none occurred in the measured
    run.  |error| / (1 + |value|) of G, S and logw for 99.5 % of the trajectories: below 1e-4 with float32 state (largest
    measured 99.5 % quantile 2.5e-5, logw under the table, whose lookup can fall into the neighbouring cell; 8e-6 or less
    under an MLP) and below 1e-6 with float64 state (measured 2.1e-7, S of K1 with the FFMA2 policy).  Per case:
    profiles/r07/science.jsonl ("replay" rows)."""
    L, R = _mods()
    K, lim, seed = 1024 if not family.startswith(("K1-", "K1u-32")) else _K(family), 2000, 77
    noise = R.noise_fill(seed, K, 1, lim, DT) if inject else None
    out = _run(family, K, bridge=True, seed=seed, lim=lim, f64=f64, stoch_int=stoch_int, noise=noise)
    nz = (noise if inject else R.noise_fill(seed, K, 1, lim, DT)).cpu().numpy()
    T = out.T.cpu().numpy()
    if family == "table":
        env = TAB._env(0.01)
        pol = CPU.table_policy(TAB._u_star(env)[1], TAB._grid(env))
    else:
        pol = CPU.mlp_policy(_policy(FAMILIES[family][0])[0], f32_input=True)
    r = CPU.bridge_replay(pol, nz, seed=seed, hit_index=T, device="cuda")
    knife = r["knife"].cpu().numpy()
    tol_knife = 1e-3 if not f64 else 1e-5
    assert (np.isnan(knife) | (knife < tol_knife)).all(), (family, np.nanmax(knife))
    assert np.isnan(knife).mean() > 0.99, (family, np.isnan(knife).mean())
    S_key = "S_exact" if stoch_int == "exact" else "S_ref"
    atol = 1e-4 if not f64 else 1e-6
    for key, ref_key in (("G", "G"), ("S", S_key), ("logw", "logw")):
        err = np.abs(getattr(out, key).double().cpu().numpy() - r[ref_key].cpu().numpy())
        scale = 1.0 + np.abs(r[ref_key].cpu().numpy())
        assert (err <= atol * scale).mean() >= 0.995, (family, key, float(np.max(err / scale)))


# ------------------------------------------------------------------------------ 3. invariance
def _schedule_counters(K):
    _, R = _mods()
    ws = R._workspace(torch.device("cuda", torch.cuda.current_device()), K)
    return ws[:48].view(torch.int64).cpu().numpy()


@pytest.mark.parametrize("f64", [False, True])
def test_outputs_do_not_depend_on_batch_shard_or_schedule(f64):
    """Bit for bit: a small batch against the head of a large one; two traj_offset shards against the whole batch; at the
    headline size (more than 128 x SMs trajectories: persistent grid), time slices of 8 passes and run-to-completion with
    the last 4 000 live trajectories handed to the warp kernel (RESUME) against the adaptive schedule.  The workspace
    counters show that each schedule engaged.  The table kernel: batch and shard."""
    K, lim = 128 * _n_sm() + 5000, 800
    kw = dict(lim=lim, f64=f64, seed=5)
    keys = ("G", "S", "T", "logw")

    def same(a, b, sl=slice(None)):
        for key in keys:
            assert torch.equal(getattr(a, key), getattr(b, key)[sl]), key

    for family in ("K1-mma", "table"):
        base = dict(FAMILIES[family][1])
        full = _run(family, K, bridge=True, **kw)
        same(_run(family, 1000, bridge=True, **kw), full, slice(0, 1000))
        half = K // 2
        for off in (0, half):
            same(_run(family, half, bridge=True, traj_offset=off, K_global=K, **kw), full, slice(off, off + half))
        if family != "table":
            assert base["tuning"]["fwd_handoff"] == -1
            same(_run(family, K, bridge=True, tuning={"fwd_quantum": 8}, **kw), full)
            q = _schedule_counters(K)
            assert q[1] > K and q[3] == 0
            same(_run(family, K, bridge=True, tuning={"fwd_quantum": -1, "fwd_handoff": 4000}, **kw), full)
            q = _schedule_counters(K)
            assert 0 < q[1] <= 4000 and q[3] >= q[1]


# ------------------------------------------------------------------------------ 4. science
def _is(env, policy, K=1_000_000, seed=2024, bridge=True):
    from rl_sde_is_b200.approximate_methods import is_estimate
    st = is_estimate(env, policy, K, n_steps_lim=10**5, seed=seed, bridge=bridge)
    assert st["n_unfinished"] == 0
    return st["is_mean"], st["is_mean"] * st["is_rel_error"] / np.sqrt(K)


def test_u_star_converges_to_psi_at_order_dt():
    """u* tabulated on h = 0.001, beta = 1, x0 = -1, K = 1e6, seed 2024, with the bridge, at dt = 0.01, 0.005, 0.0025.
    Measured on an NVIDIA B200 (1000 W power limit; profiles/r07/science.jsonl), Psi(-1) = 0.164016:
        m = 0.164509 (+0.300 %), 0.164287 (+0.165 %), 0.164179 (+0.099 %), standard errors 2.7e-5, 1.9e-5, 1.3e-5;
        bias ratios 1.82 and 1.67 (an O(dt) bias gives 2; the grid test gives 1.38);
        Richardson 2 m(0.0025) - m(0.005) = 0.164070, 5.4e-5 = 1.7 standard errors above Psi.
    Without the bridge the same runs give -4.85 %, -3.59 %, -2.61 %.  Bounds: relative bias at dt = 0.005 below 0.4 %,
    both ratios in [1.6, 2.5], Richardson within 4 standard errors of Psi."""
    from rl_sde_is_b200.hjb_1d import HJBSolution1D
    from rl_sde_is_b200.models import TabularPolicy
    sol = HJBSolution1D(TAB._env(0.001))
    u = sol.policy_opt_table(TAB._env(0.001))
    psi = float(sol.psi_at(-1.0))
    m, se = {}, {}
    for dt in (0.01, 0.005, 0.0025):
        env = TAB._env(0.001, dt=dt)
        m[dt], se[dt] = _is(env, TabularPolicy(env, u))
    assert abs(m[0.005] / psi - 1.0) < 0.004, (m, psi)
    for a, b in ((0.01, 0.005), (0.005, 0.0025)):
        ratio = (m[a] - psi) / (m[b] - psi)
        assert 1.6 <= ratio <= 2.5, (a, ratio, m, psi)
    rich = 2 * m[0.0025] - m[0.005]
    assert abs(rich - psi) <= 4 * np.hypot(2 * se[0.0025], se[0.005]), (rich, psi, m)


def test_estimate_does_not_depend_on_the_policy():
    """dt = 0.01, bridge: u = 0 (budget 1e5 passes, nothing unfinished), u* and the DP greedy table agree within 4 combined
    standard errors: exp(G - S_exact) is the exact likelihood ratio of the process stopped by the bridge test.  Measured
    (B200, profiles/r07/science.jsonl): DP 0.164554 +- 2.7e-5, u = 0 0.164615 +- 2.0e-4, u* 0.164519 +- 2.7e-5."""
    from rl_sde_is_b200.models import TabularPolicy
    env = TAB._env(0.01, dt=0.01)
    m_dp, se_dp = _is(env, TabularPolicy(env, TAB._dp_greedy(TAB._env(0.01))), seed=1)
    m_0, se_0 = _is(env, TabularPolicy(env, np.zeros((env.n_states, 1))), seed=2)
    m_u, se_u = _is(env, TabularPolicy(env, TAB._u_star(env)[1]), seed=3)
    assert abs(m_dp - m_0) <= 4 * np.hypot(se_dp, se_0), (m_dp, m_0)
    assert abs(m_dp - m_u) <= 4 * np.hypot(se_dp, se_u), (m_dp, m_u)
    assert abs(m_u - m_0) <= 4 * np.hypot(se_u, se_0), (m_u, m_0)


def test_mean_hitting_time_moves_by_order_dt():
    """estimate_fht_vectorized under u* (h = 0.01), K = 1e6: with the bridge the mean first hitting time is smaller than
    with the grid test, and it changes far less when dt is halved (O(dt) against O(sqrt(dt))).  Measured (B200,
    profiles/r07/science.jsonl): grid test 1.15716 / 1.14783 / 1.14160 at dt = 0.01 / 0.005 / 0.0025, bridge 1.12438 /
    1.12415 / 1.12450: the bridge values agree within their sampling error, the grid ones fall by 0.0093 and 0.0062."""
    from rl_sde_is_b200.approximate_methods import estimate_fht_vectorized
    from rl_sde_is_b200.models import TabularPolicy
    f = {}
    for dt in (0.01, 0.005):
        env = TAB._env(0.01, dt=dt)
        pol = TabularPolicy(env, TAB._u_star(env)[1])
        for bridge in (False, True):
            f[dt, bridge] = estimate_fht_vectorized(env, pol, 1_000_000, k_max=10**5, seed=9, bridge=bridge)
    assert f[0.01, True] < f[0.01, False] and f[0.005, True] < f[0.005, False], f
    d_bridge = abs(f[0.01, True] - f[0.005, True])
    d_grid = abs(f[0.01, False] - f[0.005, False])
    assert d_bridge < 0.5 * d_grid, f
