"""Tabulated 1-D controls (models.TabularPolicy, rlsde_rollout_fwd_table) on the CPU: the lookup against the environment's
own index function, the float64 table rollout (the yardstick of tests/test_gpu_tabular_policy.py) against a plain NumPy
loop, the argument checks of the C entry point and the refusal to train a table."""
from unittest import mock

import numpy as np
import pytest
import torch

from oracle import reference_semantics as ref

DT = 0.005


def _env(h=0.01, dt=DT):
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D
    env = DoubleWellStoppingTime1D(beta=1.0, alpha=1.0, dt=dt)
    env.discretize_state_space(h)
    return env


def rollout_reference_table(table, table_grid, noise, *, hit_rule=ref.HIT_X0_IN_LB_RB, alpha=1.0, beta=1.0, dt=DT, **kw):
    """oracle.reference_semantics.rollout_reference (d = 1, by default alpha = beta = 1, dt = 0.005) with the control
    u = table[idx(x)], idx(x) = floor((clip(x, lo, hi) - lo) / h) clamped to the table, in place of the MLP: the lookup
    sees the state in the replay's precision, everything else is the replay's arithmetic.  ``table_grid = (lo, hi, h)``;
    the ``grid=`` of rollout_reference belongs to its ``policy_opt``."""
    lo, hi, h = (float(v) for v in table_grid)
    kw.setdefault("device", "cpu")
    dtype = kw.get("dtype", torch.float64)
    tab = torch.as_tensor(np.asarray(table, dtype=np.float32).reshape(-1)).to(device=kw["device"], dtype=dtype)

    def lookup(_params, x):
        gi = torch.floor((x[:, 0].clamp(lo, hi) - lo) / h).long().clamp(0, tab.numel() - 1)
        return tab[gi][:, None]

    with mock.patch.object(ref, "policy_torch", lookup):
        return ref.rollout_reference(1, alpha, beta, dt, {}, noise, hit_rule=hit_rule, **kw)


def test_forward_is_the_environment_index():
    """forward(x) = actions[env.get_state_idx_truncate(x)]: every point of the h = 0.01 grid (about a fifth of them,
    rounded to three decimals, floor into the cell below), points outside [-2, 2], x = 2 exactly and random points."""
    from rl_sde_is_b200.models import TabularPolicy
    env = _env()
    actions = np.random.default_rng(0).normal(size=(env.n_states, 1)).astype(np.float32)
    pol = TabularPolicy(env, actions)
    grid_pts = env.state_space_h.reshape(-1, 1)
    below = env.get_state_idx_truncate(grid_pts) != np.arange(env.n_states)
    assert 0.1 < below.mean() < 0.3
    x = np.concatenate([grid_pts, [[-7.5], [-2.0000001], [2.0], [2.0000001], [3.0], [1e6], [-1e6]],
                        np.random.default_rng(1).uniform(-2.5, 2.5, (1000, 1))])
    want = actions[env.get_state_idx_truncate(x)]
    assert np.array_equal(pol(x).numpy(), want)
    assert np.array_equal(pol(torch.as_tensor(x)).numpy(), want)
    assert pol(np.array([[2.0]])).item() == actions[-1, 0]
    # the DP form: a 1-D action array indexed by the greedy action of each state
    env.set_action_space_bounds(); env.discretize_action_space(0.01)
    idx = np.random.default_rng(2).integers(0, env.n_actions, env.n_states)
    dp = TabularPolicy(env, env.action_space_h[idx])
    assert np.array_equal(dp(grid_pts).numpy()[:, 0], env.action_space_h[idx][env.get_state_idx_truncate(grid_pts)].astype(np.float32))
    with pytest.raises(ValueError):
        TabularPolicy(env, actions[:-1])


def _numpy_table_rollout(table, grid, noise, lb=1.0, rb=2.0, x0=-1.0):
    """The NumPy path of the reference, written out pass by pass for one trajectory at a time (float64 state)."""
    lo, hi, h = grid
    sigma = np.sqrt(2.0)
    n_pass, K, _ = noise.shape
    out = {k: np.zeros(K) for k in ("G", "S_exact", "S_ref", "logw")}
    out["T"] = np.full(K, -1)
    for i in range(K):
        x, G, S = x0, 0.0, 0.0
        for k in range(n_pass):
            gi = min(max(int(np.floor((min(max(x, lo), hi) - lo) / h)), 0), len(table) - 1)
            u = float(table[gi])
            dB = float(noise[k, i, 0])
            if lb <= x <= rb:
                out["T"][i] = k
                out["S_ref"][i] = S + u * dB
                break
            G += -(1.0 + 0.5 * u * u) * DT
            S += u * dB
            x = x + (-(4.0 * x * (x * x - 1.0)) + sigma * u) * DT + sigma * dB
        out["G"][i], out["S_exact"][i], out["logw"][i] = G, S, G - S
        if out["T"][i] < 0:
            out["S_ref"][i] = S
    return out


def test_reference_table_rollout_matches_numpy_loop():
    """The float64 table replay against the plain loop on injected increments: same hit passes, G / S / logw to 1e-12."""
    rng = np.random.default_rng(5)
    K, n_pass = 48, 1500
    noise = (np.sqrt(DT) * rng.standard_normal((n_pass, K, 1))).astype(np.float32)
    grid = (-2.0, 2.0, 0.05)
    table = (1.5 * np.cos(np.linspace(-2.0, 2.0, 81))).astype(np.float32)
    got = rollout_reference_table(table, grid, noise)
    want = _numpy_table_rollout(table, grid, noise.astype(np.float64))
    assert np.array_equal(got["T"].numpy(), want["T"])
    assert (want["T"] >= 0).sum() >= K // 2
    for key in ("G", "S_exact", "S_ref", "logw"):
        assert np.allclose(got[key].numpy(), want[key], rtol=0, atol=1e-12), key


def test_c_entry_point_argument_checks():
    """rlsde_rollout_fwd_table refuses bad arguments before it touches a device: d = 2 is unsupported; a null table,
    n_grid = 0 and grid_h = 0 (or NaN) are invalid."""
    from rl_sde_is_b200 import _lib as L
    lib = L.load()
    fake = 1 << 20                             # never dereferenced: every call below fails its argument checks first
    ws_bytes = int(lib.rlsde_workspace_bytes(64))

    def call(d=1, table=fake, n_grid=401, h=0.01):
        env = L.make_env(d, 1.0, np.sqrt(2.0), DT, 1.0, 2.0, np.full(d, -1.0), L.HIT_X0_IN_LB_RB)
        cfg = L.RlsdeRolloutCfg()
        cfg.K, cfg.K_global, cfg.n_steps_lim = 64, 64, 100
        cfg.n_grid, cfg.grid_lo, cfg.grid_hi, cfg.grid_h = n_grid, -2.0, 2.0, h
        return lib.rlsde_rollout_fwd_table(env, table, cfg, 0, 0, fake, fake, fake, 0, 0, 0, fake, ws_bytes, 0)

    RLSDE_ERR_INVALID_ARG, RLSDE_ERR_UNSUPPORTED = -1, -2
    assert call(d=2) == RLSDE_ERR_UNSUPPORTED
    assert call(table=0) == RLSDE_ERR_INVALID_ARG
    assert call(n_grid=0) == RLSDE_ERR_INVALID_ARG
    assert call(n_grid=-5) == RLSDE_ERR_INVALID_ARG
    assert call(h=0.0) == RLSDE_ERR_INVALID_ARG
    assert call(h=float("nan")) == RLSDE_ERR_INVALID_ARG


def test_training_refuses_a_table():
    """A table has no parameters: the training entry points raise before any launch (no device needed to see it)."""
    from rl_sde_is_b200 import _lib as L
    from rl_sde_is_b200.models import TabularPolicy
    from rl_sde_is_b200.reinforce_deterministic_core import _loss_and_grads_fused, sample_loss_vectorized
    env = _env()
    pol = TabularPolicy(env, np.zeros((env.n_states, 1)))
    assert list(pol.parameters()) == []
    with pytest.raises(L.RlsdeError, match="no gradient"):
        sample_loss_vectorized(env, pol, 16)
    with pytest.raises(L.RlsdeError, match="no gradient"):
        _loss_and_grads_fused(env, pol, 16)
