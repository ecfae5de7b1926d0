"""The float64 yardstick and the environment packing away from the default environment, on the CPU.

oracle.reference_semantics.rollout_reference is pinned on the reference's fixtures (tests/test_reference_f64.py) at
alpha = 1 in every coordinate for d >= 2 and x0 = -1 everywhere; tests/test_gpu_env_params.py holds every kernel to it
with per-coordinate alpha and x0, beta != 1, a shifted lb and a start above rb.  Here the yardstick is compared with a
plain NumPy float64 loop in exactly those environments, its gradients with central finite differences, and the
environment packing (rollout.env_struct, _lib.make_env) with the values it is given."""
import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import reference_semantics as ref


def _params(d, H, bias, seed):
    from rl_sde_is_b200.models import DeterministicPolicy
    torch.manual_seed(seed)
    m = DeterministicPolicy(d, d, [H, H], nn.Tanh())
    m.policy[4].bias.data.fill_(bias)
    return {k: v.detach().clone() for k, v in m.state_dict().items()}


def _numpy_rollout(params, noise, alpha, beta, dt, x0, lb, rb, two):
    """The rollout the kernels compute, written out pass by pass in float64 NumPy, drift alpha_i 4 x_i (x_i^2 - 1) per
    coordinate: hit test on x_k (lb <= x_0 <= rb if ``two``, else all(x >= lb)), u_k, accumulators, Euler-Maruyama step."""
    W = [np.asarray(params[k].numpy(), dtype=np.float64) for k in ref.PARAM_KEYS]
    n_pass, K, d = noise.shape
    a = np.broadcast_to(np.asarray(alpha, dtype=np.float64), (d,))
    sigma = np.sqrt(2.0 / beta)
    x = np.tile(np.broadcast_to(np.asarray(x0, dtype=np.float64), (d,)), (K, 1))
    out = {k: np.zeros(K) for k in ("G", "S_exact", "S_ref")}
    out["T"] = np.full(K, -1)
    path = np.full((K, n_pass, d), np.nan)
    G, S = np.zeros(K), np.zeros(K)
    alive = np.ones(K, dtype=bool)
    for k in range(n_pass):
        path[:, k] = x                     # a stopped trajectory keeps its last state
        hit = ((x[:, 0] >= lb) & (x[:, 0] <= rb)) if two else (x >= lb).all(axis=1)
        u = np.tanh(np.tanh(x @ W[0].T + W[1]) @ W[2].T + W[3]) @ W[4].T + W[5]
        dB = noise[k].astype(np.float64)
        stop = alive & hit
        out["T"][stop] = k
        out["G"][stop], out["S_exact"][stop] = G[stop], S[stop]
        out["S_ref"][stop] = S[stop] + (u * dB).sum(axis=1)[stop]
        alive &= ~stop
        G = np.where(alive, G - (1.0 + 0.5 * (u * u).sum(axis=1)) * dt, G)
        S = np.where(alive, S + (u * dB).sum(axis=1), S)
        x = np.where(alive[:, None], x + (-(a * 4.0 * x * (x * x - 1.0)) + sigma * u) * dt + sigma * dB, x)
    for key, v in (("G", G), ("S_exact", S), ("S_ref", S)):
        out[key] = np.where(out["T"] >= 0, out[key], v)
    out["logw"] = out["G"] - out["S_exact"]
    return out, path


def _cycle(values, d):
    return [values[i % len(values)] for i in range(d)]


# (d, alpha, x0, beta, dt, lb, rb, two-sided hit rule)
YARDSTICK_CASES = [
    (1, 0.5, -1.25, 0.5, 0.002, 0.75, 1.5, True),
    (1, 0.5, 1.75, 0.5, 0.002, 0.75, 1.5, True),          # starts above rb: the rb side of the hit test decides
    (1, 0.75, -1.5, 2.0, 0.004, 0.75, 2.0, False),
    (3, [0.5, 1.5, 0.75], [-1.25, -0.75, -1.5], 2.0, 0.004, 0.75, 2.0, False),
    (3, [2.0, 0.5, 1.5], [-1.0, -1.25, -0.75], 0.5, 0.002, 0.75, 2.0, False),
    (10, _cycle((0.5, 1.5, 0.75, 2.0), 10), _cycle((-1.25, -0.75, -1.5, -1.0), 10), 2.0, 0.004, 0.75, 2.0, False),
]


@pytest.mark.parametrize("d,alpha,x0,beta,dt,lb,rb,two", YARDSTICK_CASES)
def test_reference_rollout_matches_numpy_loop(d, alpha, x0, beta, dt, lb, rb, two):
    """rollout_reference with per-coordinate alpha and x0, beta = 0.5 / 2, a shifted lb and (d = 1) a start above rb:
    hit passes equal, states along the path, G, S_exact, S_ref and logw within 1e-12 of the NumPy loop.  The coordinates
    differ, so a yardstick that used coordinate 0's alpha or x0 everywhere would fail, and most trajectories hit within
    the budget (the hit test is exercised)."""
    rng = np.random.default_rng(d * 100 + int(10 * beta))
    K, n_pass = 24, 700
    noise = (np.sqrt(dt) * rng.standard_normal((n_pass, K, d))).astype(np.float32)
    params = _params(d, 32, 2.5 if d > 1 else 1.0, 5 + d)
    rule = ref.HIT_X0_IN_LB_RB if two else ref.HIT_ALL_GE_LB
    got = ref.rollout_reference(d, alpha, beta, dt, params, noise, hit_rule=rule, lb=lb, rb=rb, x0=x0, keep_path=True)
    want, path = _numpy_rollout(params, noise, alpha, beta, dt, x0, lb, rb, two)
    T = got["T"].numpy()
    assert np.array_equal(T, want["T"])
    assert (T >= 0).mean() > 0.5 and (T > 0).any()
    for key in ("G", "S_exact", "S_ref", "logw"):
        assert np.abs(got[key].numpy() - want[key]).max() <= 1e-12 * (1.0 + np.abs(want[key]).max()), key
    p = got["path"].numpy()
    assert np.abs(p - path[:, :p.shape[1]]).max() <= 1e-12
    if np.ndim(alpha):
        # coordinate 0's alpha broadcast is another rollout
        other, _ = _numpy_rollout(params, noise, alpha[0], beta, dt, x0, lb, rb, two)
        assert np.abs(other["G"] - want["G"]).max() > 1e-6


def test_gradients_match_central_differences():
    """One grad_modes entry per parameter block, both modes, d = 2 with per-coordinate alpha and x0, beta = 2, lb = 0.75:
    autograd of mean(-G - sg(G) S) against a central difference of the float64 loss along the hit passes of the unperturbed
    rollout (sg(G) held at its unperturbed value).  The parameters are float32, so the difference quotient divides by the
    float32 perturbation actually applied."""
    d, alpha, x0, beta, dt = 2, [0.5, 1.5], [-1.25, -0.75], 2.0, 0.004
    kw = dict(lb=0.75, x0=x0)
    rng = np.random.default_rng(3)
    noise = (np.sqrt(dt) * rng.standard_normal((400, 32, d))).astype(np.float32)
    params = _params(d, 32, 3.0, 11)
    base = ref.rollout_reference(d, alpha, beta, dt, params, noise, grad_modes=("exact", "reference"), **kw)
    T = base["T"].numpy()
    assert (T >= 0).mean() > 0.8
    G0 = base["G"].numpy()
    done = T >= 0
    for key in ref.PARAM_KEYS:
        idx = np.unravel_index(int(np.argmax(np.abs(base["grads"]["exact"][key]))), params[key].shape)
        theta = float(params[key][idx])
        vals = []
        for sign in (1.0, -1.0):
            p = {k: v.clone() for k, v in params.items()}
            p[key][idx] = theta + sign * 1e-3
            r = ref.rollout_reference(d, alpha, beta, dt, p, noise, hit_index=T, **kw)
            vals.append((float(p[key][idx]), r["G"].numpy(), r["S_exact"].numpy(), r["S_ref"].numpy()))
        (tp, Gp, Sxp, Srp), (tm, Gm, Sxm, Srm) = vals
        for mode, Sp, Sm in (("exact", Sxp, Sxm), ("reference", Srp, Srm)):
            fd = np.where(done, -(Gp - Gm) - G0 * (Sp - Sm), 0.0).sum() / T.size / (tp - tm)
            g = base["grads"][mode][key][idx]
            assert abs(g - fd) <= 1e-5 * abs(g) + 1e-9, (key, mode, g, fd)


def test_env_struct_packs_per_coordinate_values():
    """rollout.env_struct / _lib.make_env copy a per-coordinate env.alpha and state_init into rlsde_env unchanged, with
    sigma, dt, lb, rb and the hit rule; coordinates past d are zero.  A scalar alpha is broadcast."""
    from rl_sde_is_b200 import _lib as L, rollout as R
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D, DoubleWellStoppingTimeND
    d = 5
    env = DoubleWellStoppingTimeND(d, beta=2.0, alpha=1.0, dt=0.004)
    env.alpha = np.array([0.5, 1.5, 0.75, 2.0, 1.25])
    env.alpha_tensor = torch.tensor(env.alpha, dtype=torch.float32)
    env.state_init = np.array([[-1.25, -0.75, -1.5, -1.0, -0.5]], dtype=np.float32)
    env.lb, env.rb = 0.75, 1.75
    e = R.env_struct(env, L.HIT_ALL_GE_LB)
    assert e.d == d and e.hit_rule == L.HIT_ALL_GE_LB
    assert list(e.alpha[:d]) == list(env.alpha) and list(e.x0[:d]) == list(env.state_init[0].astype(np.float64))
    assert all(v == 0.0 for v in e.alpha[d:]) and all(v == 0.0 for v in e.x0[d:])
    assert (e.sigma, e.dt, e.lb, e.rb) == (1.0, 0.004, 0.75, 1.75)
    one = DoubleWellStoppingTime1D(beta=0.5, alpha=0.5, dt=0.002)
    one.state_init = np.array([[1.75]], dtype=np.float32)
    e1 = R.env_struct(one, L.HIT_X0_IN_LB_RB)
    assert (e1.d, e1.hit_rule, e1.alpha[0], e1.x0[0], e1.sigma, e1.dt) == (1, L.HIT_X0_IN_LB_RB, 0.5, 1.75, 2.0, 0.002)
    assert list(L.make_env(3, 0.75, 1.0, 0.004, 1.0, 2.0, [-1.0, -1.25, -1.5], 0).alpha[:3]) == [0.75] * 3
