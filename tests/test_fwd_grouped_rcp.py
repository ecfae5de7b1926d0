"""The precise tanh of the tensor-core forward policy with one reciprocal per group of activations (rsig_group in
csrc/common.cuh): r = 1 / (2^z + 1) of four pre-activations of one row from one MUFU.RCP (G = 4) or two (G = 2).

The CPU tests restate the float32 arithmetic with correctly rounded EX2 / RCP and check it against float64 over
z in [-200, 200], including groups whose product would overflow float32 without the clamp; the unclamped form is shown to
be wrong there.  The GPU test compares every action a rollout records with the float64 policy at the recorded state."""
import numpy as np
import pytest
import torch
import torch.nn as nn

F32 = np.float32
ZMAX = {2: 63.0, 4: 31.0}
# |r - 1 / (2^z + 1)| <= ULPS[G] 2^-24 (r + 2^-31) + 2^-31 with correctly rounded EX2 / RCP (the 2^-31: the clamp)
ULPS = {1: 2.5, 2: 3.5, 4: 4.5}


def _ex2(z):
    with np.errstate(over="ignore"):
        return np.exp2(z.astype(np.float64)).astype(F32)


def _rcp(x):
    return (1.0 / x.astype(np.float64)).astype(F32)


def _grouped(z, G, clamp=True):
    """rsig_group on z[..., 0:4] = (za, zb) of one row, every operation rounded to float32."""
    z = z.astype(F32)
    if G == 1:
        return _rcp(_ex2(z) + F32(1))
    if clamp:
        z = np.minimum(z, F32(ZMAX[G]))
    with np.errstate(over="ignore", invalid="ignore"):
        d = _ex2(z) + F32(1)
        da, db = d[..., 0:2], d[..., 2:4]
        p = da * db
        if G == 2:
            q = _rcp(p)
        else:
            R = _rcp(p[..., 0] * p[..., 1])
            q = np.stack([R * p[..., 1], R * p[..., 0]], -1)
        return np.concatenate([q * db, q * da], -1)


def _groups():
    rng = np.random.default_rng(7)
    z = [rng.uniform(-200, 200, (200000, 4)), rng.uniform(-40, 40, (200000, 4))]
    big = rng.uniform(64, 200, (20000, 4))                  # z0 + z2 >= 128: the product overflows unclamped
    big[:, 1] = rng.uniform(-5, 5, 20000)
    big[:, 3] = rng.uniform(-5, 5, 20000)
    z.append(big)
    edge = np.array([[31, 31, 31, 31], [63, 63, 63, 63], [64, 64, -3, 0.5], [200, -200, 0, 128]], dtype=np.float64)
    z.append(edge)
    return np.concatenate(z).astype(F32)


@pytest.mark.parametrize("G", [1, 2, 4])
def test_grouped_reciprocal_is_within_its_bound(G):
    """Every r is finite and within ULPS[G] 2^-24 (r + 2^-31) + 2^-31 of 1 / (2^z + 1) in float64, over the whole range."""
    z = _groups()
    r = _grouped(z, G).astype(np.float64)
    assert np.isfinite(r).all()
    truth = 1.0 / (np.exp2(z.astype(np.float64)) + 1.0)
    err = np.abs(r - truth)
    assert (err <= ULPS[G] * 2.0 ** -24 * (truth + 2.0 ** -31) + 2.0 ** -31).all(), (err / (2.0 ** -24 * truth + 2.0 ** -31)).max()
    if G > 1:       # the bound is tight enough to tell the group's extra roundings from the ungrouped form's
        assert (err > ULPS[1] * 2.0 ** -24 * (truth + 2.0 ** -31) + 2.0 ** -31).any()


@pytest.mark.parametrize("G", [2, 4])
def test_grouped_reciprocal_without_the_clamp_is_wrong(G):
    """Without the clamp a group whose product overflows gives 0 or NaN for its smaller members."""
    z = _groups()
    r = _grouped(z, G, clamp=False).astype(np.float64)
    truth = 1.0 / (np.exp2(z.astype(np.float64)) + 1.0)
    with np.errstate(invalid="ignore"):
        bad = ~(np.abs(r - truth) <= ULPS[G] * 2.0 ** -24 * (truth + 2.0 ** -31) + 2.0 ** -31)
    assert bad.any()


# ------------------------------------------------------------------------------ GPU: recorded actions against float64
def _policy64(params, x):
    W1, b1 = params["policy.0.weight"].double().numpy(), params["policy.0.bias"].double().numpy()
    W2, b2 = params["policy.2.weight"].double().numpy(), params["policy.2.bias"].double().numpy()
    W3, b3 = params["policy.4.weight"].double().numpy(), params["policy.4.bias"].double().numpy()
    h1 = np.tanh(x[:, None] * W1[:, 0] + b1)
    h2 = np.tanh(h1 @ W2.T + b2)
    return (h2 @ W3.T + b3)[:, 0], h1, h2


def _action_bound(params, h1, h2):
    """First-order bound on the action error from a relative error eps = 8 x 2^-24 of every r (the grouped reciprocal with
    MUFU EX2 / RCP), the float16 hi / lo split of layer 2's operands (2^-22) and float32 accumulation (2^-21 of the
    magnitudes summed)."""
    W2, b2 = params["policy.2.weight"].double().numpy(), params["policy.2.bias"].double().numpy()
    W3, b3 = params["policy.4.weight"].double().numpy(), params["policy.4.bias"].double().numpy()
    s = 2.0 * np.log2(np.e)
    eps = 8 * 2.0 ** -24
    r1, r2 = (1 - h1) / 2, (1 - h2) / 2
    W2f = np.abs(2 * s * W2)                                                  # |folded layer-2 weights| [out][in]
    dz2 = (r1 * (eps + 2.0 ** -22)) @ W2f.T + 2.0 ** -21 * (np.abs(s * (b2 + W2.sum(1))) + r1 @ W2f.T) + 2.0 ** -31
    dr2 = eps * r2 + np.log(2) / 4 * dz2 + 2.0 ** -31
    W3f = np.abs(2 * W3[0])
    return dr2 @ W3f + 2.0 ** -21 * (np.abs(b3[0] + W3.sum()) + r2 @ W3f)


@pytest.mark.gpu
@pytest.mark.parametrize("state_f64", [False, True])
def test_recorded_actions_match_the_float64_policy(monkeypatch, state_f64):
    """rollout_transitions at d = 1, hidden width 32 takes the tensor-core policy (the same tuples as with it forced, others
    than with FFMA2); every recorded action is within _action_bound of the float64 policy at the recorded state, and the
    mean error is at most 1.5x that of the FFMA2 arithmetic on the states of a rollout with the same increments."""
    from rl_sde_is_b200 import _lib as L, rollout as R
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D
    from rl_sde_is_b200.models import DeterministicPolicy
    for name in ("FWD_QUANTUM", "FWD_HANDOFF", "FWD_BLOCKS_PER_SM", "FWD_POLICY"):
        monkeypatch.delenv("RLSDE_" + name, raising=False)
    torch.manual_seed(17)
    m = DeterministicPolicy(1, 1, [32, 32], nn.Tanh())
    m.policy[4].bias.data.fill_(0.5)
    params = {k: v.detach().clone() for k, v in m.state_dict().items()}
    flat = R.flat_parameters(m).detach().numpy()
    env_c = R.env_struct(DoubleWellStoppingTime1D(beta=1.0, alpha=1.0, dt=0.005), L.HIT_X0_IN_LB_RB)

    def run(policy):
        if policy is None:
            monkeypatch.delenv("RLSDE_FWD_POLICY", raising=False)
        else:
            monkeypatch.setenv("RLSDE_FWD_POLICY", policy)
        tr = R.rollout_transitions(env_c, L.make_mlp(1, 32), flat, 20000, seed=31, n_max=1000, state_f64=state_f64,
                                   order="trajectory")
        return tr.states.cpu().numpy()[:, 0].astype(np.float64), tr.actions.cpu().numpy()[:, 0].astype(np.float64)

    x_auto, u_auto = run(None)
    x_mma, u_mma = run("mma")
    assert np.array_equal(x_auto, x_mma) and np.array_equal(u_auto, u_mma)
    u64, h1, h2 = _policy64(params, x_mma)
    err = np.abs(u_mma - u64)
    bound = _action_bound(params, h1, h2)
    assert (err <= bound).all(), (err / bound).max()
    # FFMA2 on the same increments: its rollout visits the same states up to rounding, and is measured at its own
    x_ffma, u_ffma = run("ffma")
    assert not (len(u_ffma) == len(u_mma) and np.array_equal(u_ffma, u_mma))
    u64f, _, _ = _policy64(params, x_ffma)
    err_ffma = np.abs(u_ffma - u64f)
    assert err.mean() <= 1.5 * err_ffma.mean(), (err.mean(), err_ffma.mean())
