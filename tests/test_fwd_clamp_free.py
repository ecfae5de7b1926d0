"""The clamp-free precise tanh of the tensor-core forward policy (d = 1, hidden width 32).

rsig_group clamps each pre-activation z to 31 before MUFU.EX2, so that a product of four 2^z + 1 cannot overflow.  Where the
clamp cannot bind it is the identity, and the forward rollout leaves it out (fwd_mma_clamp_bounds in csrc/mlp_mma.cuh):
  * layer 2, for the whole launch, when the host proves every z2 <= 30 (its inputs r lie in [0, 1]);
  * layer 1, per warp and pass, when every state of the warp satisfies |x| <= X1, the host's bound for z1 <= 30.

The CPU tests check the host bounds (rlsde_fwd_mma_clamp_bounds) against brute force over the folded, pre-scaled image.
The GPU test scales policies until the layer-2 bound exceeds 30 and X1 lies inside the states the trajectories visit, so
that the clamped kernel and the per-warp fallback run and the clamp binds; every output must then equal, bit for bit, that
of the warp-per-trajectory continuation, which keeps the clamp everywhere."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn as nn

SAFE_Z = 30.0
TWO_LOG2E = 2.8853900817779268


def _policy(seed, w1_scale=1.0, w2_scale=1.0):
    from rl_sde_is_b200 import rollout as R
    from rl_sde_is_b200.models import DeterministicPolicy
    np.random.seed(seed)
    torch.manual_seed(seed)
    m = DeterministicPolicy(1, 1, [32, 32], nn.Tanh())
    with torch.no_grad():
        m.policy[0].weight.mul_(w1_scale)
        m.policy[2].weight.mul_(w2_scale)
    return np.ascontiguousarray(R.flat_parameters(m).detach().numpy(), dtype=np.float32)


def _bounds(flat):
    from rl_sde_is_b200 import _lib as L
    out = (ctypes.c_double * 2)()
    assert L.load().rlsde_fwd_mma_clamp_bounds(flat.ctypes.data_as(ctypes.c_void_p), out) == 0
    return out[0], out[1]


def _folded(flat):
    """pack_mlp_const_folded restated: W1', b1' (layer 1) and W2' [out][in], b2' (layer 2) as float32, in float64."""
    f = flat.astype(np.float64)
    W1, b1, W2, b2 = f[:32], f[32:64], f[64:1088].reshape(32, 32), f[1088:1120]
    s = TWO_LOG2E
    W1f = (s * W1).astype(np.float32).astype(np.float64)
    b1f = (s * b1).astype(np.float32).astype(np.float64)
    W2f = -2.0 * (s * W2).astype(np.float32).astype(np.float64)
    b2f = (s * (b2 + W2.sum(axis=1))).astype(np.float32).astype(np.float64)
    return W1f, b1f, W2f, b2f


def _check_bounds(flat):
    z2_max, x1_max = _bounds(flat)
    W1, b1, W2, b2 = _folded(flat)
    rng = np.random.default_rng(0)
    # layer 2: r in [0, 1]^32.  Random points and the vertices around the maximiser stay below the bound; the maximiser
    # (r_k = 1 where W2'_nk > 0) attains it.
    r = rng.random((20000, 32))
    r[:32] = (W2 > 0)[np.argmax(b2 + np.where(W2 > 0, W2, 0).sum(axis=1))] ^ np.eye(32, dtype=bool)
    assert (r @ W2.T + b2).max() <= z2_max * (1 + 1e-12) + 1e-12
    assert np.isclose((b2 + np.where(W2 > 0, W2, 0).sum(axis=1)).max(), z2_max, rtol=1e-9, atol=1e-9)
    # layer 1 (d = 1): z1 = b1' + W1' x <= 30 on a grid of |x| <= X1, and it reaches 30 at x = +-X1
    if x1_max < 0:
        assert (b1 > SAFE_Z).any()
        return z2_max, x1_max
    assert x1_max > 0
    xs = np.concatenate([np.linspace(-x1_max, x1_max, 4001), [-x1_max, x1_max]])
    z1 = b1[None, :] + W1[None, :] * xs[:, None]
    assert z1.max() <= SAFE_Z * (1 + 1e-12)
    assert np.isclose(z1.max(), SAFE_Z, rtol=1e-9)
    beyond = np.array([-x1_max, x1_max]) * (1 + 1e-6)
    assert (b1[None, :] + W1[None, :] * beyond[:, None]).max() > SAFE_Z
    return z2_max, x1_max


def test_bounds_of_the_headline_policy():
    """bench.py's policy (seed 1): the clamp-free layer 2 applies, and layer 1 is clamp-free far beyond the double well."""
    z2_max, x1_max = _check_bounds(_policy(1))
    assert z2_max <= SAFE_Z and x1_max > 3.0


@pytest.mark.parametrize("seed", [2, 5, 11])
@pytest.mark.parametrize("w1_scale,w2_scale", [(1.0, 1.0), (40.0, 1.0), (1.0, 6.0), (300.0, 20.0)])
def test_bounds_against_brute_force(seed, w1_scale, w2_scale):
    _check_bounds(_policy(seed, w1_scale, w2_scale))


def test_bounds_with_a_large_bias():
    """A layer-1 bias above 30 leaves no state for which layer 1 is clamp-free."""
    flat = _policy(3)
    flat[32 + 7] = 12.0                     # b1 of unit 7: 12 * 2 log2(e) > 30
    assert _check_bounds(flat)[1] < 0


# ------------------------------------------------------------------------------ GPU: every path against the clamped one
@pytest.fixture
def _no_schedule_overrides(monkeypatch):
    for name in ("FWD_QUANTUM", "FWD_HANDOFF", "FWD_BLOCKS_PER_SM", "FWD_POLICY"):
        monkeypatch.delenv("RLSDE_" + name, raising=False)


def _scaled_policy(seed, clamp_layer2):
    """A policy whose layer-1 bound X1 is 1.3 (inside the visited states: the well at -1 reaches beyond -1.3, and there z1
    exceeds 31) and whose layer-2 bound is 2x above 30 (clamp_layer2) or at most 30."""
    flat = _policy(seed)
    z2, x1 = _bounds(flat)
    g = 2.0 * SAFE_Z / z2 if clamp_layer2 else 1.0
    flat = _policy(seed, w1_scale=x1 / 1.3, w2_scale=g)
    z2, x1 = _bounds(flat)
    assert (z2 > SAFE_Z) == clamp_layer2
    assert 1.2 < x1 < 1.4
    return flat


@pytest.mark.gpu
@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("clamp_layer2", [False, True])
def test_clamp_free_paths_match_the_clamped_continuation(f64, clamp_layer2, _no_schedule_overrides):
    from rl_sde_is_b200 import _lib as L, rollout as R
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D
    flat = _scaled_policy(7, clamp_layer2)
    env_c = R.env_struct(DoubleWellStoppingTime1D(beta=1.0, alpha=1.0, dt=0.005), L.HIT_X0_IN_LB_RB)
    K, lim = 40000, 2000

    def run(handoff):
        return R.rollout_forward(env_c, L.make_mlp(1, 32), flat, K, seed=123, n_steps_lim=lim, stoch_int="exact",
                                 state_f64=f64, want_logw=True, kernel="thread",
                                 tuning={"fwd_policy": "mma", "fwd_quantum": -1, "fwd_handoff": handoff})

    k1 = run(-1)           # the whole rollout in K1: clamp-free where proven, clamped elsewhere
    cont = run(K)          # after the first passes every trajectory moves to the continuation, which always clamps
    assert torch.isfinite(k1.G).all() and torch.isfinite(k1.S).all()
    for name in ("G", "S", "T", "logw"):
        assert torch.equal(getattr(k1, name), getattr(cont, name)), name
