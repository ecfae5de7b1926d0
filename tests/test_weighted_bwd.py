"""The weighted reverse pass (rlsde_rollout_bwd_weighted, sample_returns_vectorized) on the CPU: its float64 yardstick,
the C ABI's refusals and the Python signature.

``weighted_grad_reference`` is the float64 autograd gradient of sum_k [T_k >= 0] (cG_k G_k + cS_k S_k) along given hit
passes: the rollout of oracle.reference_semantics.rollout_reference, teacher-forced, with the per-trajectory loss replaced.
It is pinned here against that function's own gradient (the case cG = -1, cS = -G) and against central differences;
tests/test_gpu_weighted_bwd.py holds every reverse kernel family to it."""
import inspect

import numpy as np
import pytest
import torch

from oracle import reference_semantics as ref

DT = 0.005


def _replay(d, alpha, beta, dt, p, noise, hit_index, x0):
    """(G, S_exact, S_ref) [K] of the float64 rollout with parameters ``p`` (dict of float64 tensors) and the stop forced on
    pass ``hit_index`` (-1 = none: such trajectories never stop and take no part in a loss)."""
    dev, dtype = noise.device, noise.dtype
    K = noise.shape[1]
    sigma, dt_ = float(np.sqrt(2.0 / beta)), float(dt)
    c4a = torch.as_tensor(np.broadcast_to(4.0 * np.asarray(alpha, dtype=np.float64), (d,)).copy(), device=dev, dtype=dtype)
    x = torch.as_tensor(np.broadcast_to(np.asarray(x0, dtype=np.float64), (d,)).copy(), device=dev, dtype=dtype).expand(K, d)
    zero = torch.zeros(K, device=dev, dtype=dtype)
    G, S, G_out, Sx_out, Sr_out = zero, zero, zero, zero, zero
    for k in range(int(hit_index.max()) + 1):
        u = ref.policy_torch(p, x)
        dB = noise[k]
        udB = (u * dB).sum(dim=1)
        stop = hit_index == k
        G_out = torch.where(stop, G, G_out)
        Sx_out = torch.where(stop, S, Sx_out)
        Sr_out = torch.where(stop, S + udB, Sr_out)
        alive = (hit_index > k) | (hit_index < 0)
        G = G + torch.where(alive, -(1.0 + 0.5 * (u * u).sum(dim=1)) * dt_, zero)
        S = S + torch.where(alive, udB, zero)
        x = torch.where(alive[:, None], x + (-(c4a * x * (x * x - 1.0)) + sigma * u) * dt_ + sigma * dB, x)
    return G_out, Sx_out, Sr_out


def _weighted_loss(d, alpha, beta, dt, p, noise, cG, cS, mode, hit_index, x0):
    G, Sx, Sr = _replay(d, alpha, beta, dt, p, noise, hit_index, x0)
    S = {"reference": Sr, "exact": Sx}[mode]
    cG = torch.as_tensor(np.asarray(cG, dtype=np.float64), device=noise.device)
    cS = torch.as_tensor(np.asarray(cS, dtype=np.float64), device=noise.device)
    return torch.where(hit_index >= 0, cG * G + cS * S, torch.zeros_like(G)).sum()


def weighted_grad_reference(d, alpha, beta, dt, params, noise, cG, cS, *, mode, hit_index, x0=-1.0, device="cpu"):
    """Flat float64 gradient (state_dict order) of sum_k [T_k >= 0] (cG_k G_k + cS_k S_k), S = S_ref (``mode="reference"``)
    or S_exact (``"exact"``), w.r.t. the float32 parameters ``params`` (state_dict), along the float32 increments
    ``noise[n_pass, K, d]`` with the stop of trajectory k forced on pass ``hit_index[k]``."""
    dev = torch.device(device)
    noise = torch.as_tensor(np.asarray(noise.cpu() if torch.is_tensor(noise) else noise, dtype=np.float32)).to(dev, torch.float64)
    hit = torch.as_tensor(np.asarray(hit_index.cpu() if torch.is_tensor(hit_index) else hit_index, dtype=np.int64), device=dev)
    p = {k: torch.as_tensor(np.asarray(v.detach().cpu().numpy() if torch.is_tensor(v) else v, dtype=np.float32))
         .to(dev, torch.float64).requires_grad_(True) for k, v in params.items()}
    loss = _weighted_loss(d, alpha, beta, dt, p, noise, cG, cS, mode, hit, x0)
    gs = torch.autograd.grad(loss, [p[k] for k in ref.PARAM_KEYS])
    return np.concatenate([g.detach().cpu().numpy().reshape(-1) for g in gs]).astype(np.float64)


def _case(d, K=24, lim=1000, seed=5):
    from rl_sde_is_b200.models import DeterministicPolicy
    torch.manual_seed(seed)
    m = DeterministicPolicy(d, d, [8, 8], torch.nn.Tanh())
    m.policy[4].bias.data.fill_(2.0 if d == 1 else 3.0)
    params = {k: v.detach().clone() for k, v in m.state_dict().items()}
    noise = (np.random.default_rng(seed).standard_normal((lim, K, d)) * np.sqrt(DT)).astype(np.float32)
    return params, noise


@pytest.mark.parametrize("d", [1, 2])
@pytest.mark.parametrize("mode", ["reference", "exact"])
def test_yardstick_special_case_is_the_surrogate_gradient(d, mode):
    """With cG = -1 and cS = -G the yardstick is rollout_reference's gradient of mean(-G - sg(G) S), times K."""
    params, noise = _case(d)
    K = noise.shape[1]
    r = ref.rollout_reference(d, 1.0, 1.0, DT, params, noise, grad_modes=(mode,))
    T, G = r["T"].numpy(), r["G"].numpy()
    assert (T >= 0).all()
    want = np.concatenate([r["grads"][mode][k].reshape(-1) for k in ref.PARAM_KEYS])
    got = weighted_grad_reference(d, 1.0, 1.0, DT, params, noise, -np.ones(K), -G, mode=mode, hit_index=T) / K
    assert np.abs(got - want).max() <= 1e-14 * np.abs(want).max()


@pytest.mark.parametrize("d", [1, 2])
@pytest.mark.parametrize("mode", ["reference", "exact"])
def test_yardstick_matches_central_differences(d, mode):
    """Random weights (mixed signs, magnitudes over six binades, exact zeros): the yardstick against central differences
    of sum_k (cG_k G_k + cS_k S_k) with the hit passes held fixed."""
    params, noise = _case(d, K=8, lim=1000, seed=9)
    K = noise.shape[1]
    T = ref.rollout_reference(d, 1.0, 1.0, DT, params, noise)["T"].numpy()
    assert (T >= 0).all()
    rng = np.random.default_rng(3)
    cG, cS = (rng.choice([-1.0, 1.0], K) * 10.0 ** rng.uniform(-3, 3, K) * (rng.random(K) > 0.2) for _ in range(2))
    g = weighted_grad_reference(d, 1.0, 1.0, DT, params, noise, cG, cS, mode=mode, hit_index=T)
    noise64 = torch.as_tensor(noise, dtype=torch.float64)
    hit = torch.as_tensor(T, dtype=torch.int64)
    base = {k: v.to(torch.float64) for k, v in params.items()}
    offs = np.cumsum([0] + [base[k].numel() for k in ref.PARAM_KEYS])
    h = 1e-6
    for flat in np.random.default_rng(4).choice(offs[-1], 16, replace=False):
        i = int(np.searchsorted(offs, flat, side="right") - 1)
        key = ref.PARAM_KEYS[i]
        f = []
        for s in (1.0, -1.0):
            p = dict(base)
            p[key] = base[key].clone().reshape(-1)
            p[key][flat - offs[i]] += s * h
            p[key] = p[key].reshape(base[key].shape)
            f.append(float(_weighted_loss(d, 1.0, 1.0, DT, p, noise64, cG, cS, mode, hit, -1.0)))
        fd = (f[0] - f[1]) / (2 * h)
        assert abs(fd - g[flat]) <= 1e-6 * np.abs(g).max(), (key, flat, fd, g[flat])


def test_c_abi_refusals():
    """rlsde_rollout_bwd_weighted refuses before any device work: a NULL coefficient pointer, RLSDE_F_HIT_BRIDGE and a
    missing RLSDE_F_STORE_PATH (RLSDE_ERR_INVALID_ARG), float64 state and hidden width 48 (RLSDE_ERR_UNSUPPORTED)."""
    from rl_sde_is_b200 import _lib as L
    lib = L.load()
    fake = 1 << 20                             # never dereferenced: every call below fails its argument checks first
    params = np.zeros(1 + 48 + 48 * 48 + 48 + 48 + 1 + 64, dtype=np.float32)
    RLSDE_ERR_INVALID_ARG, RLSDE_ERR_UNSUPPORTED = -1, -2

    def call(flags, cG=fake, cS=fake, H=32):
        c = L.RlsdeRolloutCfg()
        c.K, c.K_global, c.n_steps_lim, c.flags = 64, 64, 100, flags
        c.ckpt_every, c.ckpt_stride = 1, 100
        env = L.make_env(1, 1.0, np.sqrt(2.0), DT, 1.0, 2.0, np.full(1, -1.0), L.HIT_ALL_GE_LB)
        return lib.rlsde_rollout_bwd_weighted(env, L.make_mlp(1, H), params.ctypes.data, c, 0, cG, cS, fake, fake, 0, 1.0,
                                              fake, fake, 1 << 40, 0)

    P = L.F_STORE_PATH
    assert call(P, cG=0) == RLSDE_ERR_INVALID_ARG
    assert call(P, cS=0) == RLSDE_ERR_INVALID_ARG
    assert call(P | L.F_HIT_BRIDGE) == RLSDE_ERR_INVALID_ARG
    assert call(0) == RLSDE_ERR_INVALID_ARG
    assert call(P | L.F_STATE_F64) == RLSDE_ERR_UNSUPPORTED
    assert call(P, H=48) == RLSDE_ERR_UNSUPPORTED


def test_sample_returns_signature():
    """The reference-compatible positional arguments, the rollout extras as keywords, and no shard or bridge option."""
    from rl_sde_is_b200.reinforce_deterministic_core import sample_returns_vectorized
    sig = inspect.signature(sample_returns_vectorized)
    assert list(sig.parameters)[:3] == ["env", "model", "K"]
    kw = {n: p.default for n, p in sig.parameters.items() if p.kind is inspect.Parameter.KEYWORD_ONLY}
    assert kw == dict(noise=None, seed=None, n_steps_lim=10**6, tanh="precise", stoch_int="reference", ckpt_every=None,
                      device=None, kernel="auto")
    assert "bridge" not in sig.parameters and "dist" not in sig.parameters


def test_sample_returns_frees_the_rollout(monkeypatch):
    """After backward() and with the outputs dropped, nothing keeps the rollout (its checkpoint path) alive: the autograd
    node must not hold the tensors it returns, or G, S, the node and the rollout form a cycle that gc.collect() does not
    break.  The launches are replaced by stand-ins on the CPU; tests/test_gpu_weighted_bwd.py repeats this on the device."""
    import gc
    import weakref
    from rl_sde_is_b200 import reinforce_deterministic_core as core, rollout as R
    K, P = 8, 5
    refs, coefs = [], []

    def fake_forward(env_c, mlp_c, params_host, K, **kw):
        out = R.RolloutOut(G=torch.randn(K), S=torch.randn(K), T=torch.full((K,), 3, dtype=torch.int32), l2=None, logw=None,
                           path=torch.zeros(K, 4, 1), stats_dev=torch.zeros(13, dtype=torch.float64))
        refs.append(weakref.ref(out.path))
        return out

    def fake_backward(env_c, mlp_c, params_host, fwd, loss_scale, *, coef, **kw):
        coefs.append(coef)
        return torch.ones(P)

    monkeypatch.setattr(R, "rollout_forward", fake_forward)
    monkeypatch.setattr(R, "rollout_backward", fake_backward)
    flat = torch.zeros(P, requires_grad=True)
    for _ in range(3):
        G, S = core._ReturnsWithAux.apply(flat, None, None, K, {}, {})
        want = torch.autograd.grad(torch.var(G - S, unbiased=False), [G, S], retain_graph=True)
        torch.var(G - S, unbiased=False).backward()
        assert all(torch.equal(a, b) for a, b in zip(coefs[-1], want))
        del G, S, want
    gc.collect()
    assert len(refs) == 3 and all(r() is None for r in refs)
    assert torch.equal(flat.grad, torch.full((P,), 3.0))
