"""The weighted reverse pass (rlsde_rollout_bwd_weighted) of every kernel family, and sample_returns_vectorized.

- With cG = -1 and cS = -G it is rlsde_rollout_bwd bit for bit, in every family, both integral modes and both tanh modes.
- With random per-trajectory coefficients (mixed signs, exact zeros, magnitudes over 1e-3 .. 1e3) it matches the float64
  yardstick of tests/test_weighted_bwd.py along the kernel's hit passes, within the families' GRAD_TOL of
  tests/test_gpu_fp64_reference.py (max |dg| / max |g|); swapping the two coefficients lands far outside.
- Through autograd, any loss over (G, S) trains: eff_loss reproduces sample_loss_vectorized, the log-variance loss
  matches the yardstick fed with autograd's coefficients, gradients accumulate."""
import importlib.util
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

pytestmark = pytest.mark.gpu


def _load(name):
    """a test module of this directory, loaded by path: tests/ is not a package"""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), name + ".py")
    spec = importlib.util.spec_from_file_location("_" + name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


FP = _load("test_gpu_fp64_reference")
EP = _load("test_gpu_env_params")
WB = _load("test_weighted_bwd")


@pytest.fixture(autouse=True)
def _no_schedule_overrides(monkeypatch):
    for name in ("FWD_QUANTUM", "FWD_HANDOFF", "BWD_WARP_SHARE", "FWD_BLOCKS_PER_SM", "BWD_KERNEL", "WIDE_KERNEL", "FWD_POLICY"):
        monkeypatch.delenv("RLSDE_" + name, raising=False)


def _mods():
    from rl_sde_is_b200 import _lib as L, rollout as R
    return L, R


def _dist(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


# The split case with random coefficients: max |dg| / max |g| 1.1e-6 (d = 1, exact mode; 7.0e-7 at d = 2; NVIDIA B200) against
# GRAD_TOL["split"] = 5e-7 measured with (-1, -G): with 19 144 trajectories whose coefficients span six binades, the float32
# partial sums of the largest contributions carry the error.  2.7x margin.
GRAD_TOL_SPLIT = 3e-6


def _coefs(K, seed, scale=1.0):
    """cG, cS: independent signs, ~20 % exact zeros, magnitudes log-uniform over 1e-3 .. 1e3 across trajectories."""
    rng = np.random.default_rng(seed)
    return tuple((rng.choice([-1.0, 1.0], K) * 10.0 ** rng.uniform(-3, 3, K) * (rng.random(K) > 0.2) * scale).astype(np.float32)
                 for _ in range(2))


class _Case:
    """One forward per (case, tanh mode), shared by the bitwise and the float64 checks (as _grad_case builds it)."""

    def __init__(self, family, d, H, ckpt, K=192, lim=400, extra_cfg=None, env=None, tanh="precise"):
        L, R = _mods()
        s = FP._spec(env)
        seed = 77 + 100 * d + H
        _, self.params, self.flat = FP._policy(d, H, 2.0 if d == 1 else 3.0, seed)
        _, self.env_c = FP._env_c(d, L.HIT_ALL_GE_LB, env)
        self.mlp_c = L.make_mlp(d, H)
        self.noise = R.noise_fill(seed, K, d, lim, s["dt"])
        fkw, cfg_set = FP.BWD_FAMILIES[family]
        self.fwd = R.rollout_forward(self.env_c, self.mlp_c, self.flat, K, noise=self.noise, n_steps_lim=lim, stoch_int="exact",
                                     store_path=True, ckpt_every=ckpt, want_logw=False, tanh=tanh, **fkw)
        self.T = self.fwd.T.cpu().numpy()
        assert (self.T >= 0).mean() > 0.9
        for k, v in {**cfg_set, **(extra_cfg or {})}.items():
            setattr(self.fwd.cfg, k, v)
        self.d, self.K, self.s = d, K, s

    def set_mode(self, mode):
        L, _ = _mods()
        f = self.fwd.cfg.flags
        self.fwd.cfg.flags = (f | L.F_STOCH_INT_EXACT) if mode == "exact" else (f & ~L.F_STOCH_INT_EXACT)

    def grad(self, coef=None, scale=1.0):
        _, R = _mods()
        if coef is not None:
            coef = tuple(torch.as_tensor(c, dtype=torch.float32, device=self.fwd.G.device).contiguous() for c in coef)
        return R.rollout_backward(self.env_c, self.mlp_c, self.flat, self.fwd, scale, noise=self.noise, coef=coef)

    def yardstick(self, cG, cS, mode):
        s = self.s
        return WB.weighted_grad_reference(self.d, s["alpha"], s["beta"], s["dt"], self.params, self.noise, cG, cS, mode=mode,
                                          hit_index=self.T, x0=s["x0"], device="cuda")


def _bitwise(case):
    """rlsde_rollout_bwd_weighted(-1, -G, 1/K) against rlsde_rollout_bwd(1/K) in both integral modes."""
    cG = torch.full_like(case.fwd.G, -1.0)
    cS = (-case.fwd.G).contiguous()
    for mode in ("exact", "reference"):
        case.set_mode(mode)
        a = case.grad(scale=1.0 / case.K)
        b = case.grad((cG, cS), scale=1.0 / case.K)
        assert torch.equal(a, b), (mode, (a - b).abs().max().item())


def _against_float64(case, tol, seed, scales=(1.0,), g_only=False):
    """Random coefficients in both modes against the yardstick; the swapped coefficients' yardstick is > 10 tol away.
    ``g_only``: every scale once more with cS = 0 (a loss over G alone: the coefficient of u dt alone sets the range)."""
    errs = {}
    for mode in ("exact", "reference"):
        case.set_mode(mode)
        for sc in scales + ((tuple(-s for s in scales)) if g_only else ()):
            cG, cS = _coefs(case.K, seed, abs(sc))
            if sc < 0:
                cS = np.zeros_like(cS)
            g = case.grad((cG, cS)).cpu().numpy().astype(np.float64)
            want = case.yardstick(cG, cS, mode)
            errs[(mode, sc)] = _dist(g, want)
            assert errs[(mode, sc)] <= tol, (mode, sc, errs)
            if sc == 1.0:
                wrong = _dist(g, case.yardstick(cS, cG, mode))
                assert wrong > 10 * tol, (mode, wrong)
    print("ratios", errs)
    return errs


@pytest.mark.parametrize("family,d,H,ckpt", FP.BWD_CASES)
def test_weighted_reverse_pass(family, d, H, ckpt):
    """Every reverse family: the special case bit for bit in both tanh modes; random coefficients against float64 (one
    shape per tensor-core family also with every coefficient scaled by 1e4 and by 1e-4, and with cS = 0)."""
    for tanh in ("fast", "precise"):
        case = _Case(family, d, H, ckpt, tanh=tanh)
        _bitwise(case)
    scaled = (family, d, H, ckpt) in (("K2m", 1, 32, 1), ("K2u", 1, 256, 1))
    _against_float64(case, FP.GRAD_TOL[family], seed=d + H + ckpt, scales=(1.0, 1e4, 1e-4) if scaled else (1.0,), g_only=scaled)


@pytest.mark.parametrize("bulk,d", [("K2m", 1), ("K2m", 2)])
def test_weighted_split_between_families(bulk, d):
    """Large batches with bwd_warp_share: the 1 000 longest trajectories on the warp kernel, the rest on K2m adding onto
    its gradient; bit for bit against rlsde_rollout_bwd, and against float64 with random coefficients."""
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    case = _Case(bulk, d, 32, 1, K=128 * n_sm + 200, lim=300, extra_cfg={"bwd_warp_share": 1000})
    _bitwise(case)
    _against_float64(case, GRAD_TOL_SPLIT, seed=11)


@pytest.mark.parametrize("family,d,H,env", [("K2m", 1, 32, "E_1"), ("K2u", 2, 128, "E_d")])
def test_weighted_non_default_environment(family, d, H, env):
    """One family at d = 1 in E_1 and one at d = 2 in E_d (tests/test_gpu_env_params.py): per-coordinate alpha and x0,
    beta != 1, shifted lb."""
    case = _Case(family, d, H, 1, lim=EP.BWD_LIM[env], env=EP.ENVS[env](d))
    _bitwise(case)
    _against_float64(case, EP.GRAD_TOL_ENV.get(family, FP.GRAD_TOL[family]), seed=21)


# ---------------------------------------------------------------------------------------------------- autograd API
def _model(seed=5, d=1, H=32):
    from rl_sde_is_b200.models import DeterministicPolicy
    torch.manual_seed(seed)
    m = DeterministicPolicy(d, d, [H, H], nn.Tanh())
    m.policy[4].bias.data.fill_(2.0)
    return m


def _env():
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D
    return DoubleWellStoppingTime1D(beta=1.0, alpha=1.0, dt=FP.DT)


def _pgrad(m):
    return torch.cat([p.grad.reshape(-1) for p in m.parameters()]).double().numpy()


def test_autograd_eff_loss_reproduces_sample_loss():
    """eff_loss written in torch over (G, S) gives sample_loss_vectorized's gradient (same seed)."""
    from rl_sde_is_b200.reinforce_deterministic_core import sample_loss_vectorized, sample_returns_vectorized
    env, K = _env(), 3000
    m1, m2 = _model(), _model()
    loss, G_np, ts = sample_loss_vectorized(env, m1, K, seed=17)
    loss.backward()
    G, S, ts2 = sample_returns_vectorized(env, m2, K, seed=17)
    assert G.is_cuda and S.is_cuda and G.shape == (K,) and G.grad_fn is not None
    np.testing.assert_array_equal(G.detach().cpu().numpy(), G_np)
    np.testing.assert_array_equal(ts, ts2)
    eff = torch.mean(-G - G.detach() * S)
    assert abs(float(eff) - float(loss)) <= 1e-6 * abs(float(loss))
    eff.backward()
    assert _dist(_pgrad(m2), _pgrad(m1)) <= 2 * FP.GRAD_TOL["K2m"]


def _api_case(loss_fn, stoch_int, K=192, lim=2000):
    """(p.grad after loss_fn(G, S).backward(), the float64 yardstick fed with autograd's dL/dG, dL/dS) on injected noise."""
    from rl_sde_is_b200.reinforce_deterministic_core import sample_returns_vectorized
    _, R = _mods()
    env, m = _env(), _model(seed=8)
    noise = R.noise_fill(31, K, 1, lim, FP.DT)
    G, S, ts = sample_returns_vectorized(env, m, K, noise=noise, stoch_int=stoch_int, n_steps_lim=lim)
    loss_fn(G, S).backward()
    Gd, Sd = G.detach().clone().requires_grad_(True), S.detach().clone().requires_grad_(True)
    cG, cS = torch.autograd.grad(loss_fn(Gd, Sd), [Gd, Sd], allow_unused=True)
    cG = np.zeros(K) if cG is None else cG.double().cpu().numpy()
    cS = np.zeros(K) if cS is None else cS.double().cpu().numpy()
    params = {k: v.detach().clone() for k, v in m.state_dict().items()}
    want = WB.weighted_grad_reference(1, 1.0, 1.0, FP.DT, params, noise, cG, cS,
                                      mode=stoch_int, hit_index=(ts - 1).astype(np.int64), device="cuda")
    return m, _pgrad(m), want


def test_autograd_log_variance_loss():
    """Var(G - S_exact): the gradient matches the float64 yardstick with the coefficients autograd produced."""
    _, g, want = _api_case(lambda G, S: torch.var(G - S, unbiased=False), "exact")
    assert _dist(g, want) <= FP.GRAD_TOL["K2w"]


def test_autograd_loss_over_G_only_and_accumulation():
    """A loss over G alone (S gets no gradient) works, and a second backward adds onto p.grad."""
    m, g, want = _api_case(lambda G, S: G.mean(), "reference")
    assert _dist(g, want) <= FP.GRAD_TOL["K2w"]
    from rl_sde_is_b200.reinforce_deterministic_core import sample_returns_vectorized
    _, R = _mods()
    G, S, _ = sample_returns_vectorized(_env(), m, 192, noise=R.noise_fill(31, 192, 1, 2000, FP.DT), n_steps_lim=2000)
    G.mean().backward()
    np.testing.assert_allclose(_pgrad(m), 2 * g, rtol=1e-6, atol=0)


def test_autograd_unfinished_raise():
    from rl_sde_is_b200 import _lib as L
    from rl_sde_is_b200.reinforce_deterministic_core import sample_returns_vectorized
    with pytest.raises(L.RlsdeError, match="did not reach the target set"):
        sample_returns_vectorized(_env(), _model(), 64, seed=3, n_steps_lim=5)


def test_autograd_frees_the_rollout(monkeypatch):
    """A training loop over sample_returns_vectorized keeps no rollout alive: after backward() and with G, S dropped, the
    checkpoint path of every iteration is freed."""
    import gc
    import weakref
    from rl_sde_is_b200.reinforce_deterministic_core import sample_returns_vectorized
    _, R = _mods()
    refs, forward = [], R.rollout_forward

    def recording_forward(*a, **kw):
        out = forward(*a, **kw)
        refs.append(weakref.ref(out.path))
        return out

    monkeypatch.setattr(R, "rollout_forward", recording_forward)
    m = _model()
    for it in range(3):
        G, S, _ = sample_returns_vectorized(_env(), m, 512, seed=40 + it, stoch_int="exact")
        torch.var(G - S, unbiased=False).backward()
        del G, S
    gc.collect()
    assert len(refs) == 3 and all(r() is None for r in refs)
