"""The ragged checkpoint store (rlsde_rollout_fwd_ragged / rlsde_rollout_bwd_ragged) on the GPU.

- Forward, every family: the store gathered into the dense layout is the dense store bit for bit over every checkpoint it
  holds; G, S, T and the statistics record are the dense forward's; nothing is written outside a trajectory's rows.
- Reverse, every family: with random coefficients the ragged pass is rlsde_rollout_bwd_weighted on the dense store bit
  for bit, with (-1, -G) it is rlsde_rollout_bwd.
- Python: where the dense store does not fit the budget, the training entry points take the ragged store and return the
  dense route's loss, returns, hit indices and gradient bit for bit."""
import gc
import importlib.util
import os
import weakref

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
CANARY = -12345.0


@pytest.fixture(autouse=True)
def _no_schedule_overrides(monkeypatch):
    for name in ("FWD_QUANTUM", "FWD_HANDOFF", "BWD_WARP_SHARE", "FWD_BLOCKS_PER_SM", "BWD_KERNEL", "WIDE_KERNEL", "FWD_POLICY"):
        monkeypatch.delenv("RLSDE_" + name, raising=False)


def _mods():
    from rl_sde_is_b200 import _lib as L, rollout as R
    return L, R


def _setup(d, H, seed):
    L, _ = _mods()
    _, _, flat = FP._policy(d, H, 2.0 if d == 1 else 3.0, seed)
    _, env_c = FP._env_c(d, L.HIT_ALL_GE_LB, None)
    return env_c, L.make_mlp(d, H), flat


def _ragged_like(dense, env_c, mlp_c, flat, K, C, counts=None, **kw):
    """The ragged forward with the dense forward's arguments; ``counts`` (rows per trajectory) defaults to the layout of
    the dense rollout's hit indices.  Returns (rollout, base)."""
    _, R = _mods()
    if counts is None:
        counts = R.ragged_ckpt_counts(dense.T, C)
    base, total = R.slot_offsets(counts)
    out = R.rollout_forward(env_c, mlp_c, flat, K, store_path=True, ckpt_every=C, want_logw=False, path_base=base,
                            n_slots=int(total), **kw)
    return out, base


# (family, d, H, C, rollout keywords): K1 in both policy arithmetics, with forced time slices and hand-off, K1w, K1x, K1u
def _fwd_cases():
    thread = lambda pol, **t: dict(kernel="thread", tuning=dict(fwd_policy=pol, **t))
    cases = []
    for C in (1, 4, 32):
        cases += [("K1 mma", 1, 32, C, thread("mma")), ("K1 ffma", 1, 32, C, thread("ffma"))]
        cases += [("K1", d, 32, C, dict(kernel="thread")) for d in (2, 10)]
    cases += [("K1w", d, 32, 1, dict(kernel="warp")) for d in (1, 2, 10)]
    cases += [("K1 slices", d, 32, 4, dict(kernel="thread", tuning=dict(fwd_quantum=8), K="big")) for d in (1, 2)]
    cases += [("K1 hand-off", 1, 32, 1, dict(kernel="thread", tuning=dict(fwd_quantum=0, fwd_handoff=3000, fwd_policy=p), K="big"))
              for p in ("mma", "ffma")]
    cases += [("K1x", d, H, 1, dict(tuning=dict(wide_kernel="ffma"))) for d in (1, 2) for H in (64, 128, 256)]
    cases += [("K1u", d, H, 1, dict(tuning=dict(wide_kernel="umma"))) for d in (1, 2) for H in (64, 128, 256)]
    cases += [("K1u", d, 32, C, dict(kernel="tensor")) for d in (2, 10) for C in (1, 32)]
    return cases


@pytest.mark.parametrize("family,d,H,C,kw", _fwd_cases(), ids=lambda v: str(v).replace(" ", "_") if not isinstance(v, dict) else "")
def test_forward_matches_dense_store(family, d, H, C, kw):
    L, R = _mods()
    kw = dict(kw)
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    K = 128 * n_sm + 500 if kw.pop("K", None) == "big" else 1500
    lim = 600
    env_c, mlp_c, flat = _setup(d, H, 5 + d + H + C)
    kw.update(seed=1234 + d, n_steps_lim=lim, stoch_int="exact")
    dense = R.rollout_forward(env_c, mlp_c, flat, K, store_path=True, ckpt_every=C, want_logw=False, **kw)
    rag, base = _ragged_like(dense, env_c, mlp_c, flat, K, C, **kw)
    for name in ("G", "S", "T", "stats_dev"):
        assert torch.equal(getattr(rag, name), getattr(dense, name)), name
    T = dense.T.to(torch.int64)
    assert (T >= 0).float().mean() > 0.5
    counts = R.ragged_ckpt_counts(T, C)
    traj = torch.repeat_interleave(torch.arange(K, device=T.device), counts)
    ci = torch.arange(int(counts.sum()), device=T.device) - torch.repeat_interleave(base[:-1], counts)
    assert torch.equal(rag.path[:int(counts.sum())], dense.path[traj, ci])

    # canary: every even finished trajectory gets one row fewer than it needs (its last checkpoint must be dropped), every
    # odd one a row of slack, and the store one row more at its end; the rows a trajectory does not write keep their
    # canary.  An unfinished trajectory with a row (odd ones) fills it with its checkpoint 0: it runs the whole budget.
    idx = torch.arange(K, device=T.device)
    alloc = torch.where(idx % 2 == 0, (counts - 1).clamp(min=0), counts + 1)
    base2, total2 = R.slot_offsets(alloc)
    n_rows = int(total2) + 1
    written = torch.where(T >= 0, torch.minimum(alloc, counts), alloc)
    rows = torch.arange(n_rows, device=T.device)
    owner = torch.searchsorted(base2, rows, right=True) - 1
    local = rows - base2[owner.clamp(max=K - 1)]
    inside = (owner < K) & (local < written[owner.clamp(max=K - 1)])
    buf = torch.full((n_rows, d), CANARY, dtype=torch.float32, device=T.device)
    lib = L.load()
    cfg = rag.cfg
    G, S, T3 = torch.empty_like(rag.G), torch.empty_like(rag.S), torch.empty_like(rag.T)
    ws = R._workspace(T.device, K)
    with torch.cuda.device(T.device):
        rc = lib.rlsde_rollout_fwd_ragged(env_c, mlp_c, np.ascontiguousarray(flat, dtype=np.float32).ctypes.data, cfg, 0,
                                          base2.data_ptr(), G.data_ptr(), S.data_ptr(), T3.data_ptr(), buf.data_ptr(), 0,
                                          ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
    L.check(rc, "rlsde_rollout_fwd_ragged")
    assert torch.equal(T3, dense.T)
    assert (buf[~inside] == CANARY).all()
    sel = rows[inside]
    assert torch.equal(buf[sel], dense.path[owner[sel], local[sel]])


def _bwd_pair(family, d, H, ckpt, K=192, lim=400, extra_cfg=None):
    L, R = _mods()
    seed = 77 + 100 * d + H
    env_c, mlp_c, flat = _setup(d, H, seed)
    noise = R.noise_fill(seed, K, d, lim, FP._spec(None)["dt"])
    fkw, cfg_set = FP.BWD_FAMILIES[family]
    kw = dict(noise=noise, n_steps_lim=lim, stoch_int="exact", **fkw)
    dense = R.rollout_forward(env_c, mlp_c, flat, K, store_path=True, ckpt_every=ckpt, want_logw=False, **kw)
    rag, _ = _ragged_like(dense, env_c, mlp_c, flat, K, ckpt, **kw)
    assert torch.equal(rag.T, dense.T) and torch.equal(rag.G, dense.G)
    for f in (dense, rag):
        for k, v in {**cfg_set, **(extra_cfg or {})}.items():
            setattr(f.cfg, k, v)
    return env_c, mlp_c, flat, noise, dense, rag


def _bwd_bitwise(env_c, mlp_c, flat, noise, dense, rag, seed):
    L, R = _mods()
    K = dense.T.numel()
    rng = np.random.default_rng(seed)
    cG, cS = (torch.as_tensor((rng.choice([-1.0, 1.0], K) * 10.0 ** rng.uniform(-3, 3, K)).astype(np.float32), device="cuda")
              for _ in range(2))
    for mode in ("exact", "reference"):
        for f in (dense, rag):
            f.cfg.flags = (f.cfg.flags | L.F_STOCH_INT_EXACT) if mode == "exact" else (f.cfg.flags & ~L.F_STOCH_INT_EXACT)
        a = R.rollout_backward(env_c, mlp_c, flat, dense, 1.0 / K, noise=noise, coef=(cG, cS))
        b = R.rollout_backward(env_c, mlp_c, flat, rag, 1.0 / K, noise=noise, coef=(cG, cS))
        assert torch.equal(a, b), (mode, (a - b).abs().max().item())
        a = R.rollout_backward(env_c, mlp_c, flat, dense, 1.0 / K, noise=noise)
        b = R.rollout_backward(env_c, mlp_c, flat, rag, 1.0 / K, noise=noise)
        assert torch.equal(a, b), (mode, (a - b).abs().max().item())


@pytest.mark.parametrize("family,d,H,ckpt", FP.BWD_CASES)
def test_reverse_matches_dense_store(family, d, H, ckpt):
    env_c, mlp_c, flat, noise, dense, rag = _bwd_pair(family, d, H, ckpt)
    _bwd_bitwise(env_c, mlp_c, flat, noise, dense, rag, seed=d + H + ckpt)


@pytest.mark.parametrize("bulk,d", [("K2m", 1), ("K2m", 2)])
def test_reverse_split_between_families(bulk, d):
    """The longest trajectories on the warp kernel, the rest on K2m."""
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    pair = _bwd_pair(bulk, d, 32, 1, K=128 * n_sm + 200, lim=300, extra_cfg={"bwd_warp_share": 1000})
    _bwd_bitwise(*pair, seed=3)


def _model(d, H, seed):
    """A policy with a drift towards the target (head bias 1.5), so that every trajectory finishes within the budgets
    below: the training entry points raise on an unfinished one."""
    from rl_sde_is_b200 import rollout as R
    from rl_sde_is_b200.models import DeterministicPolicy
    torch.manual_seed(seed)
    model = DeterministicPolicy(d, d, [H, H], nn.Tanh())
    with torch.no_grad():
        R.policy_linears(model)[2].bias.fill_(1.5)
    return model


def _env(d):
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D, DoubleWellStoppingTime2D
    return DoubleWellStoppingTime1D(beta=1.0, alpha=1.0, dt=0.005) if d == 1 else DoubleWellStoppingTime2D(beta=1.0, alpha=1.0, dt=0.005)


def _grads(model):
    return torch.cat([p.grad.reshape(-1) for p in model.parameters()])


@pytest.mark.parametrize("d,H,kernel", [(1, 32, "thread"), (2, 32, "thread"), (1, 64, "auto")])
def test_python_routes_match_dense(monkeypatch, d, H, kernel):
    """sample_loss_vectorized(...).backward(), the sample_returns_vectorized log-variance loss and rollout_loss_and_grad:
    with the budget lowered below the dense store they take the ragged one and match the dense route at the spacing the
    ragged route picked (kernels forced on both sides)."""
    L, R = _mods()
    from rl_sde_is_b200.reinforce_deterministic_core import sample_loss_vectorized, sample_returns_vectorized
    K, lim, seed = 3000, 4000, 99
    env = _env(d)
    model = _model(d, H, 7)
    if H > 32:
        # above width 32 the dense store may take 32 GiB whatever the budget: stand in for a batch where it does not fit
        dense_chooser = R.choose_ckpt_every
        monkeypatch.setattr(R, "choose_ckpt_every", lambda K_, *a, **k: dense_chooser(K_ * 10**6, *a, **k))
    calls = []
    real = R.rollout_forward_ragged
    monkeypatch.setattr(R, "rollout_forward_ragged", lambda *a, **k: calls.append(1) or real(*a, **k))

    def loss_route(ckpt):
        model.zero_grad()
        loss, G, T = sample_loss_vectorized(env, model, K, seed=seed, n_steps_lim=lim, kernel=kernel, ckpt_every=ckpt)
        loss.backward()
        return loss.detach(), G, T, _grads(model).clone()

    monkeypatch.setattr(R, "PATH_BUDGET_BYTES", 1 << 40)
    T = loss_route(1)[2].astype(np.int64) - 1
    monkeypatch.setattr(R, "PATH_BUDGET_BYTES", (int((T // 32 + 1).sum()) * d * 4) * 2 if H == 32 else 1 << 40)
    C = R.choose_ragged_ckpt_every([int((T // c + 1).sum()) for c in R.RAGGED_SPACINGS], d, hidden=H)
    if H == 32:
        assert R.choose_path_store(K, d, lim, hidden=H) is None
    n0 = len(calls)
    rag = loss_route(None)
    assert len(calls) == n0 + 1
    dense = loss_route(C)
    assert torch.equal(rag[0], dense[0]) and np.array_equal(rag[1], dense[1]) and np.array_equal(rag[2], dense[2])
    assert torch.equal(rag[3], dense[3])

    def logvar(ckpt):
        model.zero_grad()
        G, S, _ = sample_returns_vectorized(env, model, K, seed=seed, n_steps_lim=lim, kernel=kernel, stoch_int="exact",
                                            ckpt_every=ckpt)
        torch.var(G - S, unbiased=False).backward()
        return G.detach(), _grads(model).clone()

    a, b = logvar(None), logvar(C)
    assert len(calls) == n0 + 2
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])

    env_c, mlp_c = R.env_struct(env, L.HIT_ALL_GE_LB), L.make_mlp(d, H)
    flat = R.flat_parameters(model).detach().numpy()
    x = R.rollout_loss_and_grad(env_c, mlp_c, flat, K, seed=seed, n_steps_lim=lim, ckpt_every=None, kernel=kernel)
    y = R.rollout_loss_and_grad(env_c, mlp_c, flat, K, seed=seed, n_steps_lim=lim, ckpt_every=C, kernel=kernel)
    for u, v in zip(x, y):
        assert np.array_equal(u, v)


def test_autograd_frees_the_ragged_rollout(monkeypatch):
    """After backward() and with the outputs dropped, the ragged store is released."""
    _, R = _mods()
    from rl_sde_is_b200.reinforce_deterministic_core import sample_loss_vectorized
    monkeypatch.setattr(R, "PATH_BUDGET_BYTES", 512 << 10)      # the dense store needs 1 MB at spacing 32
    env, model = _env(1), _model(1, 32, 3)
    seen = []
    real = R.rollout_forward_ragged
    monkeypatch.setattr(R, "rollout_forward_ragged", lambda *a, **k: seen.append(real(*a, **k)) or seen[-1])
    loss, _, _ = sample_loss_vectorized(env, model, 2000, seed=1, n_steps_lim=4000, kernel="thread")
    loss.backward()
    ref = weakref.ref(seen.pop().path)
    del loss
    gc.collect()
    assert ref() is None


def test_full_size_wide_default_budget():
    """d = 1, H = 256, K = 6e4 at the default budget of 10**6 passes: the dense store does not fit, the ragged route trains,
    and its gradient is the dense route's at a budget just above the longest trajectory (tcgen05 kernels on both sides)."""
    L, R = _mods()
    K, H = 60000, 256
    env, model = _env(1), _model(1, H, 11)
    assert R.choose_path_store(K, 1, 10**6, hidden=H) is None
    env_c, mlp_c = R.env_struct(env, L.HIT_ALL_GE_LB), L.make_mlp(1, H)
    flat = R.flat_parameters(model).detach().numpy()
    tune = dict(wide_kernel="umma")
    rag = R.rollout_loss_and_grad(env_c, mlp_c, flat, K, seed=5, n_steps_lim=10**6, ckpt_every=None, tuning=tune)
    T = rag[3]
    assert (T >= 0).all()
    dense = R.rollout_loss_and_grad(env_c, mlp_c, flat, K, seed=5, n_steps_lim=int(T.max()) + 2, ckpt_every=1, tuning=tune)
    for u, v in zip(rag, dense):
        assert np.array_equal(u, v)
