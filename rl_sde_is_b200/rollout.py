"""Device-side rollout API: thin, typed wrappers over the C ABI plus the autograd Function.

This is the layer the reference-named drop-ins (reinforce_deterministic_core.sample_loss_vectorized,
approximate_methods.test_policy_vectorized, ...) are built on.  Tensors are torch CUDA tensors used
only as device memory; all arithmetic happens in librlsde_b200.so.
"""
import math
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from . import _lib as L
from .models import TabularPolicy


# ---------------------------------------------------------------------------------------------------
# env / policy description
# ---------------------------------------------------------------------------------------------------
def env_struct(env, hit_rule):
    """rlsde_env from any object with the reference env's attributes (environments.py:7-40)."""
    d = int(env.d)
    x0 = np.asarray(env.state_init, dtype=np.float64).reshape(-1)
    return L.make_env(d, env.alpha, float(env.sigma), float(env.dt), float(env.lb), float(env.rb), x0, hit_rule)


def policy_linears(model):
    """The three nn.Linear layers of a reference-style policy (models.py:4-18 + DeterministicPolicy).

    The fused kernels evaluate exactly ``Linear -> Tanh -> Linear -> Tanh -> Linear [-> Identity]``; any other stack
    (another nonlinearity, an output activation, dropout, ...) would be computed wrongly without an error, so the
    structure is checked positively."""
    if isinstance(model, TabularPolicy):
        raise L.RlsdeError("a TabularPolicy has no parameters, so no gradient: train an MLP policy; tables are rolled out by "
                           "test_policy_vectorized, estimate_fht_vectorized and is_estimate")
    seq = getattr(model, "policy", model)
    if not isinstance(seq, torch.nn.Sequential):
        raise L.RlsdeError("the policy must be an nn.Sequential (or expose one as .policy), as built by models.mlp")
    layers = [m for m in seq if not isinstance(m, torch.nn.Identity)]
    want = (torch.nn.Linear, torch.nn.Tanh, torch.nn.Linear, torch.nn.Tanh, torch.nn.Linear)
    if len(layers) != len(want) or not all(type(m) is w for m, w in zip(layers, want)):
        got = " -> ".join(type(m).__name__ for m in seq)
        raise L.RlsdeError("fused kernels cover Linear -> Tanh -> Linear -> Tanh -> Linear -> Identity "
                           f"(n_layers=3 with Tanh, what the reference builds); got {got}")
    linears = [layers[0], layers[2], layers[4]]
    if any(lin.bias is None for lin in linears):
        raise L.RlsdeError("fused kernels need Linear layers with bias (the reference's default)")
    return linears


def policy_shape(model):
    l1, l2, l3 = policy_linears(model)
    d, H = l1.in_features, l1.out_features
    if l2.in_features != H or l2.out_features != H or l3.in_features != H or l3.out_features != d:
        raise L.RlsdeError("policy must be d -> H -> H -> d")
    return d, H


def flat_parameters(model):
    """Differentiable flat view of the policy parameters in state_dict order."""
    ps = []
    for lin in policy_linears(model):
        ps += [lin.weight.reshape(-1), lin.bias.reshape(-1)]
    return torch.cat(ps)


_workspaces = {}


def _workspace(device, K=0, mlp=None):
    """Scratch buffer for the library, one per (device, stream): the work counters inside must not be shared by concurrent
    launches.  Sized by the largest batch seen (the forward rollout keeps one 24..168-byte record per trajectory there);
    with ``mlp`` (a reverse pass will follow) also by what the tcgen05 reverse kernel of that policy shape needs."""
    key = (device.type, device.index, torch.cuda.current_stream(device).cuda_stream)
    lib = L.load()
    n = int(lib.rlsde_workspace_bytes(int(K)))
    if mlp is not None:
        with torch.cuda.device(device):
            n = max(n, int(lib.rlsde_workspace_bytes_bwd(int(K), int(mlp.d_in), int(mlp.d_hidden))))
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < n:
        ws = torch.empty(n, dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _cuda_device(device=None):
    if not torch.cuda.is_available():
        raise L.RlsdeError("a CUDA device is required (no CPU fallback)")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.type != "cuda":
        raise L.RlsdeError("device must be a CUDA device")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    return dev


@dataclass
class RolloutOut:
    G: torch.Tensor                     # return_fht, float32 (float64 with state_f64)
    S: torch.Tensor                     # stoch_int_fht
    T: torch.Tensor                     # int32 hit index k* (-1 = not detected within n_steps_lim)
    l2: Optional[torch.Tensor]
    logw: Optional[torch.Tensor]
    path: Optional[torch.Tensor]
    stats_dev: torch.Tensor             # float64[RLSDE_NSTATS] on the device
    cfg: object = None
    path_base: Optional[torch.Tensor] = None    # int64[K + 1]: path is the ragged store (rlsde_rollout_fwd_ragged); None: dense
    _stats: Optional[np.ndarray] = None

    @property
    def stats(self):
        """Host copy of the statistics record (synchronises on first access)."""
        if self._stats is None:
            self._stats = self.stats_dev.cpu().numpy()
        return self._stats


def _check_bridge(d, store_path=False):
    if d != 1:
        raise L.RlsdeError(f"the Brownian-bridge hit test is defined at d = 1 only (the target of env.d = {d} is an orthant)")
    if store_path:
        raise L.RlsdeError("the Brownian-bridge hit test has no reverse pass: it cannot be combined with store_path")


def rollout_forward(env_c, mlp_c, params_host, K, *, seed=0, n_steps_lim=10**6, noise=None, traj_offset=0,
                    K_global=None, tanh="precise", stoch_int="reference", state_f64=False, store_path=False,
                    ckpt_every=1, policy_opt=None, grid=None, want_logw=True, device=None, out=None, kernel="auto", tuning=None,
                    bridge=False, path_base=None, n_slots=0):
    """One launch of K1 for K trajectories.  ``params_host``: contiguous float32 numpy array (state_dict order).
    ``bridge``: also detect target hits between passes with the Brownian-bridge crossing test (RLSDE_F_HIT_BRIDGE; d = 1,
    not with ``store_path``).  ``path_base`` (int64 CUDA tensor [K + 1], with ``store_path``): checkpoints go to a ragged
    store of ``n_slots`` rows laid out by it (``rlsde_rollout_fwd_ragged``; see ``rollout_forward_ragged``)."""
    if path_base is not None and not store_path:
        raise L.RlsdeError("path_base lays out the checkpoint store: it needs store_path=True")
    if bridge:
        _check_bridge(env_c.d, store_path)
    lib = L.load()
    dev = _cuda_device(device)
    K = int(K)
    d = env_c.d
    params_host = np.ascontiguousarray(params_host, dtype=np.float32)
    if params_host.size != lib.rlsde_param_count(mlp_c):
        raise L.RlsdeError(f"expected {lib.rlsde_param_count(mlp_c)} policy parameters, got {params_host.size}")
    flags = 0
    cfg = L.RlsdeRolloutCfg()
    cfg.K, cfg.traj_offset, cfg.K_global = K, int(traj_offset), int(K_global if K_global is not None else int(traj_offset) + K)
    cfg.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    cfg.n_steps_lim = int(n_steps_lim)
    if noise is not None:
        if noise.device != dev or noise.dtype != torch.float32 or not noise.is_contiguous():
            raise L.RlsdeError("noise must be a contiguous float32 CUDA tensor [n_steps, K_global, d]")
        if noise.dim() != 3 or noise.shape[1] != cfg.K_global or noise.shape[2] != d:
            raise L.RlsdeError(f"noise must have shape [n_steps, {cfg.K_global}, {d}], got {tuple(noise.shape)}")
        flags |= L.F_NOISE_INJECTED
        cfg.noise_steps = int(noise.shape[0])
    if tanh == "fast":
        flags |= L.F_TANH_FAST
    elif tanh != "precise":
        raise L.RlsdeError("tanh must be 'precise' or 'fast'")
    if stoch_int == "exact":
        flags |= L.F_STOCH_INT_EXACT
    elif stoch_int != "reference":
        raise L.RlsdeError("stoch_int must be 'reference' or 'exact'")
    if kernel not in ("auto", "thread", "warp", "tensor"):
        raise L.RlsdeError("kernel must be 'auto', 'thread', 'warp' or 'tensor'")
    flags |= {"auto": 0, "thread": L.F_KERNEL_THREAD, "warp": L.F_KERNEL_WARP, "tensor": L.F_KERNEL_TENSOR}[kernel]
    real = torch.float64 if state_f64 else torch.float32
    if state_f64:
        flags |= L.F_STATE_F64
    path = None
    if bridge:
        flags |= L.F_HIT_BRIDGE
    if store_path:
        flags |= L.F_STORE_PATH
        lim_eff = min(cfg.n_steps_lim, cfg.noise_steps) if noise is not None else cfg.n_steps_lim
        cfg.ckpt_every = int(ckpt_every)
        if path_base is None:
            cfg.ckpt_stride = (lim_eff + cfg.ckpt_every - 1) // cfg.ckpt_every
            path = torch.empty((K, cfg.ckpt_stride, d), dtype=torch.float32, device=dev)
        else:
            if path_base.device != dev or path_base.dtype != torch.int64 or not path_base.is_contiguous() \
                    or path_base.shape != (K + 1,):
                raise L.RlsdeError(f"path_base must be a contiguous int64 tensor [{K + 1}] on {dev}")
            path = torch.empty((max(int(n_slots), 1), d), dtype=torch.float32, device=dev)    # never empty: a pointer
    pol = None
    if policy_opt is not None:
        pol = torch.as_tensor(np.ascontiguousarray(np.asarray(policy_opt, dtype=np.float32).reshape(-1)), device=dev) \
            if not torch.is_tensor(policy_opt) else policy_opt.to(device=dev, dtype=torch.float32).reshape(-1).contiguous()
        lo, hi, h = grid
        cfg.n_grid, cfg.grid_lo, cfg.grid_hi, cfg.grid_h = int(pol.numel()), float(lo), float(hi), float(h)
    cfg.flags = flags
    L.apply_tuning(cfg, tuning)
    G = torch.empty(K, dtype=real, device=dev)
    S = torch.empty(K, dtype=real, device=dev)
    T = torch.empty(K, dtype=torch.int32, device=dev)
    l2 = torch.empty(K, dtype=real, device=dev) if pol is not None else None
    logw = torch.empty(K, dtype=real, device=dev) if want_logw else None
    stats = torch.zeros(L.RLSDE_NSTATS, dtype=torch.float64, device=dev)
    if K == 0:          # nothing to launch (and empty tensors have no device pointer to hand over)
        return RolloutOut(G=G, S=S, T=T, l2=l2, logw=logw, path=path, stats_dev=stats, cfg=cfg, path_base=path_base)
    ws = _workspace(dev, K)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        if path_base is None:
            rc = lib.rlsde_rollout_fwd(env_c, mlp_c, params_host.ctypes.data, cfg, _ptr(noise), _ptr(pol), _ptr(G), _ptr(S),
                                       _ptr(T), _ptr(l2), _ptr(logw), _ptr(path), _ptr(stats), _ptr(ws), ws.numel(), stream)
        else:
            if pol is not None or logw is not None:
                raise L.RlsdeError("the ragged store's rollout has no l2 or logw output")
            rc = lib.rlsde_rollout_fwd_ragged(env_c, mlp_c, params_host.ctypes.data, cfg, _ptr(noise), _ptr(path_base), _ptr(G),
                                              _ptr(S), _ptr(T), _ptr(path), _ptr(stats), _ptr(ws), ws.numel(), stream)
    L.check(rc, "rlsde_rollout_fwd" if path_base is None else "rlsde_rollout_fwd_ragged")
    return RolloutOut(G=G, S=S, T=T, l2=l2, logw=logw, path=path, stats_dev=stats, cfg=cfg, path_base=path_base)


def rollout_forward_table(env_c, table, K, *, grid, seed=0, n_steps_lim=10**6, noise=None, traj_offset=0, K_global=None,
                          stoch_int="reference", state_f64=False, policy_opt=None, want_logw=True, device=None, tuning=None,
                          bridge=False):
    """One launch of the d = 1 rollout under the control ``table[idx(x)]`` (``rlsde_rollout_fwd_table``).  ``table``:
    float32 values on ``grid = (lo, hi, h)``; ``policy_opt`` (l2 error), if given, lives on the same grid.  ``bridge``: as
    in ``rollout_forward``."""
    lib = L.load()
    dev = _cuda_device(device)
    K = int(K)
    if env_c.d != 1:
        raise L.RlsdeError(f"a tabulated control is a 1-D policy; env.d = {env_c.d}")

    def on_dev(a):
        t = a if torch.is_tensor(a) else torch.as_tensor(np.asarray(a, dtype=np.float32))
        return t.to(device=dev, dtype=torch.float32).reshape(-1).contiguous()

    tab = on_dev(table)
    cfg = L.RlsdeRolloutCfg()
    cfg.K, cfg.traj_offset, cfg.K_global = K, int(traj_offset), int(K_global if K_global is not None else int(traj_offset) + K)
    cfg.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    cfg.n_steps_lim = int(n_steps_lim)
    lo, hi, h = grid
    cfg.n_grid, cfg.grid_lo, cfg.grid_hi, cfg.grid_h = int(tab.numel()), float(lo), float(hi), float(h)
    flags = 0
    if noise is not None:
        if noise.device != dev or noise.dtype != torch.float32 or not noise.is_contiguous() or noise.dim() != 3 \
                or noise.shape[1] != cfg.K_global or noise.shape[2] != 1:
            raise L.RlsdeError(f"noise must be a contiguous float32 CUDA tensor [n_steps, {cfg.K_global}, 1]")
        flags |= L.F_NOISE_INJECTED
        cfg.noise_steps = int(noise.shape[0])
    flags |= {"reference": 0, "exact": L.F_STOCH_INT_EXACT}[stoch_int]
    if bridge:
        flags |= L.F_HIT_BRIDGE
    real = torch.float64 if state_f64 else torch.float32
    if state_f64:
        flags |= L.F_STATE_F64
    pol = None
    if policy_opt is not None:
        pol = on_dev(policy_opt)
        if pol.numel() != cfg.n_grid:
            raise L.RlsdeError(f"policy_opt has {pol.numel()} entries, the control table {cfg.n_grid}: they share one grid")
    cfg.flags = flags
    L.apply_tuning(cfg, tuning)
    G = torch.empty(K, dtype=real, device=dev)
    S = torch.empty(K, dtype=real, device=dev)
    T = torch.empty(K, dtype=torch.int32, device=dev)
    l2 = torch.empty(K, dtype=real, device=dev) if pol is not None else None
    logw = torch.empty(K, dtype=real, device=dev) if want_logw else None
    stats = torch.zeros(L.RLSDE_NSTATS, dtype=torch.float64, device=dev)
    if K == 0:
        return RolloutOut(G=G, S=S, T=T, l2=l2, logw=logw, path=None, stats_dev=stats, cfg=cfg)
    ws = _workspace(dev, K)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = lib.rlsde_rollout_fwd_table(env_c, _ptr(tab), cfg, _ptr(noise), _ptr(pol), _ptr(G), _ptr(S), _ptr(T), _ptr(l2),
                                         _ptr(logw), _ptr(stats), _ptr(ws), ws.numel(), stream)
    L.check(rc, "rlsde_rollout_fwd_table")
    return RolloutOut(G=G, S=S, T=T, l2=l2, logw=logw, path=None, stats_dev=stats, cfg=cfg)


@dataclass
class Transitions:
    """Device-resident transition stream of a rollout (float32 / bool, like the reference's ReplayBuffer arrays)."""
    states: torch.Tensor                # [n, d]
    actions: torch.Tensor               # [n, d]
    rewards: torch.Tensor               # [n]
    next_states: torch.Tensor           # [n, d]
    done: torch.Tensor                  # [n] bool
    counts: torch.Tensor                # [K] int64: transitions of each trajectory
    rollout: RolloutOut = None

    def __len__(self):
        return int(self.rewards.numel())


def rollout_transitions(env_c, mlp_c, params_host, K, *, seed=0, n_max=10**6, noise=None, traj_offset=0, K_global=None,
                        tanh="precise", state_f64=True, order="reference", device=None):
    """All (state, action, reward, next_state, done) tuples of K rollouts (SURVEY 8f-4).

    Two launches of K1 with the same counter-based noise: the first finds every trajectory's hit index, an exclusive
    prefix sum of the pass counts gives each trajectory its slot range, the second streams the tuples out.
    ``order='reference'`` returns them pass-major (all live trajectories of pass 0 in index order, then pass 1, ...), the
    order ``sample_trajectories_buffer_vectorized`` stores them in (approximate_methods.py:513-545);
    ``order='trajectory'`` keeps the kernel's trajectory-major layout and skips the permutation."""
    lib = L.load()
    if order not in ("reference", "trajectory"):
        raise L.RlsdeError("order must be 'reference' or 'trajectory'")
    dev = _cuda_device(device)
    d = env_c.d
    common = dict(seed=seed, n_steps_lim=int(n_max), noise=noise, traj_offset=traj_offset, K_global=K_global, tanh=tanh,
                  state_f64=state_f64, want_logw=False, device=dev, kernel="thread")
    first = rollout_forward(env_c, mlp_c, params_host, K, **common)
    lim = int(n_max) if noise is None else min(int(n_max), int(noise.shape[0]))
    T = first.T.to(torch.int64)
    counts = torch.where(T >= 0, T + 1, torch.full_like(T, lim))
    offsets, total = slot_offsets(counts)
    base = offsets[:-1]
    n = int(total.item()) if K > 0 else 0
    states = torch.empty((n, d), dtype=torch.float32, device=dev)
    actions = torch.empty((n, d), dtype=torch.float32, device=dev)
    next_states = torch.empty((n, d), dtype=torch.float32, device=dev)
    rewards = torch.empty(n, dtype=torch.float32, device=dev)
    done = torch.empty(n, dtype=torch.uint8, device=dev)
    cfg = first.cfg
    real = torch.float64 if state_f64 else torch.float32
    G = torch.empty(K, dtype=real, device=dev)
    S = torch.empty(K, dtype=real, device=dev)
    T2 = torch.empty(K, dtype=torch.int32, device=dev)
    stats = torch.zeros(L.RLSDE_NSTATS, dtype=torch.float64, device=dev)
    ws = _workspace(dev, K)
    if n > 0:
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            rc = lib.rlsde_rollout_transitions(env_c, mlp_c, np.ascontiguousarray(params_host, dtype=np.float32).ctypes.data, cfg,
                                               _ptr(noise), _ptr(base), _ptr(states), _ptr(actions), _ptr(rewards),
                                               _ptr(next_states), _ptr(done), _ptr(G), _ptr(S), _ptr(T2), _ptr(stats),
                                               _ptr(ws), ws.numel(), stream)
        L.check(rc, "rlsde_rollout_transitions")
    if order == "reference" and n > 0:
        # pass index of every slot; a stable sort by it turns trajectory-major into the reference's pass-major order
        k = torch.arange(n, device=dev, dtype=torch.int64) - torch.repeat_interleave(base, counts)
        perm = torch.argsort(k, stable=True)
        states, actions, rewards, next_states, done = (t[perm] for t in (states, actions, rewards, next_states, done))
    out = RolloutOut(G=G, S=S, T=T2, l2=None, logw=None, path=None, stats_dev=stats, cfg=cfg)
    return Transitions(states=states, actions=actions, rewards=rewards, next_states=next_states, done=done.bool(),
                       counts=counts, rollout=out)


def slot_offsets(counts):
    """Offsets of per-trajectory slot ranges, on the device: ``counts`` int64 [K] -> ``(base int64 [K + 1], total)``, where
    trajectory t owns slots [base[t], base[t + 1]) and ``total`` = base[K] is a 0-d device tensor (reading it synchronises).
    The transition stream (``rollout_transitions``) and the ragged checkpoint store (``rollout_forward_ragged``) lay out
    their buffers with it."""
    base = torch.zeros(counts.numel() + 1, dtype=torch.int64, device=counts.device)
    torch.cumsum(counts, 0, out=base[1:])
    return base, base[-1]


def ragged_ckpt_counts(T, ckpt_every):
    """Checkpoints of each trajectory in the ragged store: floor(T / C) + 1 if it finished, 0 if not (T = -1)."""
    T = T.to(torch.int64)
    return torch.where(T >= 0, T // int(ckpt_every) + 1, torch.zeros_like(T))


# Device memory a training rollout's checkpoint store may take, dense (choose_ckpt_every) or ragged
# (choose_ragged_ckpt_every).  Module-level, so that a test can lower it.
PATH_BUDGET_BYTES = 8 << 30
RAGGED_SPACINGS = (1, 2, 4, 8, 16, 32)


def choose_path_store(K, d, n_steps_lim, hidden=32):
    """Checkpoint spacing of the dense store where it fits (``choose_ckpt_every`` at PATH_BUDGET_BYTES), else None: the
    ragged store, whose spacing ``rollout_forward_ragged`` picks once the trajectories' lengths are known."""
    try:
        return choose_ckpt_every(K, d, n_steps_lim, budget_bytes=PATH_BUDGET_BYTES, hidden=hidden)
    except L.RlsdeError:
        return None


def choose_ragged_ckpt_every(slot_totals, d, hidden=32):
    """Smallest spacing C of RAGGED_SPACINGS (hidden width 32; C = 1 above, where the reverse pass reads every state) whose
    ragged store fits the budget of ``choose_ckpt_every``.  ``slot_totals[i]``: sum_k (floor(T_k / C) + 1) over the
    finished trajectories at C = RAGGED_SPACINGS[i]."""
    budget = PATH_BUDGET_BYTES if hidden == 32 else max(PATH_BUDGET_BYTES, 32 << 30)
    for c, n in zip(RAGGED_SPACINGS if hidden == 32 else RAGGED_SPACINGS[:1], slot_totals):
        if int(n) * d * 4 <= budget:
            return c
    raise L.RlsdeError(f"the checkpoints of the passes the trajectories ran ({int(slot_totals[0])} states of d={d}) do not fit "
                       f"{budget / 2**30:.1f} GiB even at spacing {32 if hidden == 32 else 1}; pass a smaller batch")


def rollout_forward_ragged(env_c, mlp_c, params_host, K, *, kernel="auto", device=None, **opts):
    """``rollout_forward(store_path=True)`` into the ragged checkpoint store: memory for the passes the trajectories run,
    not for the pass budget.  Two rollouts with the same counter-based noise: the first stores nothing (a base of zeros,
    so it runs the kernels of the second) and yields the hit indices; their checkpoint counts size the store (one host
    synchronisation, which also picks the spacing, ``choose_ragged_ckpt_every``); the second fills it.  Raises if the
    two rollouts' hit indices differ.  The returned ``path_base`` marks the store as ragged for ``rollout_backward``."""
    dev = _cuda_device(device)
    K = int(K)
    d, H = env_c.d, int(mlp_c.d_hidden)
    if kernel == "auto" and H == 32 and K <= 16 * torch.cuda.get_device_properties(dev).multi_processor_count:
        # the warp-per-trajectory kernels store every state or nothing (ckpt_every = 1): the spacing is known only after
        # the first rollout, so both run the thread-per-trajectory kernel
        kernel = "thread"
    common = dict(opts, store_path=True, want_logw=False, device=dev, kernel=kernel)
    first = rollout_forward(env_c, mlp_c, params_host, K, ckpt_every=1, path_base=torch.zeros(K + 1, dtype=torch.int64, device=dev),
                            **common)
    spacings = RAGGED_SPACINGS if H == 32 else RAGGED_SPACINGS[:1]
    totals = torch.stack([ragged_ckpt_counts(first.T, c).sum() for c in spacings]).cpu().numpy() if K > 0 else [0] * len(spacings)
    c = choose_ragged_ckpt_every(totals, d, hidden=H)
    base, _ = slot_offsets(ragged_ckpt_counts(first.T, c))
    out = rollout_forward(env_c, mlp_c, params_host, K, ckpt_every=c, path_base=base, n_slots=int(totals[spacings.index(c)]),
                          **common)
    if K > 0 and not torch.equal(out.T, first.T):
        raise L.RlsdeError("the two rollouts of the ragged checkpoint store disagree on the hit indices")
    return out


def rollout_forward_stored(env_c, mlp_c, params_host, K, *, ckpt_every=1, **opts):
    """The training rollout: checkpoints in the dense store at spacing ``ckpt_every``, or in the ragged store when
    ``ckpt_every`` is None (``choose_path_store``)."""
    if ckpt_every is None:
        return rollout_forward_ragged(env_c, mlp_c, params_host, K, **opts)
    return rollout_forward(env_c, mlp_c, params_host, K, store_path=True, want_logw=False, ckpt_every=ckpt_every, **opts)


def rollout_backward(env_c, mlp_c, params_host, fwd: RolloutOut, loss_scale, *, noise=None, device=None, balance=True,
                     coef=None):
    """The reverse pass: gradient of loss_scale * sum_k(-G_k - sg(G_k) S_k) w.r.t. the flat parameters (float32 CUDA tensor).

    With ``coef=(coef_G, coef_S)`` (float32 CUDA tensors [K] on the rollout's device) the gradient is that of
    loss_scale * sum_k (coef_G[k] G_k + coef_S[k] S_k) instead (rlsde_rollout_bwd_weighted; unfinished trajectories
    contribute 0).  A rollout with the ragged store (``fwd.path_base``) takes the weighted pass over it
    (rlsde_rollout_bwd_ragged), with coefficients (-1, -G) for the plain surrogate."""
    lib = L.load()
    dev = _cuda_device(device)
    if fwd.path is None:
        raise L.RlsdeError("the forward rollout must be run with store_path=True")
    if fwd.path_base is not None and coef is None:
        coef = (torch.full_like(fwd.G, -1.0), torch.neg(fwd.G))
    if coef is not None:
        coef = tuple(coef)
        K = fwd.T.numel()
        if len(coef) != 2 or any(not isinstance(c, torch.Tensor) or c.device != dev or c.dtype != torch.float32
                                 or not c.is_contiguous() or c.shape != (K,) for c in coef):
            raise L.RlsdeError(f"coef must be (coef_G, coef_S), contiguous float32 tensors [{K}] on {dev}")
    params_host = np.ascontiguousarray(params_host, dtype=np.float32)
    grad = torch.empty(int(lib.rlsde_param_count(mlp_c)), dtype=torch.float32, device=dev)
    ws = _workspace(dev, 0, mlp_c)
    with torch.cuda.device(dev):
        # longest trajectories first (stable sort => deterministic): balances the lock-step lanes of the reverse pass
        # (the warp-per-trajectory kernels, used for small batches, take trajectories in index order)
        n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
        thread_path = (fwd.cfg.flags & L.F_KERNEL_THREAD) or not ((fwd.cfg.flags & L.F_KERNEL_WARP) or fwd.T.numel() <= 16 * n_sm)
        order = torch.argsort(fwd.T, descending=True, stable=True) if balance and thread_path and fwd.T.numel() > 32 else None
        stream = torch.cuda.current_stream(dev).cuda_stream
        if fwd.path_base is not None:
            rc = lib.rlsde_rollout_bwd_ragged(env_c, mlp_c, params_host.ctypes.data, fwd.cfg, _ptr(noise), _ptr(coef[0]),
                                              _ptr(coef[1]), _ptr(fwd.T), _ptr(fwd.path_base), _ptr(fwd.path), _ptr(order),
                                              float(loss_scale), _ptr(grad), _ptr(ws), ws.numel(), stream)
        elif coef is None:
            rc = lib.rlsde_rollout_bwd(env_c, mlp_c, params_host.ctypes.data, fwd.cfg, _ptr(noise), _ptr(fwd.G), _ptr(fwd.T),
                                       _ptr(fwd.path), _ptr(order), float(loss_scale), _ptr(grad), _ptr(ws), ws.numel(), stream)
        else:
            rc = lib.rlsde_rollout_bwd_weighted(env_c, mlp_c, params_host.ctypes.data, fwd.cfg, _ptr(noise), _ptr(coef[0]),
                                                _ptr(coef[1]), _ptr(fwd.T), _ptr(fwd.path), _ptr(order), float(loss_scale),
                                                _ptr(grad), _ptr(ws), ws.numel(), stream)
    L.check(rc, "rlsde_rollout_bwd_ragged" if fwd.path_base is not None else
            "rlsde_rollout_bwd_weighted" if coef is not None else "rlsde_rollout_bwd")
    return grad


def rollout_loss_and_grad(env_c, mlp_c, params_host, K, *, seed=0, n_steps_lim=10**6, noise=None, tanh="precise",
                          stoch_int="reference", ckpt_every=1, device=None, kernel="auto", balance=True, tuning=None,
                          dist=None):
    """One REINFORCE evaluation with a single host synchronisation: K1 (with checkpoints), the statistics reduction and
    the reverse pass are enqueued back to back, and loss numerator, gradient, returns and hit indices come back in ONE device-to-host
    copy.  (The autograd route -- sample_loss_vectorized + .backward() -- synchronises after each kernel; at the
    reference's K = 100 those round trips cost as much as the kernels.)

    Returns ``(stats float64[RLSDE_NSTATS], grad float32[P] of mean_k(-G_k - sg(G_k) S_k), G float32[K], T int32[K])``
    as NumPy arrays.  With ``dist`` (a ``distributed.Shard``) the K trajectories are this rank's shard: statistics and
    gradient are those of the global batch (one all-gather of the packed rows), G and T stay local.  ``ckpt_every=None``:
    the ragged checkpoint store (``rollout_forward_ragged``), at the cost of one more rollout and synchronisation."""
    lib = L.load()
    dev = _cuda_device(device)
    K = int(K)
    P = int(lib.rlsde_param_count(mlp_c))
    params_host = np.ascontiguousarray(params_host, dtype=np.float32)
    align = lambda n: (n + 15) & ~15
    o_stats, o_grad = 0, 128
    o_G = o_grad + align(4 * P)
    o_T = o_G + align(4 * K)
    pack = torch.empty(o_T + align(4 * K), dtype=torch.uint8, device=dev)
    pack[:128].zero_()
    stats = pack[o_stats:o_stats + 128].view(torch.float64)
    grad = pack[o_grad:o_grad + 4 * P].view(torch.float32)
    G = pack[o_G:o_G + 4 * K].view(torch.float32)
    T = pack[o_T:o_T + 4 * K].view(torch.int32)
    S = torch.empty(K, dtype=torch.float32, device=dev)
    flags = L.F_STORE_PATH
    cfg = L.RlsdeRolloutCfg()
    cfg.K, cfg.traj_offset, cfg.K_global = K, (dist.traj_offset if dist is not None else 0), (dist.K_global if dist is not None else K)
    cfg.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    cfg.n_steps_lim = int(n_steps_lim)
    if noise is not None:
        if noise.device != dev or noise.dtype != torch.float32 or not noise.is_contiguous() or noise.dim() != 3 \
                or noise.shape[1] != cfg.K_global or noise.shape[2] != env_c.d:
            raise L.RlsdeError(f"noise must be a contiguous float32 CUDA tensor [n_steps, {cfg.K_global}, {env_c.d}]")
        flags |= L.F_NOISE_INJECTED
        cfg.noise_steps = int(noise.shape[0])
    flags |= {"precise": 0, "fast": L.F_TANH_FAST}[tanh]
    flags |= {"reference": 0, "exact": L.F_STOCH_INT_EXACT}[stoch_int]
    flags |= {"auto": 0, "thread": L.F_KERNEL_THREAD, "warp": L.F_KERNEL_WARP, "tensor": L.F_KERNEL_TENSOR}[kernel]
    lim_eff = min(cfg.n_steps_lim, cfg.noise_steps) if noise is not None else cfg.n_steps_lim
    ws = _workspace(dev, K, mlp_c)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        if ckpt_every is None:
            # the ragged checkpoint store (choose_path_store): one more rollout and one more synchronisation
            out = rollout_forward_ragged(env_c, mlp_c, params_host, K, seed=seed, n_steps_lim=n_steps_lim, noise=noise, tanh=tanh,
                                         stoch_int=stoch_int, traj_offset=cfg.traj_offset, K_global=cfg.K_global, kernel=kernel,
                                         tuning=tuning, device=dev)
            grad.copy_(rollout_backward(env_c, mlp_c, params_host, out, 1.0 / cfg.K_global, noise=noise, device=dev,
                                        balance=balance))
            stats.copy_(out.stats_dev)
            G.copy_(out.G)
            T.copy_(out.T)
        else:
            cfg.ckpt_every = int(ckpt_every)
            cfg.ckpt_stride = (lim_eff + cfg.ckpt_every - 1) // cfg.ckpt_every
            cfg.flags = flags
            L.apply_tuning(cfg, tuning)
            path = torch.empty((K, cfg.ckpt_stride, env_c.d), dtype=torch.float32, device=dev)
            rc = lib.rlsde_rollout_fwd(env_c, mlp_c, params_host.ctypes.data, cfg, _ptr(noise), 0, _ptr(G), _ptr(S), _ptr(T), 0, 0,
                                       _ptr(path), _ptr(stats), _ptr(ws), ws.numel(), stream)
            L.check(rc, "rlsde_rollout_fwd")
            n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
            thread_path = (flags & L.F_KERNEL_THREAD) or not ((flags & L.F_KERNEL_WARP) or K <= 16 * n_sm)
            order = torch.argsort(T, descending=True, stable=True) if balance and thread_path and K > 32 else None
            rc = lib.rlsde_rollout_bwd(env_c, mlp_c, params_host.ctypes.data, cfg, _ptr(noise), _ptr(G), _ptr(T), _ptr(path),
                                       _ptr(order), 1.0 / cfg.K_global, _ptr(grad), _ptr(ws), ws.numel(), stream)
            L.check(rc, "rlsde_rollout_bwd")
        if dist is not None and dist.world_size > 1:
            # the iteration's ONE exchange (SURVEY 8e): every rank's [gradient | statistics] row, added in rank order
            from .distributed import pack_grad_and_stats, reduce_gathered
            g_all, s_all = reduce_gathered(dist.all_gather_rows(pack_grad_and_stats(grad, stats)), P)
            grad.copy_(g_all)
            stats.copy_(s_all)
    host = pack.cpu().numpy()                               # the iteration's only synchronisation
    return (host[o_stats:o_stats + 128].view(np.float64), host[o_grad:o_grad + 4 * P].view(np.float32),
            host[o_G:o_G + 4 * K].view(np.float32), host[o_T:o_T + 4 * K].view(np.int32))


def choose_ckpt_every(K, d, n_steps_lim, budget_bytes=8 << 30, hidden=32):
    """Smallest checkpoint spacing whose path store fits the budget (1 = keep every state).  The wide-policy reverse
    kernel (hidden width > 32) reads every state, so there the spacing is 1 or an error."""
    if hidden != 32:
        need = K * n_steps_lim * d * 4
        if need > max(budget_bytes, 32 << 30):
            raise L.RlsdeError(f"hidden width {hidden}: the reverse pass keeps every state (K={K} x n_steps_lim={n_steps_lim} x d={d} "
                               f"floats = {need / 2**30:.1f} GiB); pass a smaller n_steps_lim")
        return 1
    for c in (1, 2, 4, 8, 16, 32):
        if K * ((n_steps_lim + c - 1) // c) * d * 4 <= budget_bytes:
            return c
    raise L.RlsdeError(
        f"path checkpoints for K={K}, n_steps_lim={n_steps_lim} do not fit {budget_bytes >> 30} GiB even at spacing 32; "
        "pass a smaller n_steps_lim")


def noise_fill(seed, K, d, n_pass, dt, *, traj_offset=0, pass_begin=0, device=None):
    """Increments dB[pass, k, i] exactly as the rollout kernels generate them in-kernel."""
    lib = L.load()
    dev = _cuda_device(device)
    out = torch.empty((int(n_pass), int(K), int(d)), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = lib.rlsde_noise_fill(int(seed) & 0xFFFFFFFFFFFFFFFF, int(traj_offset), int(K), int(d), int(pass_begin),
                                  int(n_pass), float(dt), _ptr(out), stream)
    L.check(rc, "rlsde_noise_fill")
    return out


def summarize(stats, dt=None):
    """Derived quantities from a statistics record (means over finished trajectories, population variance)."""
    n = stats[L.ST_N]
    nf = n - stats[L.ST_N_UNFINISHED]
    out = {"n": int(n), "n_unfinished": int(stats[L.ST_N_UNFINISHED]), "useful_steps": float(stats[L.ST_USEFUL_STEPS]),
           "max_hit_index": int(stats[L.ST_MAX_T])}
    if nf > 0:
        mg = stats[L.ST_SUM_G] / nf
        out.update(mean_return=mg, var_return=max(stats[L.ST_SUM_G2] / nf - mg * mg, 0.0),
                   mean_hit_index=stats[L.ST_SUM_T] / nf, mean_l2=stats[L.ST_SUM_L2] / nf,
                   mean_stoch_int=stats[L.ST_SUM_S] / nf)
        mw = stats[L.ST_SUM_W] / nf
        vw = max(stats[L.ST_SUM_W2] / nf - mw * mw, 0.0)
        out.update(is_mean=mw, is_var=vw, is_rel_error=(math.sqrt(vw) / mw if mw > 0 else float("nan")))
    return out
