"""Deterministic-policy REINFORCE on the fused rollout kernels (drop-in for the reference module).

Reference: rl_sde_is/reinforce_deterministic_core.py
  * ``sample_loss_vectorized(env, model, K)`` (:30-93)  -> one K1 launch (+ the reverse pass when ``.backward()`` runs)
  * ``reinforce(env, ...)`` (:102-336)                  -> same arguments, same keys in the returned dict
  * ``sample_returns_vectorized(env, model, K)``        -> (G, S) with a ``grad_fn``: train any loss over them

Keyword-only extras (defaults = reference behaviour): ``noise`` (injected increments
``[n_steps, K, d]``), ``seed`` (Philox key), ``n_steps_lim``, ``tanh`` ('precise' | 'fast'),
``stoch_int`` ('reference' | 'exact'), ``ckpt_every``, ``device``, ``dist`` (shard the batch over a
torch.distributed process group and all-reduce the packed gradient + statistics).

Without ``ckpt_every`` the reverse pass's checkpoints go to the dense store (every trajectory reserves the whole pass
budget) where it fits ``rollout.PATH_BUDGET_BYTES``, and to the ragged store (memory for the passes run, one more
rollout and host synchronisation) where it does not (``rollout.choose_path_store``).
"""
import dataclasses
import time

import numpy as np
import torch
import torch.nn as nn
import torch.optim as optim

from . import _lib as L
from . import rollout as R
from .models import DeterministicPolicy, mlp  # noqa: F401  (re-exported like the reference module)

def _next_seed(seed):
    """Rollouts without an explicit seed draw a fresh Philox key from torch's CPU generator, so that
    ``torch.manual_seed(s)`` makes a run reproducible the way it does for the reference."""
    if seed is not None:
        return int(seed)
    return int(torch.randint(0, 2**62, (1,), dtype=torch.int64).item())


def sample_loss_vectorized(env, model, K, *, noise=None, seed=None, n_steps_lim=10**6, tanh="precise",
                           stoch_int="reference", ckpt_every=None, device=None, dist=None, kernel="auto"):
    """Sample K trajectories under the policy and return ``(eff_loss, return_fht, time_steps)``.

    ``eff_loss`` is a 0-d float32 tensor (on the parameters' device) whose ``.backward()`` fills
    ``p.grad`` of ``model.parameters()``; ``return_fht`` is ``np.float32[K]`` and ``time_steps``
    ``np.float64[K]`` (= k*+1, the 1-based pass on which the hit is detected), as in the reference.
    With ``dist`` the K trajectories are this rank's shard of ``dist.K_global``; the loss is the global
    mean and the gradient is all-reduced inside ``backward``.
    """
    d, H = R.policy_shape(model)
    if d != env.d:
        raise L.RlsdeError(f"policy dimension {d} != env.d {env.d}")
    env_c = R.env_struct(env, L.HIT_ALL_GE_LB)          # torch path: x >= lb only (environments.py:51-52)
    mlp_c = L.make_mlp(d, H)
    dev = R._cuda_device(device)
    if noise is not None and not torch.is_tensor(noise):
        noise = torch.as_tensor(np.ascontiguousarray(noise, dtype=np.float32))
    if noise is not None:
        noise = noise.to(device=dev, dtype=torch.float32).contiguous()
    lim = int(n_steps_lim) if noise is None else min(int(n_steps_lim), int(noise.shape[0]))
    if ckpt_every is None:
        ckpt_every = R.choose_path_store(int(K), d, lim, hidden=H)      # None: the ragged store
    opts = dict(seed=_next_seed(seed), n_steps_lim=n_steps_lim, noise=noise, tanh=tanh, stoch_int=stoch_int,
                ckpt_every=ckpt_every, device=dev, kernel=kernel)
    if dist is not None:
        opts.update(traj_offset=dist.traj_offset, K_global=dist.K_global)
    flat = R.flat_parameters(model)
    holder = {}
    loss = _LossWithAux.apply(flat, env_c, mlp_c, int(K), opts, holder, dist)
    out = holder["out"]
    T = out.T.cpu().numpy()
    if (T < 0).any():
        # the reference would hand back uninitialised torch.empty values here (:41-43); we refuse instead
        raise L.RlsdeError(f"{int((T < 0).sum())} of {K} trajectories did not reach the target set within "
                           f"{lim} passes; raise n_steps_lim")
    return loss, out.G.cpu().numpy(), (T + 1).astype(np.float64)


def sample_returns_vectorized(env, model, K, *, noise=None, seed=None, n_steps_lim=10**6, tanh="precise",
                              stoch_int="reference", ckpt_every=None, device=None, kernel="auto"):
    """Sample K trajectories under the policy and return ``(return_fht, stoch_int_fht, time_steps)``, so that any loss
    over the returns G and the stochastic integrals S can be trained, as the reference allows by editing its surrogate
    (:91).  ``return_fht`` and ``stoch_int_fht`` are float32 CUDA tensors [K] with a ``grad_fn``: a loss formed from them
    on the GPU and ``.backward()``-ed fills ``p.grad`` of ``model.parameters()`` (accumulating, as autograd does) through
    one weighted reverse pass (``rlsde_rollout_bwd_weighted``).  The derivative is the pathwise one along the sampled paths
    with the hit passes held fixed, the derivative the reference's autograd graph takes.  S is S_ref, or S_exact with
    ``stoch_int="exact"``; ``time_steps`` is ``np.float64[K]`` (= k*+1) as in ``sample_loss_vectorized``.

    The log-variance loss, zero under the optimal control u* (where G - S_exact = log Psi(x0)):

        G, S, _ = sample_returns_vectorized(env, model, K, stoch_int="exact")
        torch.var(G - S, unbiased=False).backward()

    ``sample_loss_vectorized``'s ``eff_loss`` is ``torch.mean(-G - G.detach() * S)`` over the reference S.
    """
    d, H = R.policy_shape(model)
    if d != env.d:
        raise L.RlsdeError(f"policy dimension {d} != env.d {env.d}")
    env_c = R.env_struct(env, L.HIT_ALL_GE_LB)
    mlp_c = L.make_mlp(d, H)
    dev = R._cuda_device(device)
    if noise is not None and not torch.is_tensor(noise):
        noise = torch.as_tensor(np.ascontiguousarray(noise, dtype=np.float32))
    if noise is not None:
        noise = noise.to(device=dev, dtype=torch.float32).contiguous()
    lim = int(n_steps_lim) if noise is None else min(int(n_steps_lim), int(noise.shape[0]))
    if ckpt_every is None:
        ckpt_every = R.choose_path_store(int(K), d, lim, hidden=H)      # None: the ragged store
    opts = dict(seed=_next_seed(seed), n_steps_lim=n_steps_lim, noise=noise, tanh=tanh, stoch_int=stoch_int,
                ckpt_every=ckpt_every, device=dev, kernel=kernel)
    holder = {}
    G, S = _ReturnsWithAux.apply(R.flat_parameters(model), env_c, mlp_c, int(K), opts, holder)
    T = holder["out"].T.cpu().numpy()
    if (T < 0).any():
        raise L.RlsdeError(f"{int((T < 0).sum())} of {K} trajectories did not reach the target set within "
                           f"{lim} passes; raise n_steps_lim")
    return G, S, (T + 1).astype(np.float64)


def _loss_and_grads_fused(env, model, K, *, noise=None, seed=None, n_steps_lim=10**6, tanh="precise", stoch_int="reference",
                          ckpt_every=None, device=None, kernel="auto", dist=None, tuning=None):
    """What ``sample_loss_vectorized`` + ``eff_loss.backward()`` produce, with one host synchronisation and without the
    autograd graph: sets ``p.grad`` of the policy's parameters and returns ``(loss float, return_fht, time_steps)``.
    Used by ``reinforce()``; results are those of the autograd route (same kernels, same arguments)."""
    d, H = R.policy_shape(model)
    if d != env.d:
        raise L.RlsdeError(f"policy dimension {d} != env.d {env.d}")
    env_c = R.env_struct(env, L.HIT_ALL_GE_LB)
    mlp_c = L.make_mlp(d, H)
    dev = R._cuda_device(device)
    if noise is not None:
        noise = torch.as_tensor(np.ascontiguousarray(noise, dtype=np.float32)) if not torch.is_tensor(noise) else noise
        noise = noise.to(device=dev, dtype=torch.float32).contiguous()
    lim = int(n_steps_lim) if noise is None else min(int(n_steps_lim), int(noise.shape[0]))
    if ckpt_every is None:
        ckpt_every = R.choose_path_store(int(K), d, lim, hidden=H)      # None: the ragged store
    linears = R.policy_linears(model)
    with torch.no_grad():
        params_host = torch.cat([t.reshape(-1) for lin in linears for t in (lin.weight, lin.bias)]).to(torch.float32).numpy()
    stats, grad, G, T = R.rollout_loss_and_grad(env_c, mlp_c, params_host, int(K), seed=_next_seed(seed), n_steps_lim=n_steps_lim,
                                                noise=noise, tanh=tanh, stoch_int=stoch_int, ckpt_every=ckpt_every,
                                                device=dev, kernel=kernel, dist=dist, tuning=tuning)
    if stats[L.ST_N_UNFINISHED] > 0:           # counted over ALL shards: every rank raises together, before touching .grad
        raise L.RlsdeError(f"{int(stats[L.ST_N_UNFINISHED])} of {int(stats[L.ST_N])} trajectories did not reach the target set "
                           f"within {lim} passes; raise n_steps_lim")
    g = torch.from_numpy(grad.copy())
    off = 0
    for lin in linears:
        for t in (lin.weight, lin.bias):
            piece = g[off:off + t.numel()].view_as(t).to(t.dtype)
            t.grad = piece if t.grad is None else t.grad + piece
            off += t.numel()
    return float(np.float32(stats[L.ST_SUM_LOSS] / stats[L.ST_N])), G.copy(), (T + 1).astype(np.float64)


class _DeviceLoop:
    """REINFORCE iterations with parameters, Adam state and logs resident on the GPU (``rlsde_reinforce_step``): each
    iteration is one C call that enqueues rollout, statistics, reverse pass and Adam update; nothing is read back until
    ``flush()``.  Small batches only (warp-per-trajectory kernels: K <= 16 x SMs, hidden width 32)."""

    def __init__(self, env, model, K, lr, n_iterations, *, n_steps_lim=10**6, tanh="precise", stoch_int="reference", device=None,
                 betas=(0.9, 0.999), eps=1e-8, dist=None):
        self.lib = L.load()
        self.env, self.model, self.K, self.lr, self.betas, self.eps = env, model, int(K), float(lr), betas, float(eps)
        d, H = R.policy_shape(model)
        self.env_c, self.mlp_c = R.env_struct(env, L.HIT_ALL_GE_LB), L.make_mlp(d, H)
        self.dev = dev = R._cuda_device(device)
        self.linears = R.policy_linears(model)
        with torch.no_grad():
            flat = torch.cat([t.reshape(-1) for lin in self.linears for t in (lin.weight, lin.bias)]).to(torch.float32)
        self.theta = flat.to(dev)
        self.m, self.v = torch.zeros_like(self.theta), torch.zeros_like(self.theta)
        self.grad = torch.empty_like(self.theta)
        # data parallel (SURVEY 8e): K is this rank's shard of dist.K_global; one all-gather per iteration, enqueued on
        # the rollout's stream between the reverse pass and the Adam kernel, so the loop stays free of host round trips
        self.dist = dist if dist is not None and dist.world_size > 1 else None
        self.P = int(self.lib.rlsde_param_count(self.mlp_c))
        cfg = L.RlsdeRolloutCfg()
        cfg.K, cfg.traj_offset, cfg.K_global = self.K, (dist.traj_offset if self.dist else 0), (dist.K_global if self.dist else self.K)
        cfg.n_steps_lim = int(n_steps_lim)
        cfg.flags = L.F_STORE_PATH | L.F_KERNEL_WARP | {"precise": 0, "fast": L.F_TANH_FAST}[tanh] \
            | {"reference": 0, "exact": L.F_STOCH_INT_EXACT}[stoch_int]
        cfg.ckpt_every, cfg.ckpt_stride = 1, int(n_steps_lim)
        self.cfg = cfg
        self.path = torch.empty((self.K, cfg.ckpt_stride, d), dtype=torch.float32, device=dev)
        self.S = torch.empty(self.K, dtype=torch.float32, device=dev)
        n = int(n_iterations)
        self.logG = torch.empty((n, self.K), dtype=torch.float32, device=dev)
        self.logT = torch.empty((n, self.K), dtype=torch.int32, device=dev)
        self.logStats = torch.zeros((n, L.RLSDE_NSTATS), dtype=torch.float64, device=dev)
        self.events = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
        self.ws = R._workspace(dev, self.K)
        if self.dist:
            self.row = torch.zeros(self.P + L.RLSDE_NSTATS, dtype=torch.float64, device=dev)
            self.local_stats = torch.zeros(L.RLSDE_NSTATS, dtype=torch.float64, device=dev)
        self.done, self.read = 0, 0
        self.events[0].record(torch.cuda.current_stream(dev))

    @staticmethod
    def supported(env, model, K, rollout_opts, device=None):
        try:
            d, H = R.policy_shape(model)
            if H != 32 or d != env.d or not torch.cuda.is_available():
                return False
            if any(k in rollout_opts for k in ("noise", "ckpt_every", "seed")) or rollout_opts.get("kernel", "auto") == "thread":
                return False
            lim = int(rollout_opts.get("n_steps_lim", 10**6))
            if int(K) * lim * d * 4 > (8 << 30):             # every state is kept for the reverse pass
                return False
            n_sm = torch.cuda.get_device_properties(R._cuda_device(device)).multi_processor_count
            return int(K) <= 16 * n_sm and all(p.device.type == "cpu" for p in model.parameters())
        except L.RlsdeError:
            return False

    def step(self):
        i = self.done
        self.cfg.seed = _next_seed(None) & 0xFFFFFFFFFFFFFFFF
        with torch.cuda.device(self.dev):
            stream = torch.cuda.current_stream(self.dev)
            if self.dist is None:
                rc = self.lib.rlsde_reinforce_step(self.env_c, self.mlp_c, self.theta.data_ptr(), self.m.data_ptr(), self.v.data_ptr(),
                                                   self.cfg, 0, self.lr, self.betas[0], self.betas[1], self.eps, i + 1,
                                                   self.logG[i].data_ptr(), self.S.data_ptr(), self.logT[i].data_ptr(),
                                                   self.path.data_ptr(), self.logStats[i].data_ptr(), self.grad.data_ptr(),
                                                   self.ws.data_ptr(), self.ws.numel(), stream.cuda_stream)
                L.check(rc, "rlsde_reinforce_step")
            else:
                rc = self.lib.rlsde_reinforce_rollout(self.env_c, self.mlp_c, self.theta.data_ptr(), self.cfg, 0,
                                                      self.logG[i].data_ptr(), self.S.data_ptr(), self.logT[i].data_ptr(),
                                                      self.path.data_ptr(), self.local_stats.data_ptr(), self.grad.data_ptr(),
                                                      self.row.data_ptr(), self.ws.data_ptr(), self.ws.numel(), stream.cuda_stream)
                L.check(rc, "rlsde_reinforce_rollout")
                rows = self.dist.all_gather_rows(self.row)            # the iteration's one collective, on this stream
                rc = self.lib.rlsde_reinforce_apply(self.mlp_c, self.theta.data_ptr(), self.m.data_ptr(), self.v.data_ptr(),
                                                    rows.data_ptr(), int(rows.shape[0]), self.lr, self.betas[0], self.betas[1],
                                                    self.eps, i + 1, self.grad.data_ptr(), self.logStats[i].data_ptr(),
                                                    stream.cuda_stream)
                L.check(rc, "rlsde_reinforce_apply")
            self.events[i + 1].record(stream)
        self.done = i + 1

    def flush(self):
        """Synchronise, copy the parameters back into the module and return the log rows of the iterations enqueued since
        the last flush: ``(first index, losses f32, returns [n, K] f32, time_steps [n, K] f64, seconds per iteration)``."""
        lo, hi = self.read, self.done
        torch.cuda.synchronize(self.dev)
        theta = self.theta.cpu()
        off = 0
        with torch.no_grad():
            for lin in self.linears:
                for t in (lin.weight, lin.bias):
                    t.copy_(theta[off:off + t.numel()].view_as(t))
                    off += t.numel()
        G = self.logG[lo:hi].cpu().numpy()
        T = self.logT[lo:hi].cpu().numpy()
        st = self.logStats[lo:hi].cpu().numpy()
        if (st[:, L.ST_N_UNFINISHED] > 0).any():
            # such a batch took no Adam step on the device (adam_step_kernel looks at the count), so theta is that of the
            # last complete iteration
            bad = int(np.flatnonzero(st[:, L.ST_N_UNFINISHED] > 0)[0])
            raise L.RlsdeError(f"iteration {lo + bad}: {int(st[bad, L.ST_N_UNFINISHED])} trajectories did not reach the target "
                               f"set within {self.cfg.n_steps_lim} passes (no parameter update was applied); raise n_steps_lim")
        secs = np.array([self.events[i].elapsed_time(self.events[i + 1]) * 1e-3 for i in range(lo, hi)])
        self.read = hi
        return lo, (st[:, L.ST_SUM_LOSS] / st[:, L.ST_N]).astype(np.float32), G, (T + 1).astype(np.float64), secs


class _LossWithAux(torch.autograd.Function):
    """eff_loss = mean_k(-G_k - sg(G_k) S_k) as a differentiable function of the flat policy parameters: forward launches
    the rollout kernel (with state checkpoints), backward the reverse kernel -- what autograd does in the reference over
    ~25 nodes per pass (reinforce_deterministic_core.py:52-93, :240).  The raw rollout is handed back through ``holder``;
    with ``dist`` the statistics and the gradient are all-reduced over the ranks."""

    @staticmethod
    def forward(ctx, flat_params, env_c, mlp_c, K, opts, holder, dist):
        params_host = flat_params.detach().to("cpu", torch.float32).contiguous().numpy()
        out = R.rollout_forward_stored(env_c, mlp_c, params_host, K, **opts)
        holder["out"] = out
        K_global = out.cfg.K_global
        if dist is not None:
            stats = dist.all_reduce_stats(out.stats_dev.clone())
            loss = float(stats[L.ST_SUM_LOSS].item()) / K_global
            holder["stats_global"] = stats.cpu().numpy()
        else:
            loss = out.stats[L.ST_SUM_LOSS] / K_global
        ctx.env_c, ctx.mlp_c, ctx.params_host, ctx.out, ctx.opts, ctx.dist = env_c, mlp_c, params_host, out, opts, dist
        return torch.tensor(loss, dtype=torch.float32, device=flat_params.device)

    @staticmethod
    def backward(ctx, grad_out):
        out = ctx.out
        g = R.rollout_backward(ctx.env_c, ctx.mlp_c, ctx.params_host, out, 1.0 / out.cfg.K_global,
                               noise=ctx.opts.get("noise"), device=ctx.opts.get("device"))
        if ctx.dist is not None:
            g = ctx.dist.all_reduce_sum(g)
        g = g.to(grad_out.device) * grad_out.to(torch.float32)
        return g, None, None, None, None, None, None


class _ReturnsWithAux(torch.autograd.Function):
    """(G, S) [K] as differentiable functions of the flat policy parameters: forward launches the rollout kernel (with
    state checkpoints), backward the weighted reverse kernel with the incoming gradients as per-trajectory coefficients,
    grad = sum_k (dL/dG_k dG_k/dtheta + dL/dS_k dS_k/dtheta)."""

    @staticmethod
    def forward(ctx, flat_params, env_c, mlp_c, K, opts, holder):
        params_host = flat_params.detach().to("cpu", torch.float32).contiguous().numpy()
        out = R.rollout_forward_stored(env_c, mlp_c, params_host, K, **opts)
        holder["out"] = out
        # ctx keeps what the reverse pass reads (T, path, cfg), not the returned G and S: outputs reachable from their own
        # grad_fn through ctx form a cycle that the garbage collector cannot see, and every rollout would stay allocated
        ctx.fwd = dataclasses.replace(out, G=None, S=None, l2=None, logw=None)
        ctx.env_c, ctx.mlp_c, ctx.params_host, ctx.opts = env_c, mlp_c, params_host, opts
        ctx.param_device = flat_params.device
        return out.G, out.S

    @staticmethod
    def backward(ctx, gG, gS):
        fwd = ctx.fwd
        coef = tuple(torch.zeros(fwd.T.shape, dtype=torch.float32, device=fwd.T.device) if g is None
                     else g.to(fwd.T.device, torch.float32).contiguous() for g in (gG, gS))
        g = R.rollout_backward(ctx.env_c, ctx.mlp_c, ctx.params_host, fwd, 1.0, noise=ctx.opts.get("noise"),
                               device=ctx.opts.get("device"), coef=coef)
        return g.to(ctx.param_device), None, None, None, None, None


def reinforce(env, gamma=1., d_hidden_layer=256, n_layers=3, batch_size=1000, lr=1e-3, n_iterations=100, seed=None,
              test_batch_size=1000, test_freq_iterations=100, backup_freq_iterations=None, policy_opt=None,
              load=False, test=False, live_plot=False, *, save=True, save_fn=None, verbose=True, device_loop=None,
              **rollout_opts):
    """Training loop with the reference's signature, result dictionary and on-disk layout (:102-336).

    ``agent.npz`` and the ``model_n-it{i}`` backups go to the reference's run directory (``utils_path``; pass
    ``save=False`` to keep everything in memory); ``load=True`` returns the stored dictionary, ``load=True, test=True``
    re-tests the stored backups like the reference.  ``save_fn(data, model, iteration)`` is an extra hook called where a
    backup is written.  Plotting (``live_plot``) is out of the hot path's scope.

    ``device_loop`` (default: whenever the batch is small enough for the warp-per-trajectory kernels): parameters, Adam
    state and per-iteration logs stay on the GPU and an iteration is one asynchronous C call
    (``rlsde_reinforce_step``); the host synchronises only where the reference looks at the model (tests, backups, the
    end).  ``cts`` are then device times per iteration.  ``device_loop=False`` steps ``torch.optim.Adam`` on the CPU
    module every iteration, like the reference.  ``gamma`` is accepted and unused in
    the loss, as in the reference (:108-117, SURVEY App. A-8).
    """
    from .approximate_methods import test_policy_vectorized
    from . import utils_path as up

    # fail before any file is written if no fused kernel exists for this policy shape
    if n_layers != 3:
        raise L.RlsdeError(f"fused kernels cover n_layers=3 (two hidden layers, what the reference's CLI builds); got {n_layers}")
    if not L.load().rlsde_supported(int(env.state_space_dim), int(d_hidden_layer), 2):
        raise L.RlsdeError(f"no fused kernel for state dimension {env.state_space_dim} with hidden width {d_hidden_layer} "
                           "(rlsde_supported)")

    rel_dir_path = None
    if save or load:
        rel_dir_path = up.get_reinforce_det_dir_path(env, agent="reinforce-deterministic", gamma=gamma,
                                                     d_hidden_layer=d_hidden_layer, batch_size=batch_size, lr=lr,
                                                     n_iterations=n_iterations, seed=seed)
    if load and not test:
        return up.load_data(rel_dir_path)
    stored = up.load_data(rel_dir_path) if load else None

    shard = rollout_opts.get("dist")
    if shard is not None and shard.world_size > 1:
        # data parallel: batch_size is the GLOBAL batch, every rank rolls its shard out.  All ranks must build the same
        # initial policy and draw the same Philox keys (the global trajectory id makes the shards' noise disjoint), so
        # an unseeded run takes rank 0's seed.
        if shard.K_global != batch_size:
            raise L.RlsdeError(f"dist.K_global ({shard.K_global}) must equal batch_size ({batch_size})")
        if seed is None:
            import torch.distributed as tdist
            box = [int(torch.randint(0, 2**31 - 1, (1,)).item())]
            tdist.broadcast_object_list(box, src=0, group=shard.group)
            np.random.seed(box[0])
            torch.manual_seed(box[0])
    K_local = shard.K_local if shard is not None else batch_size
    if seed is not None:
        np.random.seed(seed)
        torch.manual_seed(seed)
    hidden = [d_hidden_layer] * (n_layers - 1)
    model = DeterministicPolicy(state_dim=env.state_space_dim, action_dim=env.action_space_dim,
                                hidden_sizes=hidden, activation=nn.Tanh())
    try:
        optimizer = optim.Adam(model.parameters(), lr=lr, fused=True)     # one pass over the 6 small tensors (same update rule)
    except (TypeError, RuntimeError, ValueError):
        optimizer = optim.Adam(model.parameters(), lr=lr)
    fused_path = all(p.device.type == "cpu" for p in model.parameters())
    data = dict(gamma=gamma, n_layers=n_layers, d_hidden_layer=d_hidden_layer, batch_size=batch_size, lr=lr,
                n_iterations=n_iterations, seed=seed, backup_freq_iterations=backup_freq_iterations, model=model)
    if load:
        data = stored
        data["model"] = model
    if rel_dir_path is not None:
        data["rel_dir_path"] = rel_dir_path
    returns = np.empty(0, dtype=np.float32)
    time_steps = np.empty(0, dtype=np.int32)
    losses, exp_returns, var_returns, exp_time_steps, cts = (np.full(n_iterations, np.nan) for _ in range(5))
    tests = {k: np.empty(0, dtype=np.float32) for k in ("mean_returns", "var_returns", "mean_lengths", "policy_l2_errors")}

    def run_test(it):
        res = test_policy_vectorized(env, model, batch_size=test_batch_size, policy_opt=policy_opt)
        for key, val in zip(tests, res):
            tests[key] = np.append(tests[key], val)
        if verbose:
            print("it.: {:3d}, test mean return: {:2.2f}, test var return: {:.2e}, test mean time steps: {:2.2f}".format(
                it, res[0], res[1], res[2]))

    def results():
        out = dict(returns=returns, time_steps=time_steps, losses=losses, exp_returns=exp_returns,
                   var_returns=var_returns, exp_time_steps=exp_time_steps, cts=cts)
        if test:
            out.update(test_mean_returns=tests["mean_returns"], test_var_returns=tests["var_returns"],
                       test_mean_lengths=tests["mean_lengths"], test_policy_l2_errors=tests["policy_l2_errors"])
        return out

    if test:
        data.update(test_freq_iterations=test_freq_iterations, test_batch_size=test_batch_size)
    if save:
        up.save_data(data, rel_dir_path)
        if not load:
            up.save_model(model, rel_dir_path, "model_n-it{}".format(0))
    if test:
        run_test(0)

    if device_loop is None:
        device_loop = not load and _DeviceLoop.supported(env, model, K_local, rollout_opts, rollout_opts.get("device"))
    loop = None
    if device_loop and not load and n_iterations > 0:
        loop = _DeviceLoop(env, model, K_local, lr, n_iterations,
                           **{k: v for k, v in rollout_opts.items() if k in ("n_steps_lim", "tanh", "stoch_int", "device", "dist")})

    def drain():
        """Bring the device loop's finished iterations into the result arrays (one synchronisation)."""
        nonlocal returns, time_steps
        lo, ls, G, T, secs = loop.flush()
        for j in range(len(ls)):
            i_ = lo + j
            returns = np.append(returns, G[j])
            time_steps = np.append(time_steps, T[j])
            losses[i_], cts[i_] = ls[j], secs[j]
            exp_returns[i_], var_returns[i_], exp_time_steps[i_] = np.mean(G[j]), np.var(G[j]), np.mean(T[j])
            if verbose:
                print("it.: {:2d}, loss: {:.3e}, exp return: {:.3e}, var return: {:.1e}, ct: {:.3f}".format(
                    i_, losses[i_], exp_returns[i_], var_returns[i_], cts[i_]))

    for i in range(n_iterations):
        if loop is not None:
            loop.step()
            need_model = (test and (i + 1) % test_freq_iterations == 0) or i + 1 == n_iterations or \
                (backup_freq_iterations is not None and (i + 1) % backup_freq_iterations == 0)
            if need_model:
                drain()
        elif not load:
            t0 = time.time()
            optimizer.zero_grad()
            if fused_path:     # same kernels as sample_loss_vectorized + backward(), one host synchronisation
                eff_loss, batch_returns, batch_time_steps = _loss_and_grads_fused(env, model, K_local, **rollout_opts)
            else:
                eff_loss, batch_returns, batch_time_steps = sample_loss_vectorized(env, model, K_local, **rollout_opts)
                eff_loss.backward()
            optimizer.step()
            cts[i] = time.time() - t0          # wall clock of zero_grad -> loss -> backward -> step, like the reference's ct

            returns = np.append(returns, batch_returns)
            time_steps = np.append(time_steps, batch_time_steps)
            losses[i] = float(eff_loss.detach()) if torch.is_tensor(eff_loss) else eff_loss
            exp_returns[i] = np.mean(batch_returns)
            var_returns[i] = np.var(batch_returns)
            exp_time_steps[i] = np.mean(batch_time_steps)
            if verbose:
                print("it.: {:2d}, loss: {:.3e}, exp return: {:.3e}, var return: {:.1e}, ct: {:.3f}".format(
                    i, losses[i], exp_returns[i], var_returns[i], cts[i]))
        if test and (i + 1) % test_freq_iterations == 0:
            if load:
                try:                               # re-test the stored backup of this iteration (:95-99, :267-270)
                    up.load_model(model, rel_dir_path, "model_n-it{}".format(i + 1))
                except FileNotFoundError:
                    print("there is no backup for iteration {:d}".format(i + 1))
            run_test(i + 1)
        if not load and backup_freq_iterations is not None and (i + 1) % backup_freq_iterations == 0:
            if save:
                up.save_model(model, rel_dir_path, "model_n-it{}".format(i + 1))
                data.update(results())
                up.save_data(data, rel_dir_path)
            if save_fn is not None:
                save_fn(data, model, i + 1)

    if not load:
        data.update(results())
    elif test:
        data.update({k: v for k, v in results().items() if k.startswith("test_")})
    if save:
        up.save_data(data, rel_dir_path)
    return data
