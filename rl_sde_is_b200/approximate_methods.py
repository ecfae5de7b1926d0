"""No-grad policy rollouts on the fused kernel (drop-in for the reference's hot functions).

Reference: rl_sde_is/approximate_methods.py
  * ``test_policy_vectorized(env, model, batch_size, k_max, policy_opt)`` (:577-648)
  * ``estimate_fht_vectorized(env, model, batch_size, k_max)`` (:650-695)
Both follow the NumPy path of the reference: float64 state and accumulators with a float32 policy
(SURVEY App. A-5), hit rule ``lb <= x <= rb`` in 1-D (:48-49), hit index ``ep_lens = k*`` (0-based).

``sample_trajectories_buffer_vectorized(env, model, replay_buffer, batch_size, n_max)`` (:513-545) is the TD3 data
path (SURVEY 8f-4): the same rollout with a transition-stream epilogue, stored through ``store_vectorized``.

``is_estimate`` is build-side (SURVEY App. C): the importance-sampling estimator of
Psi(x0) = E[exp(-tau)] from the same rollout, mean and relative error.
"""
import numpy as np
import torch

from . import _lib as L
from . import rollout as R
from .models import TabularPolicy
from .reinforce_deterministic_core import _next_seed


def _numpy_path_rollout(env, model, batch_size, k_max, policy_opt, *, noise, seed, tanh, state_f64, device, dist, kernel="auto",
                        stoch_int="reference", want_logw=False, bridge=False):
    """An MLP policy runs on the fused MLP kernels; a ``TabularPolicy`` on ``rlsde_rollout_fwd_table`` (``tanh`` and
    ``kernel`` do not apply to it).  ``bridge``: the Brownian-bridge hit test between passes (d = 1)."""
    table = isinstance(model, TabularPolicy)
    if table:
        if env.d != 1:
            raise L.RlsdeError(f"a TabularPolicy is a 1-D control; env.d = {env.d}")
    else:
        d, H = R.policy_shape(model)
        if d != env.d:
            raise L.RlsdeError(f"policy dimension {d} != env.d {env.d}")
    if bridge:
        R._check_bridge(env.d)
    rule = L.HIT_X0_IN_LB_RB if env.d == 1 else L.HIT_ALL_GE_LB      # environments.py:48-49 / environments_2d.py:56-57
    env_c = R.env_struct(env, rule)
    dev = R._cuda_device(device)
    if noise is not None:
        noise = torch.as_tensor(np.ascontiguousarray(noise, dtype=np.float32)) if not torch.is_tensor(noise) else noise
        noise = noise.to(device=dev, dtype=torch.float32).contiguous()
    grid = None
    if policy_opt is not None:
        if env.d != 1:
            raise L.RlsdeError("the policy l2 error lookup is defined for the 1-D state grid only (environments.py:318-321)")
        grid = (env.state_space_low, env.state_space_high, env.h_state)
    opts = dict(seed=_next_seed(seed), n_steps_lim=int(k_max), noise=noise, state_f64=state_f64, policy_opt=policy_opt,
                want_logw=want_logw, stoch_int=stoch_int, device=dev, bridge=bridge)
    if dist is not None:
        opts.update(traj_offset=dist.traj_offset, K_global=dist.K_global)
    if table:
        if grid is not None and tuple(float(v) for v in grid) != model.grid:
            raise L.RlsdeError(f"policy_opt lives on grid {grid}, the TabularPolicy on {model.grid}: they must share one")
        out = R.rollout_forward_table(env_c, model.table, int(batch_size), grid=model.grid, **opts)
    else:
        params_host = R.flat_parameters(model).detach().to("cpu", torch.float32).contiguous().numpy()
        out = R.rollout_forward(env_c, L.make_mlp(d, H), params_host, int(batch_size), tanh=tanh, kernel=kernel, grid=grid,
                                **opts)
    stats = out.stats_dev
    if dist is not None:
        stats = dist.all_reduce_stats(stats.clone())
    return out, stats.cpu().numpy()


def test_policy_vectorized(env, model, batch_size=10, k_max=10**7, policy_opt=None, *, noise=None, seed=None,
                           tanh="precise", state_f64=True, device=None, dist=None, kernel="auto", bridge=False):
    """``(mean return, var return (ddof=0), mean hit index[, mean policy l2 error])``; all-NaN if any
    trajectory has not reached the target set within ``k_max`` passes (reference :640-643).  ``bridge=True`` also detects
    hits between passes (Brownian-bridge crossing test, d = 1: ``rollout.rollout_forward``).

    Unlike the reference (which crashes at :610-611), ``policy_opt=None`` is accepted and returns the
    3-tuple its last branch (:647-648) intends."""
    _, st = _numpy_path_rollout(env, model, batch_size, k_max, policy_opt, noise=noise, seed=seed, tanh=tanh, kernel=kernel,
                                state_f64=state_f64, device=device, dist=dist, bridge=bridge)
    n_out = 4 if policy_opt is not None else 3
    if st[L.ST_N_UNFINISHED] > 0:
        return (np.nan,) * n_out
    n = st[L.ST_N]
    mean_ret = st[L.ST_SUM_G] / n
    var_ret = st[L.ST_SUM_G2] / n - mean_ret * mean_ret
    res = (np.float64(mean_ret), np.float64(max(var_ret, 0.0)), np.float64(st[L.ST_SUM_T] / n))
    if policy_opt is not None:
        res += (np.float64(st[L.ST_SUM_L2] / n),)
    return res


test_policy_vectorized.__test__ = False     # not a pytest test, despite the reference's name


def estimate_fht_vectorized(env, model, batch_size=int(1e5), k_max=10**7, *, noise=None, seed=None, tanh="precise", kernel="auto",
                            state_f64=True, device=None, dist=None, bridge=False):
    """Mean first hitting time ``mean(dt * k*)`` (reference :650-695).  NaN if a trajectory is unfinished
    (the reference would average uninitialised ``np.empty`` slots).  ``bridge``: as in ``test_policy_vectorized``."""
    out, st = _numpy_path_rollout(env, model, batch_size, k_max, None, noise=noise, seed=seed, tanh=tanh, kernel=kernel,
                                  state_f64=state_f64, device=device, dist=dist, bridge=bridge)
    if st[L.ST_N_UNFINISHED] > 0:
        return np.nan
    if dist is None:
        # the reference's own expression, np.mean(dt * ep_fhts) with int32 hit indices (:695): identical rounding
        return np.mean(env.dt * out.T.cpu().numpy())
    return np.float64(env.dt * st[L.ST_SUM_T] / st[L.ST_N])


def is_estimate(env, model, batch_size, n_steps_lim=10**7, *, noise=None, seed=None, tanh="precise", state_f64=False, kernel="auto",
                device=None, dist=None, bridge=False):
    """Importance-sampling estimate of Psi(x0) = E[exp(-tau)] under the policy's change of measure
    (SURVEY App. C): weights exp(G - S_exact).  Returns a dict with the estimator mean, its relative
    error std/mean, return statistics, mean hitting index and the unfinished count.  ``bridge=True`` also detects hits
    between passes (Brownian-bridge crossing test, d = 1), which removes the O(sqrt(dt)) bias of a hit tested only on the
    time grid; the weights stay exact, so every policy estimates the same Psi."""
    _, st = _numpy_path_rollout(env, model, batch_size, n_steps_lim, None, noise=noise, seed=seed, tanh=tanh, kernel=kernel,
                                state_f64=state_f64, device=device, dist=dist, stoch_int="exact", want_logw=True,
                                bridge=bridge)
    return R.summarize(st)


def sample_transitions(env, model, batch_size, n_max, *, noise=None, seed=None, tanh="precise", state_f64=True,
                       order="reference", device=None):
    """Device-resident ``rollout.Transitions`` of ``batch_size`` episodes under the policy (NumPy-path arithmetic)."""
    d, H = R.policy_shape(model)
    if d != env.d:
        raise L.RlsdeError(f"policy dimension {d} != env.d {env.d}")
    rule = L.HIT_X0_IN_LB_RB if env.d == 1 else L.HIT_ALL_GE_LB
    env_c = R.env_struct(env, rule)
    mlp_c = L.make_mlp(d, H)
    dev = R._cuda_device(device)
    params_host = R.flat_parameters(model).detach().to("cpu", torch.float32).contiguous().numpy()
    if noise is not None:
        noise = torch.as_tensor(np.ascontiguousarray(noise, dtype=np.float32)) if not torch.is_tensor(noise) else noise
        noise = noise.to(device=dev, dtype=torch.float32).contiguous()
    return R.rollout_transitions(env_c, mlp_c, params_host, int(batch_size), seed=_next_seed(seed), n_max=int(n_max),
                                 noise=noise, tanh=tanh, state_f64=state_f64, order=order, device=dev)


def sample_trajectories_buffer_vectorized(env, model, replay_buffer, batch_size, n_max, *, noise=None, seed=None,
                                          tanh="precise", state_f64=True, device=None):
    """Roll ``batch_size`` episodes out (at most ``n_max`` passes each) and append every transition to ``replay_buffer``
    through its ``store_vectorized`` -- one call with the tuples in the reference's pass-major order (:513-545).

    ``replay_buffer`` is a host ``ReplayBuffer`` (NumPy arrays, like the reference's) or a ``DeviceReplayBuffer``
    (the tuples then never leave the GPU).  Returns the number of transitions stored."""
    from .replay_buffers import DeviceReplayBuffer
    tr = sample_transitions(env, model, batch_size, n_max, noise=noise, seed=seed, tanh=tanh, state_f64=state_f64,
                            order="reference", device=device)
    if isinstance(replay_buffer, DeviceReplayBuffer):
        replay_buffer.store_vectorized(tr.states, tr.actions, tr.rewards, tr.next_states, tr.done)
    else:
        replay_buffer.store_vectorized(tr.states.cpu().numpy(), tr.actions.cpu().numpy(), tr.rewards.cpu().numpy(),
                                       tr.next_states.cpu().numpy(), tr.done.cpu().numpy())
    return len(tr)
