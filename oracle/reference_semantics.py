"""CPU restatement of the reference's hot path -- TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline legs may import this
module; nothing under ``rl_sde_is_b200/`` does (the product path fails loudly without the CUDA
library instead of falling back to this).

Parity pinning: every function here is checked bit-for-bit (values) against fixtures recorded from
the UNMODIFIED reference (tests/golden/make_golden.py -> tests/golden/*.npz; tests/test_oracle_golden.py),
so "matches the oracle" means "matches riberaborrell/rl-sde-is v1.0.0 on numpy 2.3 / torch 2.11".

The restatement is functional and noise-explicit: every sampler takes the Brownian increments
``noise[n_pass, K, d]`` that the reference would have drawn (environments.py:145,208) instead of
drawing them, and returns per-trajectory arrays instead of only their means.

Citations are into /root/reference/src/rl_sde_is/.
"""
import numpy as np
import torch
from scipy.special import ndtr


# --------------------------------------------------------------------------------------------------
# policy:  a = W3 tanh(W2 tanh(W1 x + b1) + b2) + b3            models.py:4-18
# --------------------------------------------------------------------------------------------------
PARAM_KEYS = ("policy.0.weight", "policy.0.bias", "policy.2.weight", "policy.2.bias", "policy.4.weight", "policy.4.bias")


def params_from_npz(npz, prefix):
    """dict of float32 torch tensors from ``<prefix>param.<key>`` fixture entries."""
    return {k: torch.from_numpy(np.array(npz[f"{prefix}param.{k}"], dtype=np.float32)) for k in PARAM_KEYS}


def flatten_params(params):
    return np.concatenate([np.asarray(params[k].detach().numpy() if torch.is_tensor(params[k]) else params[k],
                                      dtype=np.float32).reshape(-1) for k in PARAM_KEYS])


def policy_torch(params, x):
    lin = torch.nn.functional.linear
    h = torch.tanh(lin(x, params["policy.0.weight"], params["policy.0.bias"]))
    h = torch.tanh(lin(h, params["policy.2.weight"], params["policy.2.bias"]))
    return lin(h, params["policy.4.weight"], params["policy.4.bias"])


# --------------------------------------------------------------------------------------------------
# torch path: sample_loss_vectorized + backward     reinforce_deterministic_core.py:30-93, :240
# --------------------------------------------------------------------------------------------------
def rollout_loss_torch(d, alpha, beta, dt, params, noise, lb=1.0, x0=-1.0, need_grad=True):
    """Replay of the reference's torch rollout on recorded increments.

    Per pass n = 1, 2, ... (SURVEY App. A): u = policy(X); X' = X + (-gradV(X) + sigma u) dt + sigma dB
    (environments.py:212-214); done is tested on the CURRENT state (:217-218); the running return adds
    -(1 + |u|^2/2) dt unless done (:121-127); the stochastic integral adds u . dB on every pass, the
    detection pass included (:64-67); the first pass on which done is seen fixes return_fht,
    stoch_int_fht and time_steps = n (:70-81).  All float32.

    Returns dict(loss, return_fht[K] f32, stoch_int_fht[K] f32, time_steps[K] (1-based; 0 = never hit),
    grads{key: ndarray} if need_grad).
    """
    noise = torch.as_tensor(np.asarray(noise, dtype=np.float32))
    n_pass, K, dd = noise.shape
    assert dd == d
    p = {k: v.clone().requires_grad_(need_grad) for k, v in params.items()}
    dt_t = torch.tensor(dt, dtype=torch.float32)                      # environments.py:23
    sigma_t = torch.tensor(np.sqrt(2.0 / beta), dtype=torch.float32)  # :18-19
    # 1-D: python float 4*alpha times an f32 tensor; d-D: 4 * alpha_tensor (f32) -- the same f32 number
    c4a = torch.tensor(np.full(d, 4.0 * alpha), dtype=torch.float32)
    x = torch.full((K, d), float(x0), dtype=torch.float32)
    G_run = torch.zeros(K)
    S_run = torch.zeros(K)
    G_fht = torch.zeros(K)
    S_fht = torch.zeros(K)
    steps = np.zeros(K, dtype=np.int64)
    seen = torch.zeros(K, dtype=torch.bool)
    for n in range(1, n_pass + 1):
        dB = noise[n - 1]
        u = policy_torch(p, x)
        grad_v = c4a * x * (x ** 2 - 1)                                # :45-46 / environments_2d.py:53-54
        x_next = x + (-grad_v + sigma_t * u) * dt_t + sigma_t * dB     # :212-214
        done = (x >= lb).all(dim=1)                                    # :51-52 / environments_2d.py:59-60
        running = -(torch.ones(K) + 0.5 * torch.linalg.norm(u, dim=1) ** 2) * dt_t
        G_run = G_run + torch.where(done, -torch.zeros(K), running)    # :61, :121-127
        S_run = S_run + torch.matmul(u[:, None, :], dB[:, :, None]).squeeze()   # :64-67
        fresh = done & ~seen                                           # :70, environments.py:239-248
        if fresh.any():
            G_fht = torch.where(fresh, G_run, G_fht)
            S_fht = torch.where(fresh, S_run, S_fht)
            steps[fresh.numpy()] = n
            seen = seen | fresh
        if bool(seen.all()):
            break
        x = x_next                                                     # :88 (never detached)
    loss = torch.mean(-G_fht - G_fht.detach() * S_fht)                 # :91
    out = dict(loss=loss.detach().numpy().copy(), return_fht=G_fht.detach().numpy().copy(),
               stoch_int_fht=S_fht.detach().numpy().copy(), time_steps=steps, all_hit=bool(seen.all()))
    if need_grad:
        loss.backward()
        out["grads"] = {k: v.grad.detach().numpy().copy() for k, v in p.items()}
    return out


# --------------------------------------------------------------------------------------------------
# numpy path: test_policy_vectorized / estimate_fht_vectorized        approximate_methods.py:577-695
# --------------------------------------------------------------------------------------------------
def rollout_stats_numpy(d, alpha, beta, dt, params, noise, policy_opt=None, h_state=None, lb=1.0, rb=2.0,
                        lo=-2.0, hi=2.0, x0=-1.0):
    """Replay of the reference's NumPy rollout on recorded increments.

    dtypes follow numpy >= 2 promotion (SURVEY App. A-5): the state starts float32 (environments.py:30)
    and becomes float64 after the first pass because sigma is np.float64 (:18, :148-150); the policy
    input is cast back to float32 every pass (approximate_methods.py:601); accumulators are float64.
    Hit rule: 1-D ``lb <= x <= rb`` (environments.py:48-49), d-D ``all(x >= lb)`` (environments_2d.py:56-57).
    ``ep_lens`` is the 0-based pass index (approximate_methods.py:597,627).

    Returns dict(ep_rets[K], ep_lens[K] (-1 = never hit), l2[K] or None, all_hit).
    """
    noise = np.asarray(noise, dtype=np.float32)
    n_pass, K, dd = noise.shape
    assert dd == d
    sigma = np.sqrt(2.0 / beta)                                        # np.float64
    alpha_v = alpha if d == 1 else np.full(d, alpha)                   # python float (1-D) vs f64 array (d-D)
    states = np.full((K, d), np.float32(x0))                           # float32, approximate_methods.py:594
    total = np.zeros(K)
    ep_rets = np.full(K, np.nan)
    ep_lens = np.full(K, -1, dtype=np.int64)
    l2_run = np.zeros(K)
    l2_fht = np.full(K, np.nan)
    seen = np.zeros(K, dtype=bool)
    for k in range(n_pass):
        with torch.no_grad():
            actions = policy_torch(params, torch.FloatTensor(states)).numpy()      # :600-601
        dbt = noise[k]
        nxt = states + (-(4 * alpha_v * states * (states ** 2 - 1)) + sigma * actions) * dt + sigma * dbt   # :148-150
        if d == 1:
            done = (states[:, 0] >= lb) & (states[:, 0] <= rb)
        else:
            done = (states >= lb).all(axis=1)
        running = -(np.ones(K) + 0.5 * np.linalg.norm(actions, axis=1) ** 2) * dt   # :104-110
        total += np.where(done, -np.zeros(K), running)                               # :607
        if policy_opt is not None:
            idx = np.floor((np.clip(states, lo, hi) - lo) / h_state).astype(int)[:, 0]   # environments.py:318-321
            l2_run += (np.linalg.norm(actions - policy_opt[idx], axis=1) ** 2) * dt      # :610-615
        fresh = done & ~seen
        if fresh.any():
            ep_rets[fresh] = total[fresh]
            ep_lens[fresh] = k
            l2_fht[fresh] = l2_run[fresh]
            seen |= fresh
        if seen.all():
            break
        states = nxt
    return dict(ep_rets=ep_rets, ep_lens=ep_lens, l2=l2_fht if policy_opt is not None else None, all_hit=bool(seen.all()))


# --------------------------------------------------------------------------------------------------
# high-precision replay: the same rollout in float64 (or any dtype), batched, on any device
# --------------------------------------------------------------------------------------------------
HIT_ALL_GE_LB, HIT_X0_IN_LB_RB = "all_ge_lb", "x0_in_lb_rb"


def rollout_reference(d, alpha, beta, dt, params, noise, *, hit_rule=HIT_ALL_GE_LB, lb=1.0, rb=2.0, x0=-1.0,
                      n_steps_lim=None, hit_index=None, f32_policy_input=False, policy_opt=None, grid=None,
                      keep_path=False, keep_margin=False, grad_modes=(), dtype=torch.float64, device="cpu"):
    """The rollout the kernels compute, evaluated in ``dtype`` (float64 by default) from the float32 policy parameters and
    the float32 increments ``noise[n_pass, K, d]`` (cast to ``dtype``).  Unlike the float32 replays above, which
    reproduce the reference's own rounding, this one is the yardstick for the size of the kernels' rounding.

    Per pass k (0-based), on the CURRENT state x_k: the hit test (``hit_rule`` all(x >= lb), or lb <= x_0 <= rb);
    u_k = policy(x_k) (with ``f32_policy_input`` the policy sees x_k cast to float32, as in the NumPy path); then
    x_{k+1} = x_k + (-grad V(x_k) + sigma u_k) dt + sigma dB_k.  On the first hit pass k*:
        T = k*,   G = -sum_{j<k*} (1 + |u_j|^2 / 2) dt,   S_exact = sum_{j<k*} u_j . dB_j,
        S_ref = S_exact + u_k* . dB_k*,   l2 = sum_{j<=k*} |u_j - policy_opt[idx(x_j)]|^2 dt,   logw = G - S_exact.
    No hit within lim = min(n_steps_lim, n_pass) passes: T = -1, G and S (both modes) over all lim passes, logw = G - S.

    ``hit_index`` (int[K], -1 = never) teacher-forces the pass on which each trajectory stops, so that outputs can be
    compared with a kernel's along the kernel's own hit passes.  Whatever stops a trajectory, the function returns its own
    decisions.  The margin of a state is its signed distance to the target boundary (>= 0 means "in the target set");
    ``T_own`` is the first pass with margin >= 0 among the passes a trajectory ran (-1 = none), and ``margin_first`` the
    margin at the first pass where the own decision and the forced stop disagree (pass min(T_own, T); NaN where they never
    do), i.e. how close the reference's state was to deciding the other way.  ``keep_margin``: also return the margin of
    every decision pass, ``margin[n_run, K]`` (NaN after a trajectory stopped).
    ``grid = (lo, hi, h)`` with ``policy_opt[n_grid, d]``: idx(x) = floor((clip(x_0, lo, hi) - lo) / h) (clamped).
    ``keep_path``: also return ``path[K, n_run, d]``, the states x_0 .. x_{n_run - 1}.
    ``grad_modes`` (any of 'reference', 'exact'): autograd of mean_i(-G_i - sg(G_i) S_i) over all K trajectories
    (unfinished ones contribute 0), with S = S_ref or S_exact, w.r.t. the parameters: ``grads[mode][key]`` float64 arrays.

    Returns a dict of ``dtype`` tensors on ``device`` (T, T_own int64)."""
    dev = torch.device(device)
    noise = torch.as_tensor(np.asarray(noise, dtype=np.float32) if not torch.is_tensor(noise) else noise)
    noise = noise.to(device=dev, dtype=dtype)
    n_pass, K, dd = noise.shape
    assert dd == d
    lim = n_pass if n_steps_lim is None else min(int(n_steps_lim), n_pass)
    p = {k: torch.as_tensor(np.asarray(v.detach().cpu().numpy() if torch.is_tensor(v) else v, dtype=np.float32))
         .to(device=dev, dtype=dtype).requires_grad_(bool(grad_modes)) for k, v in params.items()}
    sigma, dt_ = float(np.sqrt(2.0 / beta)), float(dt)
    c4a = torch.as_tensor(np.broadcast_to(4.0 * np.asarray(alpha, dtype=np.float64), (d,)).copy(), device=dev, dtype=dtype)
    forced = None
    if hit_index is not None:
        forced = torch.as_tensor(np.asarray(hit_index.cpu() if torch.is_tensor(hit_index) else hit_index, dtype=np.int64),
                                 device=dev)
    pol = None
    if policy_opt is not None:
        pol = torch.as_tensor(np.asarray(policy_opt, dtype=np.float64).reshape(-1, d), device=dev, dtype=dtype)
        g_lo, g_hi, g_h = (float(v) for v in grid)
    x = torch.as_tensor(np.broadcast_to(np.asarray(x0, dtype=np.float64), (d,)).copy(), device=dev, dtype=dtype).expand(K, d)
    zero = torch.zeros(K, device=dev, dtype=dtype)
    G, S, L2 = zero, zero, zero
    G_out, Sx_out, Sr_out, L2_out = zero, zero, zero, zero
    alive = torch.ones(K, dtype=torch.bool, device=dev)
    T = torch.full((K,), -1, dtype=torch.int64, device=dev)
    T_own = torch.full((K,), -1, dtype=torch.int64, device=dev)
    margin = torch.full((lim, K), float("nan"), device=dev, dtype=dtype) if keep_margin else None
    margin_first = torch.full((K,), float("nan"), device=dev, dtype=dtype)
    path = torch.full((K, lim, d), float("nan"), device=dev, dtype=dtype) if keep_path else None
    n_run = 0
    with torch.set_grad_enabled(bool(grad_modes)):
        for k in range(lim):
            if not bool(alive.any()):
                break
            n_run = k + 1
            xd = x.detach()
            if keep_path:
                path[:, k] = xd
            m = xd.min(dim=1).values - lb if hit_rule == HIT_ALL_GE_LB else torch.minimum(xd[:, 0] - lb, rb - xd[:, 0])
            if keep_margin:
                margin[k] = torch.where(alive, m, margin[k])
            own = alive & (m >= 0)
            T_own = torch.where(own & (T_own < 0), torch.full_like(T_own, k), T_own)
            stop = alive & ((forced == k) if forced is not None else own)
            margin_first = torch.where((own != stop) & torch.isnan(margin_first), m, margin_first)
            xin = x.float().to(dtype) if f32_policy_input else x
            u = policy_torch(p, xin)
            dB = noise[k]
            udB = (u * dB).sum(dim=1)
            r = -(1.0 + 0.5 * (u * u).sum(dim=1)) * dt_
            if pol is not None:
                gi = torch.floor((xd[:, 0].clamp(g_lo, g_hi) - g_lo) / g_h).long().clamp(0, pol.shape[0] - 1)
                L2 = L2 + torch.where(alive, ((u - pol[gi]) ** 2).sum(dim=1) * dt_, zero)
            G_out = torch.where(stop, G, G_out)
            Sx_out = torch.where(stop, S, Sx_out)
            Sr_out = torch.where(stop, S + udB, Sr_out)
            L2_out = torch.where(stop, L2, L2_out)
            T = torch.where(stop, torch.full_like(T, k), T)
            alive = alive & ~stop
            G = G + torch.where(alive, r, zero)
            S = S + torch.where(alive, udB, zero)
            x_next = x + (-(c4a * x * (x * x - 1.0)) + sigma * u) * dt_ + sigma * dB
            x = torch.where(alive[:, None], x_next, x)
        done = T >= 0
        G_out = torch.where(done, G_out, G)
        Sx_out = torch.where(done, Sx_out, S)
        Sr_out = torch.where(done, Sr_out, S)
        L2_out = torch.where(done, L2_out, L2)
        out = dict(T=T, T_own=T_own, G=G_out.detach(), S_exact=Sx_out.detach(), S_ref=Sr_out.detach(),
                   logw=(G_out - Sx_out).detach(), l2=L2_out.detach() if pol is not None else None,
                   margin_first=margin_first, margin=margin[:n_run] if keep_margin else None,
                   path=path[:, :n_run] if keep_path else None)
        out["grads"] = {}
        for i, mode in enumerate(grad_modes):
            Ssel = {"reference": Sr_out, "exact": Sx_out}[mode]
            loss = torch.where(done, -G_out - G_out.detach() * Ssel, zero).sum() / K
            gs = torch.autograd.grad(loss, [p[k] for k in PARAM_KEYS], retain_graph=i + 1 < len(grad_modes))
            out["grads"][mode] = {k: g.detach().cpu().numpy().astype(np.float64) for k, g in zip(PARAM_KEYS, gs)}
    return out


def transitions_numpy(d, alpha, beta, dt, params, noise, n_max, lb=1.0, rb=2.0, x0=-1.0):
    """Replay of ``sample_trajectories_buffer_vectorized`` (approximate_methods.py:513-545) on recorded increments:
    what ``ReplayBuffer.store_vectorized`` (replay_buffers.py:56-68) has received when the sampler returns.

    Every pass stores the tuples of the episodes whose hit had not been detected BEFORE that pass (the detecting pass
    itself is stored, with done = True and reward -0), in episode order; the float64 next state / reward of the NumPy
    step are cast to the buffer's float32 arrays on assignment.  Returns dict(states, actions, rewards, next_states, done).
    """
    noise = np.asarray(noise, dtype=np.float32)
    K = noise.shape[1]
    sigma = np.sqrt(2.0 / beta)
    alpha_v = alpha if d == 1 else np.full(d, alpha)
    states = np.full((K, d), np.float32(x0))
    seen = np.zeros(K, dtype=bool)
    cols = {k: [] for k in ("states", "actions", "rewards", "next_states", "done")}
    for k in range(min(int(n_max), noise.shape[0])):
        with torch.no_grad():
            actions = policy_torch(params, torch.FloatTensor(states)).numpy()
        nxt = states + (-(4 * alpha_v * states * (states ** 2 - 1)) + sigma * actions) * dt + sigma * noise[k]
        done = ((states[:, 0] >= lb) & (states[:, 0] <= rb)) if d == 1 else (states >= lb).all(axis=1)
        running = -(np.ones(K) + 0.5 * np.linalg.norm(actions, axis=1) ** 2) * dt
        r = np.where(done, -np.zeros(K), running)
        live = ~seen
        cols["states"].append(states[live].astype(np.float32))
        cols["actions"].append(actions[live].astype(np.float32))
        cols["rewards"].append(r[live].astype(np.float32))
        cols["next_states"].append(nxt[live].astype(np.float32))
        cols["done"].append(done[live])
        seen |= done
        if seen.all():
            break
        states = nxt
    return {k: np.concatenate(v, axis=0) for k, v in cols.items()}


def test_policy_result(stats, with_l2):
    """The reference's return tuple (approximate_methods.py:640-648) from ``rollout_stats_numpy`` output."""
    if not stats["all_hit"]:
        return (np.nan,) * (4 if with_l2 else 3)
    res = (np.mean(stats["ep_rets"]), np.var(stats["ep_rets"]), np.mean(stats["ep_lens"]))
    return res + ((np.mean(stats["l2"]),) if with_l2 else ())


# --------------------------------------------------------------------------------------------------
# single passes: env.step / env.step_torch                       environments.py:139-162, 201-226
# --------------------------------------------------------------------------------------------------
def env_step_numpy(d, alpha, beta, dt, state, action, dbt, reward_type="state-action", lb=1.0, rb=2.0):
    sigma = np.sqrt(2.0 / beta)
    alpha_v = alpha if d == 1 else np.full(d, alpha)
    nxt = state + (-(4 * alpha_v * state * (state ** 2 - 1)) + sigma * action) * dt + sigma * dbt
    probe = state if reward_type == "state-action" else nxt
    done = ((probe[:, 0] >= lb) & (probe[:, 0] <= rb)) if d == 1 else (probe >= lb).all(axis=1)
    running = -(np.ones(state.shape[0]) + 0.5 * np.linalg.norm(action, axis=1) ** 2) * dt
    r = np.where(done, -np.zeros(state.shape[0]), running) if reward_type == "state-action" else running
    return nxt, r, done


def env_step_torch(d, alpha, beta, dt, state, action, dbt, reward_type="state-action", lb=1.0):
    dt_t = torch.tensor(dt, dtype=torch.float32)
    sigma_t = torch.tensor(np.sqrt(2.0 / beta), dtype=torch.float32)
    c4a = torch.tensor(np.full(d, 4.0 * alpha), dtype=torch.float32)
    nxt = state + (-(c4a * state * (state ** 2 - 1)) + sigma_t * action) * dt_t + sigma_t * dbt
    probe = state if reward_type == "state-action" else nxt
    done = (probe >= lb).all(dim=1)
    running = -(torch.ones(state.shape[0]) + 0.5 * torch.linalg.norm(action, dim=1) ** 2) * dt_t
    r = torch.where(done, -torch.zeros(state.shape[0]), running) if reward_type == "state-action" else running
    return nxt, r, done


# --------------------------------------------------------------------------------------------------
# tables: compute_r_table / compute_p_tensor_batch                  dynamic_programming.py:3-36
# --------------------------------------------------------------------------------------------------
def r_table(state_grid, action_grid, is_in_ts, dt):
    """R[s, a] = -g = -0 on the target set, else -(f + |a|^2/2) dt  (environments.py:104-110), float64."""
    run = -(1.0 + 0.5 * np.abs(action_grid) ** 2) * dt
    out = np.broadcast_to(run, (state_grid.shape[0], action_grid.shape[0])).copy()
    out[is_in_ts, :] = -0.0
    return out


def p_tensor(state_grid, action_grid, is_in_ts, alpha, beta, dt, h_state, sprime=None, s_idx=None, a_idx=None):
    """P[s', s, a] (dynamic_programming.py:18-36 with environments.py:87-102), vectorised over all columns.

    Optional index arrays restrict the computation to a sub-block (the full h = 0.01 tensor is 773 MB):
    ``sprime`` next-state indices, ``s_idx`` state indices, ``a_idx`` action indices.
    """
    Ns = state_grid.shape[0]
    sp = np.arange(Ns) if sprime is None else np.asarray(sprime)
    ss = np.arange(Ns) if s_idx is None else np.asarray(s_idx)
    aa = np.arange(action_grid.shape[0]) if a_idx is None else np.asarray(a_idx)
    sigma = np.sqrt(2.0 / beta)
    h = h_state / 2                                                    # dynamic_programming.py:34
    xs = state_grid[ss][:, None]
    act = action_grid[aa][None, :]
    mu = xs + (-(4 * alpha * xs * (xs ** 2 - 1)) + sigma * act) * dt   # environments.py:90
    sd = sigma * np.sqrt(dt)                                           # :91
    xn = state_grid[sp][:, None, None]
    # scipy.stats.norm.cdf(x, mu, sd) == ndtr((x - mu) / sd)
    prob = ndtr((xn + h - mu[None]) / sd) - ndtr((xn - h - mu[None]) / sd)          # :94-95
    left = ndtr((state_grid[0] - h - mu) / sd)                                        # :98
    right = 1 - ndtr((state_grid[-1] + h - mu) / sd)                                  # :99
    first, last = np.flatnonzero(sp == 0), np.flatnonzero(sp == Ns - 1)
    if first.size:
        prob[first[0]] += left
    if last.size:
        prob[last[0]] += right
    ts_cols = is_in_ts[ss]
    n_ts = int(is_in_ts.sum())
    prob[:, ts_cols, :] = np.where(is_in_ts[sp], 1.0 / n_ts, 0.0)[:, None, None]      # dynamic_programming.py:25-26
    return prob


# --------------------------------------------------------------------------------------------------
# DP sweeps over the tables (SURVEY 8f-1)
# --------------------------------------------------------------------------------------------------
def bellman_values(r_table, p_tensor, is_in_ts, v, gamma):
    """values[s, a] = r[s, a] + (1 - d[s]) gamma sum_s' P[s', s, a] v[s']: the contraction shared by
    q_table_update_vect (tabular_dp_qvalue_iteration.py:35-43), v_table_update_vect (tabular_dp_value_iteration.py:41-52)
    and policy_update_vect (tabular_dp_policy_iteration.py:37-49)."""
    live = 1 - np.where(is_in_ts, 1, 0)[:, None]
    return r_table + live * gamma * np.einsum("psa,p->sa", p_tensor, v)


def q_sweep(r_table, p_tensor, is_in_ts, q, gamma):
    return bellman_values(r_table, p_tensor, is_in_ts, q.max(axis=1), gamma)


def v_sweep(r_table, p_tensor, is_in_ts, v, gamma):
    return bellman_values(r_table, p_tensor, is_in_ts, v, gamma).max(axis=1)


def greedy_policy_indices(r_table, p_tensor, is_in_ts, v, gamma, null_action_idx):
    idx = np.argmax(bellman_values(r_table, p_tensor, is_in_ts, v, gamma), axis=1)
    idx[is_in_ts] = null_action_idx
    return idx
