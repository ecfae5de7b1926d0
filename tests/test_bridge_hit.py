"""The Brownian-bridge hit test between passes (RLSDE_F_HIT_BRIDGE, d = 1) on the CPU: the crossing probability against a
fine-grid simulation of the bridge, the float64 bridge replay (the yardstick of tests/test_gpu_bridge_hit.py) against a
plain NumPy loop, the uniform's Philox counter layout against the C oracle, and the refusals of the C ABI and of Python."""
import inspect

import numpy as np
import pytest
import torch

from oracle import c_oracle
from oracle import reference_semantics as ref

DT = 0.005
BRIDGE_TAG = 0x42524447          # "BRDG": fourth counter word of the uniform's Philox stream
ARG_MAX = 23.0                   # exponents above this give p < 2^-33 <= U: no draw, no crossing
MASK32 = (1 << 32) - 1


def philox(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 on arrays of counters (uint64 arrays holding 32-bit words), the C oracle's rounds vectorised."""
    c0, c1, c2, c3 = (np.asarray(v, dtype=np.uint64) & np.uint64(MASK32) for v in (c0, c1, c2, c3))
    k0, k1 = np.uint64(k0 & MASK32), np.uint64(k1 & MASK32)
    m32 = np.uint64(MASK32)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & m32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & m32
        k0 = (k0 + np.uint64(0x9E3779B9)) & m32
        k1 = (k1 + np.uint64(0xBB67AE85)) & m32
    return c0, c1, c2, c3


def bridge_uniform(seed, traj, k):
    """U = (r.x + 0.5) 2^-32 of Philox(counter (traj_lo, traj_hi, k, "BRDG"), key seed), traj = global trajectory ids."""
    traj = np.asarray(traj, dtype=np.uint64)
    r = philox(traj & np.uint64(MASK32), traj >> np.uint64(32), np.full(traj.shape, k, dtype=np.uint64),
               np.full(traj.shape, BRIDGE_TAG, dtype=np.uint64), int(seed) & MASK32, (int(seed) >> 32) & MASK32)
    return (r[0].astype(np.float64) + 0.5) * 2.0 ** -32


def bridge_replay(policy, noise, *, seed, traj_offset=0, hit_rule=ref.HIT_X0_IN_LB_RB, lb=1.0, rb=2.0, x0=-1.0, dt=DT,
                  alpha=1.0, beta=1.0, n_steps_lim=None, hit_index=None, policy_opt=None, grid=None, bridge=True,
                  dtype=torch.float64, device="cpu"):
    """The d = 1 rollout with the Brownian-bridge hit test, in ``dtype`` (float64) from the float32 increments
    ``noise[n_pass, K, 1]``.  ``policy(x)`` maps the states [K] (``dtype``) to the actions [K].  Per pass k, as
    oracle.reference_semantics.rollout_reference: hit test on x_k, u_k = policy(x_k), accumulators, Euler-Maruyama step
    to b = x_{k+1} from a = x_k; then, if the trajectory goes on, the crossing test: b outside the target on the other
    side of it from a crossed; b beyond the same barrier c as a crossed if U < exp(-2 (c - a)(c - b) / (sigma^2 dt)), U
    from the host Philox stream (drawn where the exponent is <= 23); a crossing sets x_{k+1} = c (c = lb if a < lb,
    else rb).  ``hit_index`` (int[K], -1 = never) teacher-forces the passes on which trajectories stop: a trajectory
    forced to stop at k + 1 whose b lies outside the target crossed (the kernel detected it there), any other did not.
    ``bridge=False`` is the rollout without the test.

    Returns T, G, S_exact, S_ref, logw, l2 (``dtype``) and ``knife``: per trajectory, at the first pass where an own
    decision (grid hit or crossing) differs from the forced one, how close it was (|margin| of the hit test, |U - p| of a
    crossing draw, distance of b to the barrier for a sure crossing); NaN where none differs.  ``n_draws`` counts the
    uniforms drawn, ``n_passes`` the passes that ran the test."""
    dev = torch.device(device)
    noise = torch.as_tensor(np.asarray(noise, dtype=np.float32)).to(device=dev, dtype=dtype)
    n_pass, K, _ = noise.shape
    lim = n_pass if n_steps_lim is None else min(int(n_steps_lim), n_pass)
    sigma = float(np.sqrt(2.0 / beta))
    inv = 1.0 / (sigma * sigma * dt)
    c4a = 4.0 * float(alpha)
    two = hit_rule == ref.HIT_X0_IN_LB_RB
    rb_eff = rb if two else float("inf")
    forced = None if hit_index is None else torch.as_tensor(np.asarray(hit_index, dtype=np.int64), device=dev)
    gids = np.arange(K, dtype=np.uint64) + np.uint64(traj_offset)
    pol = None
    if policy_opt is not None:
        pol = torch.as_tensor(np.asarray(policy_opt, dtype=np.float64).reshape(-1), device=dev, dtype=dtype)
        g_lo, g_hi, g_h = (float(v) for v in grid)
    x = torch.full((K,), float(np.float32(x0)), device=dev, dtype=dtype)
    zero = torch.zeros(K, device=dev, dtype=dtype)
    G, S, L2 = zero, zero, zero
    G_out, Sx_out, Sr_out, L2_out = zero, zero, zero, zero
    alive = torch.ones(K, dtype=torch.bool, device=dev)
    T = torch.full((K,), -1, dtype=torch.int64, device=dev)
    knife = torch.full((K,), float("nan"), device=dev, dtype=dtype)
    n_draws = n_passes = 0

    def note(mask, val):
        nonlocal knife
        knife = torch.where(mask & torch.isnan(knife), val.abs(), knife)

    for k in range(lim):
        if not bool(alive.any()):
            break
        m = torch.minimum(x - lb, rb_eff - x)
        own = alive & (m >= 0)
        stop = alive & ((forced == k) if forced is not None else own)
        note(own != stop, m)
        u = policy(x)
        dB = noise[k, :, 0]
        udB = u * dB
        if pol is not None:
            gi = torch.floor((x.clamp(g_lo, g_hi) - g_lo) / g_h).long().clamp(0, pol.numel() - 1)
            L2 = L2 + torch.where(alive, (u - pol[gi]) ** 2 * dt, zero)
        G_out = torch.where(stop, G, G_out)
        Sx_out = torch.where(stop, S, Sx_out)
        Sr_out = torch.where(stop, S + udB, Sr_out)
        L2_out = torch.where(stop, L2, L2_out)
        T = torch.where(stop, torch.full_like(T, k), T)
        alive = alive & ~stop
        G = G + torch.where(alive, -(1.0 + 0.5 * u * u) * dt, zero)
        S = S + torch.where(alive, udB, zero)
        a = x
        b = a + (-(c4a * a * (a * a - 1.0)) + sigma * u) * dt + sigma * dB
        if bridge:
            b_lo, b_hi, a_lo = b < lb, b > rb_eff, a < lb
            outside = alive & (b_lo | b_hi)
            c = torch.where(a_lo, torch.full_like(a, lb), torch.full_like(a, rb))
            sure = outside & (a_lo != b_lo)
            arg = 2.0 * (c - a) * (c - b) * inv
            need = outside & ~sure & (arg <= ARG_MAX)
            cross = sure.clone()
            p = torch.exp(-arg)
            U = torch.ones_like(a)
            idx = torch.nonzero(need).flatten().cpu().numpy()
            if idx.size:
                U[idx] = torch.as_tensor(bridge_uniform(seed, gids[idx], k), device=dev, dtype=dtype)
                cross = cross | (need & (U < p))
            n_draws += int(idx.size)
            n_passes += int(alive.sum())
            if forced is not None:
                want = outside & (forced == k + 1)
                note(want != cross, torch.where(sure, (b - c), U - p))
                cross = want
            b = torch.where(cross, c, b)
        x = torch.where(alive, b, x)
    done = T >= 0
    G_out = torch.where(done, G_out, G)
    Sx_out = torch.where(done, Sx_out, S)
    Sr_out = torch.where(done, Sr_out, S)
    L2_out = torch.where(done, L2_out, L2)
    return dict(T=T, G=G_out, S_exact=Sx_out, S_ref=Sr_out, logw=G_out - Sx_out, l2=L2_out, knife=knife,
                n_draws=n_draws, n_passes=n_passes)


def mlp_policy(params, dtype=torch.float64, f32_input=False):
    """u = policy(x) of the reference MLP (float32 parameters evaluated in ``dtype``); ``f32_input``: the policy sees x
    cast to float32, as the kernels' policy does."""
    p = {k: torch.as_tensor(np.asarray(v, dtype=np.float32)).to(dtype) for k, v in params.items()}

    def f(x):
        xin = x.float().to(x.dtype) if f32_input else x
        pp = {k: v.to(x.device) for k, v in p.items()}
        return ref.policy_torch(pp, xin[:, None])[:, 0]
    return f


def table_policy(table, grid):
    lo, hi, h = (float(v) for v in grid)
    tab = torch.as_tensor(np.asarray(table, dtype=np.float32).reshape(-1)).to(torch.float64)

    def f(x):
        gi = torch.floor((x.clamp(lo, hi) - lo) / h).long().clamp(0, tab.numel() - 1)
        return tab.to(x.device, x.dtype)[gi]
    return f


# ------------------------------------------------------------------------------ the crossing probability
@pytest.mark.parametrize("a,b", [(0.9, 0.95), (0.8, 0.97), (0.95, 0.8), (2.05, 2.12)])
def test_crossing_probability_against_a_simulated_bridge(a, b):
    """p = exp(-2 (c - a)(c - b) / (sigma^2 dt)) against the fraction of 1e5 Brownian bridges from a to b over dt (2 000
    substeps, sigma^2 = 2 / beta = 2) whose maximum (minimum, for c = rb = 2 from above) reaches c, within 4 standard errors
    plus the O(sqrt(dt / n)) bias of the discretely sampled maximum, which the substep count keeps below 1 %."""
    rng = np.random.default_rng(17)
    sigma, n_sub, n_path = np.sqrt(2.0), 2000, 100_000
    c = 1.0 if a < 1.0 else 2.0
    hits = 0
    for chunk in range(10):
        n = n_path // 10
        w = np.cumsum(rng.standard_normal((n, n_sub)) * np.sqrt(DT / n_sub), axis=1)
        t = np.arange(1, n_sub + 1) / n_sub
        path = a + (b - a) * t + sigma * (w - t * w[:, -1:])          # Brownian bridge from a to b
        hits += int(((path >= c).any(axis=1) if c == 1.0 else (path <= c).any(axis=1)).sum())
    frac = hits / n_path
    p = np.exp(-2.0 * (c - a) * (c - b) / (sigma * sigma * DT))
    se = np.sqrt(p * (1 - p) / n_path)
    # a discretely monitored bridge misses excursions: its frequency is below p by about 0.58 sigma sqrt(dt / n) (c - x)
    bias = p * 0.5826 * 2 * sigma * np.sqrt(DT / n_sub) * (abs(c - a) + abs(c - b)) / (sigma * sigma * DT)
    assert 0.05 < p < 0.95
    assert p - bias - 4 * se <= frac <= p + 4 * se, (frac, p, bias, se)
    # the factor 2 is pinned: p^2 and sqrt(p) are far outside
    assert abs(frac - p ** 2) > 10 * se and abs(frac - np.sqrt(p)) > 10 * se


# ------------------------------------------------------------------------------ the replay against a plain loop
def _numpy_bridge_loop(table, grid, noise, seed, lb=1.0, rb=2.0, x0=-1.0, two=True, bridge=True):
    lo, hi, h = grid
    sigma = np.sqrt(2.0)
    inv = 1.0 / (sigma * sigma * DT)
    n_pass, K, _ = noise.shape
    out = {k: np.zeros(K) for k in ("G", "S_exact", "S_ref")}
    out["T"] = np.full(K, -1)
    kinds = {"sure": 0, "drawn": 0, "crossed": 0, "lb": 0, "rb": 0}
    for i in range(K):
        x, G, S = float(np.float32(x0)), 0.0, 0.0
        for k in range(n_pass):
            u = float(table[min(max(int(np.floor((min(max(x, lo), hi) - lo) / h)), 0), len(table) - 1)])
            dB = float(noise[k, i, 0])
            if lb <= x <= (rb if two else np.inf):
                out["T"][i] = k
                out["S_ref"][i] = S + u * dB
                break
            G += -(1.0 + 0.5 * u * u) * DT
            S += u * dB
            a = x
            b = a + (-(4.0 * a * (a * a - 1.0)) + sigma * u) * DT + sigma * dB
            if bridge and (b < lb or (two and b > rb)):
                c = lb if a < lb else rb
                if (a < lb) != (b < lb):
                    kinds["sure"] += 1
                    b = c
                else:
                    arg = 2.0 * (c - a) * (c - b) * inv
                    if arg <= ARG_MAX:
                        kinds["drawn"] += 1
                        U = (int(c_oracle.philox([i & MASK32, i >> 32, k, BRIDGE_TAG], [seed & MASK32, seed >> 32])[0]) + 0.5) * 2.0 ** -32
                        if U < np.exp(-arg):
                            kinds["crossed"] += 1
                            kinds["lb" if c == lb else "rb"] += 1
                            b = c
            x = b
        out["G"][i], out["S_exact"][i] = G, S
        if out["T"][i] < 0:
            out["S_ref"][i] = S
    return out, kinds


@pytest.mark.parametrize("x0,two", [(-1.0, True), (1.6, True), (-1.0, False)])
def test_replay_matches_numpy_loop(x0, two):
    """The vectorised float64 bridge replay against a plain loop that draws each uniform from the C oracle's Philox: same
    hit passes, G / S to 1e-12.  The control pushes states towards and past both barriers of a narrow target, so crossings by
    the sure rule (endpoints on opposite sides), drawn crossings at lb and at rb (x0 = 1.6 starts above rb), and draws that did
    not cross all occur; the loop applies the lazy-draw threshold itself."""
    rng = np.random.default_rng(11)
    K, n_pass, seed = 40, 1200, 0x1234_5678_9ABC
    noise = (np.sqrt(DT) * rng.standard_normal((n_pass, K, 1))).astype(np.float32)
    grid = (-2.0, 3.0, 0.05)
    xs = np.linspace(-2.0, 3.0, 101)
    table = np.where(xs < 1.0, 2.0, -3.0).astype(np.float32)
    rule = ref.HIT_X0_IN_LB_RB if two else ref.HIT_ALL_GE_LB
    rb = 1.03           # a narrow target, so that a pass can jump over it
    got = bridge_replay(table_policy(table, grid), noise, seed=seed, hit_rule=rule, x0=x0, rb=rb)
    want, kinds = _numpy_bridge_loop(table, grid, noise.astype(np.float64), seed, x0=x0, two=two, rb=rb)
    assert np.array_equal(got["T"].numpy(), want["T"])
    for key in ("G", "S_exact", "S_ref"):
        assert np.allclose(got[key].numpy(), want[key], rtol=0, atol=1e-12), key
    assert kinds["drawn"] > kinds["crossed"] > 0, kinds
    assert kinds["lb" if x0 < 1.0 else "rb"] > 0, kinds
    if two:
        assert kinds["sure"] > 0, kinds
    assert got["n_draws"] == kinds["drawn"]
    # the bridge only ever stops trajectories earlier
    plain = bridge_replay(table_policy(table, grid), noise, seed=seed, hit_rule=rule, x0=x0, rb=rb, bridge=False)
    t_b, t_p = got["T"].numpy(), plain["T"].numpy()
    t_p = np.where(t_p < 0, n_pass, t_p)
    assert (np.where(t_b < 0, n_pass, t_b) <= t_p).all() and (t_b < t_p).any()


def test_teacher_forcing_follows_the_forced_passes():
    """Forced onto its own hit passes the replay reproduces itself with no knife edge; forced one pass later on a
    trajectory that crossed, it reports the disagreement."""
    rng = np.random.default_rng(3)
    noise = (np.sqrt(DT) * rng.standard_normal((800, 64, 1))).astype(np.float32)
    pol = table_policy(np.full(5, 1.5, dtype=np.float32), (-2.0, 2.0, 1.0))
    own = bridge_replay(pol, noise, seed=9)
    again = bridge_replay(pol, noise, seed=9, hit_index=own["T"].numpy())
    for key in ("T", "G", "S_exact", "S_ref"):
        assert torch.equal(own[key], again[key]), key
    assert torch.isnan(again["knife"]).all()
    T = own["T"].numpy().copy()
    i = int(np.flatnonzero(T > 0)[0])
    T[i] += 1
    moved = bridge_replay(pol, noise, seed=9, hit_index=T)
    assert not np.isnan(moved["knife"][i].item())


# ------------------------------------------------------------------------------ the uniform's counter layout
def test_uniform_counter_layout_matches_the_oracle_philox():
    """U of trajectory t (global id, both 32-bit halves used), pass k and seed: Philox(counter (t_lo, t_hi, k, "BRDG"),
    key (seed_lo, seed_hi)), first word, (r + 0.5) 2^-32 -- the vectorised generator against c_oracle.philox."""
    rng = np.random.default_rng(0)
    for _ in range(50):
        t = int(rng.integers(0, 1 << 40))
        k = int(rng.integers(0, 1 << 31))
        seed = int(rng.integers(0, 1 << 63))
        r = c_oracle.philox([t & MASK32, t >> 32, k, BRIDGE_TAG], [seed & MASK32, seed >> 32])
        assert bridge_uniform(seed, np.array([t], dtype=np.uint64), k)[0] == (float(r[0]) + 0.5) * 2.0 ** -32
    u = bridge_uniform(5, np.arange(100_000, dtype=np.uint64), 7)
    assert 2.0 ** -33 <= u.min() and u.max() < 1.0 and abs(u.mean() - 0.5) < 0.005


# ------------------------------------------------------------------------------ refusals
def test_c_abi_refusals():
    """RLSDE_F_HIT_BRIDGE is refused before any device work: at d = 2 (RLSDE_ERR_UNSUPPORTED), with RLSDE_F_STORE_PATH,
    by the transition stream, the reverse pass and the single-step environment (RLSDE_ERR_INVALID_ARG)."""
    from rl_sde_is_b200 import _lib as L
    lib = L.load()
    fake = 1 << 20                             # never dereferenced: every call below fails its argument checks first
    ws_bytes = int(lib.rlsde_workspace_bytes(64))
    params = np.zeros(1 + 32 + 32 * 32 + 32 + 32 + 1 + 64, dtype=np.float32)
    RLSDE_ERR_INVALID_ARG, RLSDE_ERR_UNSUPPORTED = -1, -2

    def cfg(flags):
        c = L.RlsdeRolloutCfg()
        c.K, c.K_global, c.n_steps_lim, c.flags = 64, 64, 100, flags
        c.ckpt_every, c.ckpt_stride = 1, 100
        return c

    def env(d):
        return L.make_env(d, 1.0, np.sqrt(2.0), DT, 1.0, 2.0, np.full(d, -1.0), L.HIT_ALL_GE_LB)

    def fwd(d, flags):
        return lib.rlsde_rollout_fwd(env(d), L.make_mlp(d, 32), params.ctypes.data, cfg(flags), 0, 0, fake, fake, fake, 0, 0,
                                     fake, 0, fake, ws_bytes, 0)

    B = L.F_HIT_BRIDGE
    assert fwd(2, B) == RLSDE_ERR_UNSUPPORTED
    assert fwd(1, B | L.F_STORE_PATH) == RLSDE_ERR_INVALID_ARG
    assert lib.rlsde_rollout_transitions(env(1), L.make_mlp(1, 32), params.ctypes.data, cfg(B), 0, fake, fake, fake, fake,
                                         fake, fake, fake, fake, fake, 0, fake, ws_bytes, 0) == RLSDE_ERR_INVALID_ARG
    assert lib.rlsde_rollout_bwd(env(1), L.make_mlp(1, 32), params.ctypes.data, cfg(B | L.F_STORE_PATH), 0, fake, fake, fake,
                                 0, 1.0, fake, fake, 1 << 40, 0) == RLSDE_ERR_INVALID_ARG
    assert lib.rlsde_env_step(env(1), 64, fake, fake, 0, 1, 0, 0, B, 0, fake, fake, fake, 0, 0) == RLSDE_ERR_INVALID_ARG
    tab_env = L.make_env(2, 1.0, np.sqrt(2.0), DT, 1.0, 2.0, np.full(2, -1.0), L.HIT_ALL_GE_LB)
    c = cfg(B)
    c.n_grid, c.grid_lo, c.grid_hi, c.grid_h = 401, -2.0, 2.0, 0.01
    assert lib.rlsde_rollout_fwd_table(tab_env, fake, c, 0, 0, fake, fake, fake, 0, 0, 0, fake, ws_bytes, 0) == RLSDE_ERR_UNSUPPORTED


def test_python_refusals():
    """bridge=True at d = 2 raises RlsdeError before any launch; the training paths have no bridge keyword at all."""
    from rl_sde_is_b200 import _lib as L
    from rl_sde_is_b200 import approximate_methods as am, rollout as R
    from rl_sde_is_b200.environments import DoubleWellStoppingTime2D
    from rl_sde_is_b200.models import DeterministicPolicy
    from rl_sde_is_b200.reinforce_deterministic_core import reinforce, sample_loss_vectorized
    env2 = DoubleWellStoppingTime2D(beta=1.0, alpha=1.0, dt=DT)
    model = DeterministicPolicy(2, 2, [32, 32], torch.nn.Tanh())
    with pytest.raises(L.RlsdeError, match="d = 1"):
        am.is_estimate(env2, model, 16, bridge=True)
    with pytest.raises(L.RlsdeError, match="d = 1"):
        am.test_policy_vectorized(env2, model, 16, bridge=True)
    with pytest.raises(L.RlsdeError, match="d = 1"):
        R.rollout_forward(L.make_env(2, 1.0, 1.0, DT, 1.0, 2.0, [-1.0, -1.0], 0), L.make_mlp(2, 32),
                          R.flat_parameters(model).detach().numpy(), 16, bridge=True)
    with pytest.raises(L.RlsdeError, match="store_path"):
        R.rollout_forward(L.make_env(1, 1.0, 1.0, DT, 1.0, 2.0, [-1.0], 0), L.make_mlp(1, 32), np.zeros(1153, np.float32), 16,
                          bridge=True, store_path=True)
    for fn in (sample_loss_vectorized, reinforce, R.rollout_loss_and_grad):
        assert "bridge" not in inspect.signature(fn).parameters, fn.__name__
    for fn in (am.test_policy_vectorized, am.estimate_fht_vectorized, am.is_estimate, R.rollout_forward, R.rollout_forward_table):
        assert inspect.signature(fn).parameters["bridge"].kind == inspect.Parameter.KEYWORD_ONLY, fn.__name__
