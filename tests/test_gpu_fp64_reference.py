"""Every rollout kernel against the float64 reference rollout (oracle/reference_semantics.rollout_reference, pinned on the
reference's fixtures by tests/test_reference_f64.py), on the kernels' own increments.

The other GPU tests compare kernels with the reference's float32 arithmetic (parity) or with each other (schedules,
families).  Here the yardstick has no rounding of its own at float32 scale, so a systematic error -- a wrong term in the
importance weight, the detecting pass's u . dB in the exact-mode integral or in its gradient, a dropped statistics field --
shows up however small, and each test also shows that the nearest wrong answer would fail its tolerance.

Per-trajectory tolerances scale with the passes a trajectory executed: ``C (n + 1) 2^-24 (1 + |value|)``.  Each constant is
written beside the largest error measured over every case of its test on an NVIDIA B200 (1000 W power limit, max SM clock
1965 MHz); the wrong answers that the discrimination asserts check exceed the same bounds by 40x or more."""
import math

import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import reference_semantics as ref

pytestmark = pytest.mark.gpu

EPS32 = 2.0 ** -24
DT = 0.005


@pytest.fixture(autouse=True)
def _no_schedule_overrides(monkeypatch):
    """The binding falls back to these variables for any scheduling knob a call leaves unset; the families and schedules
    each test forces must not depend on the caller's environment."""
    for name in ("FWD_QUANTUM", "FWD_HANDOFF", "BWD_WARP_SHARE", "FWD_BLOCKS_PER_SM", "BWD_KERNEL", "WIDE_KERNEL"):
        monkeypatch.delenv("RLSDE_" + name, raising=False)


def _lib():
    from rl_sde_is_b200 import _lib as L, rollout as R
    return L, R


def _policy(d, H, bias, seed):
    from rl_sde_is_b200.models import DeterministicPolicy
    torch.manual_seed(seed)
    m = DeterministicPolicy(d, d, [H, H], nn.Tanh())
    m.policy[4].bias.data.fill_(bias)
    params = {k: v.detach().clone() for k, v in m.state_dict().items()}
    return m, params, ref.flatten_params(params)


# The environment every case runs in unless it names another (tests/test_gpu_env_params.py): the reference's defaults.
# ``alpha`` and ``x0`` may also be per-coordinate sequences.
DEFAULT_ENV = dict(alpha=1.0, beta=1.0, dt=DT, x0=-1.0, lb=1.0, rb=2.0)


def _spec(env):
    return {**DEFAULT_ENV, **(env or {})}


def _env_c(d, hit_rule, env=None):
    """The environment object of the spec ``env`` (keys of DEFAULT_ENV; absent keys take their default) and its rlsde_env.
    A per-coordinate alpha overwrites ``alpha`` / ``alpha_tensor`` of the d-D class, a per-coordinate x0 its float32
    ``state_init``: the attributes rollout.env_struct reads."""
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D, DoubleWellStoppingTimeND
    L, R = _lib()
    s = _spec(env)
    alpha = np.asarray(s["alpha"], dtype=np.float64)
    a0 = float(alpha.reshape(-1)[0])
    e = DoubleWellStoppingTime1D(beta=s["beta"], alpha=a0, dt=s["dt"]) if d == 1 else \
        DoubleWellStoppingTimeND(d, beta=s["beta"], alpha=a0, dt=s["dt"])
    if alpha.ndim:
        assert d > 1 and alpha.shape == (d,)
        e.alpha = alpha.copy()
        e.alpha_tensor = torch.tensor(e.alpha, dtype=torch.float32)
    e.state_init = np.broadcast_to(np.asarray(s["x0"], dtype=np.float32), (1, d)).copy()
    e.lb, e.rb = float(s["lb"]), float(s["rb"])
    return e, R.env_struct(e, hit_rule)


def _reference(d, params, noise, env=None, **kw):
    """oracle.reference_semantics.rollout_reference in the environment ``env`` (as _env_c)."""
    s = _spec(env)
    return ref.rollout_reference(d, s["alpha"], s["beta"], s["dt"], params, noise, lb=s["lb"], rb=s["rb"], x0=s["x0"], **kw)


def _bound(n, value, c):
    return c * (np.asarray(n, dtype=np.float64) + 1) * EPS32 * (1.0 + np.abs(value))


def _np(t):
    return t.detach().cpu().numpy().astype(np.float64) if torch.is_tensor(t) else np.asarray(t, dtype=np.float64)


# ------------------------------------------------------------------------------ statistics record, fsum reference
def _fsum_stats(G, S, T, l2, logw, lim):
    """The 16-double statistics record of include/rlsde.h from per-trajectory arrays, every sum by math.fsum."""
    G, S, T = _np(G), _np(S), np.asarray(T.cpu() if torch.is_tensor(T) else T, dtype=np.int64)
    fin = T >= 0
    g, s, t = G[fin], S[fin], T[fin].astype(np.float64)
    st = np.zeros(16)
    st[0], st[1] = T.size, (~fin).sum()
    st[2], st[3] = math.fsum(g), math.fsum(g * g)
    st[4], st[5] = math.fsum(t), math.fsum(t * t)
    st[6] = math.fsum(s)
    st[7] = math.fsum(_np(l2)[fin]) if l2 is not None else 0.0
    if logw is not None:
        w = np.exp(_np(logw)[fin])
        st[8], st[9] = math.fsum(w), math.fsum(w * w)
    st[10] = math.fsum(-g - g * s)
    st[11] = math.fsum(t + 1.0) + float(lim) * (~fin).sum()
    st[12] = t.max() if t.size else 0.0
    scale = np.zeros(16)                     # fsum of |terms|: the size of the rounding a double reduction may make
    scale[[2, 3, 6, 7, 8, 9, 10]] = [math.fsum(np.abs(g)), st[3], math.fsum(np.abs(s)), abs(st[7]), st[8], st[9],
                                     math.fsum(np.abs(g) + np.abs(g * s))]
    return st, scale


EXACT_FIELDS = (0, 1, 4, 5, 11, 12, 13, 14, 15)      # counts, SUM_T, SUM_T2, USEFUL_STEPS, MAX_T, the unused tail


def _assert_stats(got, G, S, T, l2, logw, lim, fields=range(16)):
    want, scale = _fsum_stats(G, S, T, l2, logw, lim)
    for f in fields:
        if f in EXACT_FIELDS:
            assert got[f] == want[f], (f, got[f], want[f])
        else:
            assert abs(got[f] - want[f]) <= 1e-12 * scale[f], (f, got[f], want[f])


def _reduce(K, lim, f64, G, S, T, l2, logw):
    L, R = _lib()
    lib = L.load()
    stats = torch.full((16,), float("nan"), dtype=torch.float64, device="cuda")
    ws = R._workspace(torch.device("cuda", torch.cuda.current_device()), K)
    rc = lib.rlsde_reduce_stats(K, lim, L.F_STATE_F64 if f64 else 0, G.data_ptr(), S.data_ptr(), T.data_ptr(),
                                0 if l2 is None else l2.data_ptr(), 0 if logw is None else logw.data_ptr(), stats.data_ptr(),
                                ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
    L.check(rc, "rlsde_reduce_stats")
    return stats.cpu().numpy()


@pytest.mark.parametrize("K", [1, 255, 256, 257, 65535, 65536, 65537, 1_000_003])
@pytest.mark.parametrize("f64", [False, True])
def test_reduce_stats_against_fsum(K, f64):
    """rlsde_reduce_stats on synthetic arrays: one block, exactly one / just over one block of 256, 256 blocks with a short
    last slice (per = ceil(K / 256)), a million trajectories; 0 / 30 / 100 % unfinished; l2 and logw null and present.
    Counts, SUM_T, SUM_T2, USEFUL_STEPS and MAX_T exact, sums within 1e-12 of the fsum of |terms|, fields 13-15 zero,
    repeated calls bit-identical.  With every trajectory unfinished MAX_T is 0 (the reduction's identity)."""
    rng = np.random.default_rng(K + 7 * f64)
    dtype = torch.float64 if f64 else torch.float32
    G = torch.as_tensor(rng.uniform(-50.0, 0.0, K), dtype=dtype, device="cuda")
    S = torch.as_tensor(rng.normal(0.0, 2.0, K), dtype=dtype, device="cuda")
    l2 = torch.as_tensor(rng.uniform(0.0, 3.0, K), dtype=dtype, device="cuda")
    logw = torch.as_tensor(rng.uniform(-40.0, 5.0, K), dtype=dtype, device="cuda")
    T0 = rng.integers(0, 5000, K)
    lim = 5000
    for frac in (0.0, 0.3, 1.0):
        T = torch.as_tensor(np.where(rng.random(K) < frac, -1, T0) if frac < 1 else np.full(K, -1), dtype=torch.int32,
                            device="cuda")
        for with_opt in (False, True):
            a, b = (l2, logw) if with_opt else (None, None)
            st = _reduce(K, lim, f64, G, S, T, a, b)
            _assert_stats(st, G, S, T, a, b, lim)
            assert np.array_equal(st, _reduce(K, lim, f64, G, S, T, a, b))
            if frac == 1.0:
                assert st[1] == K and st[12] == 0.0 and st[2] == 0.0
            if with_opt and frac < 1:
                assert st[8] > 0 and st[9] > 0 and st[7] > 0


# ------------------------------------------------------------------------------ forward kernels, per trajectory
# family -> rollout_forward arguments that force it
FAMILIES = {
    "K1": dict(kernel="thread"),                       # rollout_fwd.cuh
    "K1w": dict(kernel="warp"),                        # rollout_warp.cuh
    "K1u": dict(kernel="tensor"),                      # rollout_umma.cuh, hidden width 32 (traj_owner.cuh)
    "K1x": dict(tuning={"wide_kernel": "ffma"}),       # rollout_wide.cuh
    "K1u_wide": dict(tuning={"wide_kernel": "umma"}),  # rollout_umma.cuh, hidden width 64 / 128 / 256
}
NARROW = [(d, 32) for d in (1, 2, 3, 4, 10)]
WIDE = [(d, H) for d in (1, 2) for H in (64, 128, 256)]
FWD_CASES = [(f, d, H) for f in ("K1", "K1w", "K1u") for d, H in NARROW] + [(f, d, H) for f in ("K1x", "K1u_wide") for d, H in WIDE]

# per-trajectory constants C of _bound, (float32 state, float64 state).  Largest measured ratio |error| / bound(C = 1) over
# FWD_CASES and both schedules, and the margin:
#   state path   1.39 (K1x d=1 H=128)  / 0.20 (K1 d=1, 24 000 trajectories)  -> C = 4 / 0.6   (2.9x / 3x)
#   G            0.075                 / 0.0082  \
#   S            0.25  (K1 d=10)       / 0.11     > C = 2 / 0.3     (3.6x / 2.8x, from logw and S)
#   logw         0.56  (K1w d=3)       / 0.071   /
#   l2 (d = 1)   4.6   (K1u)           / 0.0034  -> C = 12 / 0.01   (2.6x / 3x; error including grid-cell flips, which
#                                                   _l2_cell_flips now allows for: without them 0.026 / 0.004 at 24 000 trajectories)
# The wrong answers of _discriminates exceed C = 1 bounds with ratios of 98 or more on 90 % of the trajectories.
C_PATH = (4.0, 0.6)
C_G = (2.0, 0.3)
C_S = (2.0, 0.3)
C_L2 = (12.0, 0.01)


def _path_deviation(path, xr, n):
    """Per trajectory, the largest |kernel state - reference state| over the passes 0..n it executed, and half an ulp of the
    largest |reference state| there (the path is stored in float32 whatever the state's precision).  Slots past a
    trajectory's last pass are never written: masked, not read."""
    live = torch.as_tensor(np.arange(xr.shape[1])[None, :] <= n[:, None], device=xr.device)[..., None]
    dev = _np(torch.where(live, (path[:, :xr.shape[1]].double() - xr).abs(), 0.0).amax(dim=(1, 2)))
    store = EPS32 * _np(torch.where(live, xr.abs(), 0.0).amax(dim=(1, 2)))
    return dev, store, live


def _forward_case(family, d, H, f64, stoch_int, hit_rule, K=128, lim=2000, seed=None, extra=None, ref_out=None, env=None,
                  ratios=None, tols=None):
    """One forced launch against the float64 reference on the same increments, teacher-forced on the kernel's hit passes,
    in the environment ``env`` (as _env_c).  Returns (kernel output, reference output, policy parameters) after asserting
    everything that does not need the other mode.  ``ratios`` (a dict), if given, receives the largest |error| / bound(C = 1)
    of each compared output; ``tols`` may replace any of the constants C_PATH, C_G, C_S, C_L2 (keys "path", "G", "S",
    "l2")."""
    L, R = _lib()
    s = _spec(env)
    c = {"path": C_PATH, "G": C_G, "S": C_S, "l2": C_L2, **(tols or {})}
    seed = seed if seed is not None else 1000 * d + H
    model, params, flat = _policy(d, H, 1.0 if d == 1 else 2.5, seed)
    _, env_c = _env_c(d, hit_rule, env)
    mlp_c = L.make_mlp(d, H)
    noise = R.noise_fill(seed, K, d, lim, s["dt"])
    pol = grid = None
    if d == 1:
        grid = (-2.0, 2.0, 0.05)
        pol = 1.5 * np.cos(np.linspace(-2.0, 2.0, 81))
    kw = dict(FAMILIES[family])
    kw.update(extra or {})
    out = R.rollout_forward(env_c, mlp_c, flat, K, noise=noise, n_steps_lim=lim, stoch_int=stoch_int, state_f64=f64,
                            store_path=True, ckpt_every=1, want_logw=True, policy_opt=pol, grid=grid, **kw)
    T = out.T.cpu().numpy().astype(np.int64)
    if ref_out is None:
        ref_out = _reference(d, params, noise, env, hit_rule=ref.HIT_X0_IN_LB_RB if hit_rule else ref.HIT_ALL_GE_LB,
                             hit_index=T, f32_policy_input=f64, policy_opt=None if pol is None else pol[:, None],
                             grid=grid, keep_path=True, device="cuda")
    assert np.array_equal(ref_out["T"].cpu().numpy(), T)
    prec = 1 if f64 else 0
    n = np.where(T >= 0, T, lim - 1)                                           # last pass each trajectory executed
    # state path: the largest deviation along each path is itself bounded
    xr = ref_out["path"]
    dev, store, live = _path_deviation(out.path, xr, n)
    if ratios is not None:
        ratios["path"] = float(((dev - store) / _bound(n, 1.0, 1.0)).max())
    assert np.all(dev <= store + _bound(n, 1.0, c["path"][prec])), (family, d, H, float(((dev - store) / _bound(n, 1.0, 1.0)).max()))
    # own decisions: the kernel's hit pass is the reference's unless the reference's state lies within the path deviation
    # of the boundary at the first pass where they differ
    T_own = ref_out["T_own"].cpu().numpy()
    differ = T_own != T
    margin_first = _np(ref_out["margin_first"])
    assert np.array_equal(np.isnan(margin_first), ~differ)
    assert np.all(np.abs(margin_first[differ]) <= dev[differ] + 2 * EPS32 * 2.0), (family, d, H)
    assert differ.mean() <= 0.05
    # per-trajectory outputs
    G = _np(out.G)
    S_want = _np(ref_out["S_exact" if stoch_int == "exact" else "S_ref"])
    logw = _np(out.logw)
    if ratios is not None:
        for key, got, want, scale in (("G", G, _np(ref_out["G"]), G), ("S", _np(out.S), S_want, S_want),
                                      ("logw", logw, _np(ref_out["logw"]), logw)):
            ratios[key] = float((np.abs(got - want) / _bound(n, scale, 1.0)).max())
    assert np.all(np.abs(G - _np(ref_out["G"])) <= _bound(n, G, c["G"][prec]))
    assert np.all(np.abs(_np(out.S) - S_want) <= _bound(n, S_want, c["S"][prec]))
    assert np.all(np.abs(logw - _np(ref_out["logw"])) <= _bound(n, logw, c["S"][prec]))
    if pol is not None:
        l2_want = _np(ref_out["l2"])
        flips = _l2_cell_flips(params, xr[..., 0], out.path[:, :xr.shape[1], 0].double(), live[..., 0], pol, grid, f64, s["dt"])
        if ratios is not None:
            ratios["l2"] = float(((np.abs(_np(out.l2) - l2_want) - flips) / _bound(n, l2_want, 1.0)).max())
        assert np.all(np.abs(_np(out.l2) - l2_want) <= _bound(n, l2_want, c["l2"][prec]) + flips), (family, d, H)
    # statistics record of this dispatch site = fsum reduction of the launch's own outputs
    _assert_stats(out.stats, out.G, out.S, out.T, out.l2, out.logw, lim)
    return out, ref_out, params


def _l2_cell_flips(params, x, x_kernel, live, pol, grid, f64, dt=DT):
    """Per trajectory, the most the l2 error can move because the kernel's state and the reference's lie on either side
    of a grid-cell edge: over the passes (after the first, where both hold x0 exactly) whose reference state is within the
    two states' distance (plus the float32 storage rounding of the kernel's path) of an edge, the sum of
    max |(u - pol[c'])^2 - (u - pol[c])^2| dt, c' = c -+ 1.  (Like a hit decision, the lookup is discontinuous in x;
    everywhere else l2 moves by rounding only.)"""
    lo, hi, h = grid
    pol_t = torch.as_tensor(pol, dtype=torch.float64, device=x.device)
    y = (x.clamp(lo, hi) - lo) / h
    slack = torch.where(live, (x_kernel - x).abs(), 0.0) + EPS32 * x.abs()
    near = live & ((y - torch.round(y)).abs() * h <= slack)
    near[:, 0] = False
    out = torch.zeros(x.shape[0], dtype=torch.float64, device=x.device)
    idx = near.nonzero()
    if idx.numel():
        xs = x[idx[:, 0], idx[:, 1]]
        p64 = {k: v.to(device=x.device, dtype=torch.float64) for k, v in params.items()}
        u = ref.policy_torch(p64, (xs.float().double() if f64 else xs)[:, None])[:, 0]
        c = torch.floor((xs.clamp(lo, hi) - lo) / h).long().clamp(0, pol_t.numel() - 1)
        base = (u - pol_t[c]) ** 2
        alt = torch.maximum(((u - pol_t[(c - 1).clamp(min=0)]) ** 2 - base).abs(),
                            ((u - pol_t[(c + 1).clamp(max=pol_t.numel() - 1)]) ** 2 - base).abs())
        out.index_add_(0, idx[:, 0], alt * dt)
    return _np(out)


def _discriminates(family, d, H, f64, out_ref_mode, r_ref_mode, out_exact, r, params, dt=DT):
    """The nearest wrong answers fail the same tolerances on a clear majority of the finished trajectories.  ``r`` /
    ``r_ref_mode``: the float64 replays teacher-forced on the exact-mode / reference-mode launch's hit passes; ``dt`` their
    time step."""
    prec = 1 if f64 else 0
    T = out_exact.T.cpu().numpy().astype(np.int64)
    fin = T >= 0
    assert fin.sum() >= 64
    n = T[fin]
    # logw from the reference-mode integral (includes the detecting pass's u . dB)
    wrong_logw = _np(r["G"] - r["S_ref"])[fin]
    logw = _np(out_exact.logw)[fin]
    assert (np.abs(logw - wrong_logw) > _bound(n, logw, C_S[prec])).mean() > 0.8, (family, d, H)
    # the reference-mode integral where the exact one was asked
    S = _np(out_exact.S)[fin]
    assert (np.abs(S - _np(r["S_ref"])[fin]) > _bound(n, S, C_S[prec])).mean() > 0.8, (family, d, H)
    # ... and the exact one where the reference mode was asked
    T_r = out_ref_mode.T.cpu().numpy().astype(np.int64)
    fin_r = T_r >= 0
    S = _np(out_ref_mode.S)[fin_r]
    assert (np.abs(S - _np(r_ref_mode["S_exact"])[fin_r]) > _bound(T_r[fin_r], S, C_S[prec])).mean() > 0.8, (family, d, H)
    # the return including the detecting pass's running cost -(1 + |u|^2 / 2) dt
    x_hit = r["path"][torch.as_tensor(np.flatnonzero(fin), device="cuda"), torch.as_tensor(n, device="cuda")]
    p64 = {k: v.to(device="cuda", dtype=torch.float64) for k, v in params.items()}
    xin = x_hit.float().double() if f64 else x_hit
    u = ref.policy_torch(p64, xin)
    wrong_G = _np(r["G"])[fin] + _np(-(1.0 + 0.5 * (u * u).sum(dim=1)) * dt)
    G = _np(out_exact.G)[fin]
    assert (np.abs(G - wrong_G) > _bound(n, G, C_G[prec])).mean() > 0.95, (family, d, H)


@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("family,d,H", FWD_CASES)
def test_forward_kernel_matches_float64_reference(family, d, H, f64):
    """Every compiled forward instance, float32 and float64 state, both stochastic-integral modes, logw and (d = 1) the l2
    error: state paths, hit passes, G, S, logw, l2 and the statistics record against the float64 reference.  The float32 d = 1
    exact-mode case is the headline's argument set (lb <= x <= rb hit rule, exact integral, log-weights)."""
    L, _ = _lib()
    rule_exact = L.HIT_X0_IN_LB_RB if d == 1 else L.HIT_ALL_GE_LB
    rule_ref = L.HIT_X0_IN_LB_RB if (d == 1 and f64) else L.HIT_ALL_GE_LB
    out_x, r_x, params = _forward_case(family, d, H, f64, "exact", rule_exact)
    same_rule = rule_ref == rule_exact
    out_r, r_r, _ = _forward_case(family, d, H, f64, "reference", rule_ref, ref_out=r_x if same_rule else None)
    if same_rule:
        assert torch.equal(out_r.G, out_x.G) and torch.equal(out_r.T, out_x.T) and torch.equal(out_r.logw, out_x.logw)
    _discriminates(family, d, H, f64, out_r, r_r, out_x, r_x, params)


def _schedule_counters(K):
    """Workspace counters of the last forward launch (rollout_fwd.cuh, FwdArgs::q_ctrl): [1] continuation records queued,
    [3] records taken by the warp kernel's RESUME launch (one more per warp: its last, empty claim)."""
    _, R = _lib()
    ws = R._workspace(torch.device("cuda", torch.cuda.current_device()), K)
    return ws[:48].view(torch.int64).cpu().numpy()


@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("schedule", ["slices", "handoff"])
def test_forced_schedules_match_float64_reference(schedule, f64):
    """The headline's arguments (d = 1, H = 32, lb <= x <= rb, exact integral, logw; float32 state, and the float64 state of
    the NumPy path) through the two tail strategies of the thread-per-trajectory kernel: time slices of 8 passes (FIFO of
    continuation records) and run-to-completion with the last 4 000 live trajectories handed to the warp kernel, whose
    RESUME mode then writes their G, S, logw and l2.  Both need the persistent grid (more than 128 x SMs trajectories;
    smaller launches run every trajectory to completion); the workspace counters show that the schedule engaged.  Against
    the float64 reference, with the statistics record of the launch and the discrimination asserts."""
    L, _ = _lib()
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    K, lim = 128 * n_sm + 5000, 800                                # ~2.5 % of the trajectories run into the budget
    tuning = {"fwd_quantum": 8} if schedule == "slices" else {"fwd_quantum": 0, "fwd_handoff": 4000}
    runs = {}
    for mode in ("exact", "reference"):
        out, r, params = _forward_case("K1", 1, 32, f64, mode, L.HIT_X0_IN_LB_RB, K=K, lim=lim, extra={"tuning": tuning},
                                       ref_out=runs["exact"][1] if mode == "reference" else None)
        q = _schedule_counters(K)
        T = out.T.cpu().numpy()
        assert (T < 0).sum() > 0                                       # the unfinished branch is taken too
        if schedule == "slices":
            assert q[1] > K and q[3] == 0                              # every trajectory longer than 8 passes was requeued
        else:
            assert 0 < q[1] <= 4000 and q[3] >= q[1]                   # the tail went to the RESUME launch, all of it
        runs[mode] = (out, r)
    assert torch.equal(runs["exact"][0].T, runs["reference"][0].T)
    _discriminates("K1 " + schedule, 1, 32, f64, runs["reference"][0], runs["reference"][1], runs["exact"][0], runs["exact"][1],
                   params)


# ------------------------------------------------------------------------------ statistics through the other dispatch sites
def test_stats_of_fused_loss_and_grad_and_device_loop():
    """rollout_loss_and_grad (K1 + reduction + K2 with one copy back) and rlsde_reinforce_step (the device-resident loop):
    the statistics record equals the fsum reduction of the per-trajectory outputs the call exposes."""
    L, R = _lib()
    lib = L.load()
    _, params, flat = _policy(1, 32, 1.0, 3)
    env, env_c = _env_c(1, L.HIT_ALL_GE_LB)
    mlp_c = L.make_mlp(1, 32)
    K, lim = 3000, 500
    noise = R.noise_fill(8, K, 1, lim, DT)
    st, grad, G, T = R.rollout_loss_and_grad(env_c, mlp_c, flat, K, noise=noise, n_steps_lim=lim)
    assert (T >= 0).sum() > K // 2
    _assert_stats(st, G, np.zeros(K), T, None, None, lim, fields=(0, 1, 2, 3, 4, 5, 7, 8, 9, 11, 12, 13, 14, 15))
    # device-resident step: forward (warp kernel), statistics, reverse pass, Adam
    K = 500
    noise = R.noise_fill(9, K, 1, lim, DT)
    P = int(lib.rlsde_param_count(mlp_c))
    theta = torch.as_tensor(flat, device="cuda").clone()
    m, v = torch.zeros_like(theta), torch.zeros_like(theta)
    G = torch.empty(K, dtype=torch.float32, device="cuda")
    S, T = torch.empty_like(G), torch.empty(K, dtype=torch.int32, device="cuda")
    path = torch.empty((K, lim, 1), dtype=torch.float32, device="cuda")
    stats = torch.zeros(16, dtype=torch.float64, device="cuda")
    g = torch.empty(P, dtype=torch.float32, device="cuda")
    cfg = L.RlsdeRolloutCfg()
    cfg.K = cfg.K_global = K
    cfg.n_steps_lim, cfg.noise_steps = lim, lim
    cfg.flags = L.F_STORE_PATH | L.F_NOISE_INJECTED
    cfg.ckpt_every, cfg.ckpt_stride = 1, lim
    ws = R._workspace(theta.device, K, mlp_c)
    rc = lib.rlsde_reinforce_step(env_c, mlp_c, theta.data_ptr(), m.data_ptr(), v.data_ptr(), cfg, noise.data_ptr(), 1e-2, 0.9,
                                  0.999, 1e-8, 1, G.data_ptr(), S.data_ptr(), T.data_ptr(), path.data_ptr(), stats.data_ptr(),
                                  g.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
    L.check(rc, "rlsde_reinforce_step")
    _assert_stats(stats.cpu().numpy(), G, S, T, None, None, lim)
    # and the same trajectories as the float64 reference
    r = ref.rollout_reference(1, 1.0, 1.0, DT, params, noise, hit_index=T.cpu().numpy(), device="cuda")
    n = np.where(T.cpu().numpy() >= 0, T.cpu().numpy(), lim - 1)
    assert np.all(np.abs(_np(G) - _np(r["G"])) <= _bound(n, _np(G), C_G[0]))


# ------------------------------------------------------------------------------ the importance-sampling estimate
def test_is_estimate_matches_float64_reference_at_scale():
    """The headline's estimate (d = 1, H = 32, float32 state, lb <= x <= rb, exact integral) at K = 1e5 against the float64
    reference's mean(exp(logw)) on the same increments; summarize() against NumPy over the per-trajectory outputs; and the
    estimate that uses the reference-mode integral (an extra exp(-u dB) per weight) falls outside the tolerance."""
    L, R = _lib()
    _, params, flat = _policy(1, 32, 0.5, 17)
    env, env_c = _env_c(1, L.HIT_X0_IN_LB_RB)
    K, lim = 100_000, 1000
    out = R.rollout_forward(env_c, L.make_mlp(1, 32), flat, K, seed=2024, n_steps_lim=lim, stoch_int="exact", want_logw=True)
    s = R.summarize(out.stats)
    T = out.T.cpu().numpy()
    fin = T >= 0
    assert (~fin).sum() < K // 4
    G, S, logw = _np(out.G), _np(out.S), _np(out.logw)
    w = np.exp(logw[fin])
    np.testing.assert_allclose(s["is_mean"], w.mean(), rtol=1e-12)
    np.testing.assert_allclose(s["is_var"], w.var(), rtol=1e-8)
    np.testing.assert_allclose(s["is_rel_error"], w.std() / w.mean(), rtol=1e-8)
    np.testing.assert_allclose(s["var_return"], G[fin].var(), rtol=1e-8)
    assert s["mean_hit_index"] == T[fin].mean() and s["max_hit_index"] == T.max()
    np.testing.assert_allclose(s["mean_stoch_int"], S[fin].mean(), rtol=1e-10)
    _assert_stats(out.stats, out.G, out.S, out.T, None, out.logw, lim)
    noise = R.noise_fill(2024, K, 1, lim, DT)
    r = ref.rollout_reference(1, 1.0, 1.0, DT, params, noise, hit_rule=ref.HIT_X0_IN_LB_RB, hit_index=T, device="cuda")
    is64 = float(torch.exp(r["logw"][torch.as_tensor(fin, device="cuda")]).mean())
    wrong = float(torch.exp((r["G"] - r["S_ref"])[torch.as_tensor(fin, device="cuda")]).mean())
    tol = 1e-6 * is64                       # measured 1.5e-7 relative (6.8x margin); the S_ref-based estimate is 5.9e-4 off
    assert abs(s["is_mean"] - is64) <= tol, (s["is_mean"], is64)
    assert abs(wrong - is64) > 10 * tol, (wrong, is64)
    # own decisions of the reference: at most a handful of trajectories hit on another pass
    assert (r["T_own"].cpu().numpy() != T).mean() < 1e-3


def test_test_policy_vectorized_against_numpy():
    """test_policy_vectorized's mean / population variance / mean hit index / mean l2 against NumPy over the per-trajectory
    outputs of the same launch (float64 state)."""
    from rl_sde_is_b200.approximate_methods import test_policy_vectorized
    L, R = _lib()
    model, params, flat = _policy(1, 32, 0.8, 5)
    env, env_c = _env_c(1, L.HIT_X0_IN_LB_RB)
    env.discretize_state_space(0.05)
    pol = 1.5 * np.cos(env.state_space_h).reshape(-1, 1)
    K, lim = 20000, 4000
    noise = R.noise_fill(31, K, 1, lim, DT)
    res = test_policy_vectorized(env, model, batch_size=K, k_max=lim, policy_opt=pol, noise=noise)
    out = R.rollout_forward(env_c, L.make_mlp(1, 32), flat, K, noise=noise, n_steps_lim=lim, state_f64=True, policy_opt=pol,
                            grid=(-2.0, 2.0, 0.05), want_logw=False)
    G, T, l2 = _np(out.G), out.T.cpu().numpy(), _np(out.l2)
    assert (T >= 0).all()
    np.testing.assert_allclose(res[0], G.mean(), rtol=1e-12)
    np.testing.assert_allclose(res[1], G.var(), rtol=1e-8)
    assert res[2] == T.mean()
    np.testing.assert_allclose(res[3], l2.mean(), rtol=1e-12)


# ------------------------------------------------------------------------------ reverse passes, both integral modes
# family -> (forward arguments, cfg fields set before the reverse pass)
BWD_FAMILIES = {
    "K2m": (dict(kernel="thread"), dict(bwd_kernel=1)),          # rollout_bwd_mma.cuh
    "K2w": (dict(kernel="warp"), {}),                            # rollout_warp.cuh reverse pass
    "K2x": (dict(tuning={"wide_kernel": "ffma"}), dict(wide_kernel=2)),   # rollout_wide.cuh reverse pass
    "K2u": (dict(tuning={"wide_kernel": "umma"}), dict(wide_kernel=1)),   # rollout_umma_bwd.cuh
}
BWD_CASES = ([("K2m", d, 32, c) for d in (1, 2, 3, 4, 10) for c in (1, 4, 8, 16)]
             + [("K2w", d, 32, 1) for d in (1, 2, 3, 4, 10)] + [("K2x", d, H, 1) for d in (1, 2) for H in (64, 128, 256)]
             + [("K2u", d, H, 1) for d in (1, 2) for H in (128, 256)])
# max |g_kernel - g_f64| / max |g_f64| per family, with the largest value measured over its cases (both modes) and the margin;
# the other tests hold kernels to 5e-4 of max |g| against the reference's float32 gradient.  The exact-mode kernel gradient
# differs from the reference-mode float64 gradient by 4.1e-3 (K2x / K2u, d = 1, H = 256) or more, 8.0e-4 in the split case.
GRAD_TOL = {"K2m": 1.5e-5,    # 4.4e-6 (d = 10: float16 x 3 split of the padded d-sized products), 3.4x
            "K2w": 2e-6,      # 4.1e-7, 4.9x
            "K2x": 2e-6,      # 5.0e-7, 4x
            "K2u": 3e-6,      # 7.1e-7, 4.2x
            "split": 5e-7}    # 1.9e-7 (d = 2), 2.6x


def _grad_case(family, d, H, ckpt, K=192, lim=400, extra_cfg=None, env=None, wrong_envs=None):
    """Kernel gradients in both integral modes against float64 autograd along the kernel's hit passes, in the environment
    ``env`` (as _env_c).  Returns (relative error per mode, relative distance of the exact-mode gradient from the
    reference-mode float64 one, {name: relative distance of the kernel's gradient from float64 autograd in the
    environment ``wrong_envs[name]``, the smaller of the two modes})."""
    L, R = _lib()
    s = _spec(env)
    seed = 77 + 100 * d + H
    _, params, flat = _policy(d, H, 2.0 if d == 1 else 3.0, seed)
    _, env_c = _env_c(d, L.HIT_ALL_GE_LB, env)
    mlp_c = L.make_mlp(d, H)
    noise = R.noise_fill(seed, K, d, lim, s["dt"])
    fkw, cfg_set = BWD_FAMILIES[family]
    fwd = R.rollout_forward(env_c, mlp_c, flat, K, noise=noise, n_steps_lim=lim, stoch_int="exact", store_path=True,
                            ckpt_every=ckpt, want_logw=False, **fkw)
    T = fwd.T.cpu().numpy()
    assert (T >= 0).mean() > 0.9
    for k, v in {**cfg_set, **(extra_cfg or {})}.items():
        setattr(fwd.cfg, k, v)
    grads = {}
    for mode in ("exact", "reference"):
        fwd.cfg.flags = (fwd.cfg.flags | L.F_STOCH_INT_EXACT) if mode == "exact" else (fwd.cfg.flags & ~L.F_STOCH_INT_EXACT)
        grads[mode] = R.rollout_backward(env_c, mlp_c, flat, fwd, 1.0 / K, noise=noise).cpu().numpy().astype(np.float64)
    modes = ("exact", "reference")

    def autograd(e):
        r = _reference(d, params, noise, e, hit_index=T, grad_modes=modes, device="cuda")
        return {m: np.concatenate([r["grads"][m][k].reshape(-1) for k in ref.PARAM_KEYS]) for m in modes}

    def dist(a, b):
        return np.abs(a - b).max() / np.abs(b).max()

    want = autograd(env)
    errs = {m: dist(grads[m], want[m]) for m in modes}
    wrong = dist(grads["exact"], want["reference"])
    wrong_env = {}
    for name, e in (wrong_envs or {}).items():
        w = autograd(e)
        wrong_env[name] = min(dist(grads[m], w[m]) for m in modes)
    return errs, wrong, wrong_env


@pytest.mark.parametrize("family,d,H,ckpt", BWD_CASES)
def test_reverse_pass_matches_float64_autograd(family, d, H, ckpt):
    """Every reverse family in both stochastic-integral modes against float64 autograd of mean(-G - sg(G) S) along the
    kernel's hit passes; the exact-mode gradient is told apart from the reference-mode float64 gradient (short paths with a
    drift towards the target, where the detecting pass's u . dB is a visible share of the gradient)."""
    errs, wrong, _ = _grad_case(family, d, H, ckpt)
    tol = GRAD_TOL[family]
    assert errs["exact"] <= tol and errs["reference"] <= tol, (family, d, H, ckpt, errs)
    assert wrong > 10 * tol, (family, d, H, ckpt, wrong)


@pytest.mark.parametrize("bulk,d", [("K2m", 1), ("K2m", 2)])
def test_reverse_pass_split_between_families_matches_float64_autograd(bulk, d):
    """Large batches: the 1 000 longest trajectories go to the warp reverse kernel on a second stream, the rest to K2m,
    whose reduction waits for them and adds onto their gradient; both integral modes, against float64 autograd."""
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    errs, wrong, _ = _grad_case(bulk, d, 32, 1, K=128 * n_sm + 200, lim=300, extra_cfg={"bwd_warp_share": 1000})
    tol = GRAD_TOL["split"]
    assert errs["exact"] <= tol and errs["reference"] <= tol, errs
    assert wrong > 10 * tol, wrong
