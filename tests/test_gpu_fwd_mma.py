"""The forward rollout's policy on the tensor cores (csrc/mlp_mma.cuh: layer 2 as mma.sync with float16 hi / lo operand
splits) against the FFMA2 arithmetic it replaces at d = 1, hidden width 32, and against the float64 reference rollout.

The two arithmetics round differently, so a trajectory whose state passes within rounding of the target boundary may
stop one pass earlier or later; everything else agrees to float32 accumulation error.  The tensor-core arithmetic itself
must not depend on how trajectories are scheduled: batch size, shard offset, time slices and the hand-off of the tail to
the warp-per-trajectory kernel all leave its results bit-identical.  The CPU tests restate the fragment layout of the
host packer and show that the lo halves of the split are needed."""
import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import reference_semantics as ref

DT = 0.005


@pytest.fixture(autouse=True)
def _no_schedule_overrides(monkeypatch):
    for name in ("FWD_QUANTUM", "FWD_HANDOFF", "BWD_WARP_SHARE", "FWD_BLOCKS_PER_SM", "BWD_KERNEL", "WIDE_KERNEL", "FWD_POLICY"):
        monkeypatch.delenv("RLSDE_" + name, raising=False)


def _policy(bias, seed):
    from rl_sde_is_b200 import rollout as R
    from rl_sde_is_b200.models import DeterministicPolicy
    torch.manual_seed(seed)
    m = DeterministicPolicy(1, 1, [32, 32], nn.Tanh())
    m.policy[4].bias.data.fill_(bias)
    params = {k: v.detach().clone() for k, v in m.state_dict().items()}
    return params, R.flat_parameters(m).detach().numpy()


def _env_c(hit_rule):
    from rl_sde_is_b200 import rollout as R
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D
    return R.env_struct(DoubleWellStoppingTime1D(beta=1.0, alpha=1.0, dt=DT), hit_rule)


def _np(t):
    return t.double().cpu().numpy()


# ------------------------------------------------------------------------------ mma against ffma
@pytest.mark.gpu
@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("tanh", ["precise", "fast"])
def test_mma_policy_matches_ffma_policy(f64, tanh):
    """The headline workload (K = 1e6, budget 1 000 passes, exact integral) through the thread-per-trajectory kernel with
    each policy arithmetic: hit passes agree for >= 99.5 % of the trajectories, is_mean and the mean return to 1e-6
    relative; against the float64 reference on the first 1e5 trajectories' own increments and hit passes, the tensor-core
    arithmetic's largest G / S deviation is within 2x that of the FFMA2 arithmetic."""
    from rl_sde_is_b200 import _lib as L, rollout as R
    params, flat = _policy(0.5, 17)
    env_c = _env_c(L.HIT_X0_IN_LB_RB)
    K, lim, seed = 1_000_000, 1000, 4242
    outs = {}
    for pol in ("ffma", "mma"):
        outs[pol] = R.rollout_forward(env_c, L.make_mlp(1, 32), flat, K, seed=seed, n_steps_lim=lim, stoch_int="exact",
                                      state_f64=f64, tanh=tanh, want_logw=True, kernel="thread", tuning={"fwd_policy": pol})
    Tf, Tm = outs["ffma"].T.cpu().numpy(), outs["mma"].T.cpu().numpy()
    same = float((Tf == Tm).mean())
    assert same >= 0.995, same
    sf, sm = R.summarize(outs["ffma"].stats), R.summarize(outs["mma"].stats)
    for key in ("is_mean", "mean_return"):
        assert abs(sm[key] - sf[key]) <= 1e-6 * abs(sf[key]), (key, sm[key], sf[key])
    # float64 reference along each arithmetic's own hit passes
    k_ref = 100_000
    noise = R.noise_fill(seed, k_ref, 1, lim, DT)
    dev = {}
    for pol, o in outs.items():
        T = o.T.cpu().numpy()[:k_ref]
        r = ref.rollout_reference(1, 1.0, 1.0, DT, params, noise, hit_rule=ref.HIT_X0_IN_LB_RB, hit_index=T,
                                  f32_policy_input=f64, device="cuda")
        n = np.where(T >= 0, T, lim) + 1.0
        S_ref = _np(r["S_exact"])
        dG = np.abs(_np(o.G)[:k_ref] - _np(r["G"])) / n
        dS = np.abs(_np(o.S)[:k_ref] - S_ref) / n
        dev[pol] = (dG.max(), dS.max())
    for i, name in enumerate(("G", "S")):
        assert dev["mma"][i] <= 2.0 * dev["ffma"][i], (name, dev)


# ------------------------------------------------------------------------------ bitwise invariance of the mma arithmetic
def _run(L, R, env_c, flat, K, *, f64, seed=99, traj_offset=0, K_global=None, quantum=None, handoff=None, store_path=False):
    tuning = {"fwd_policy": "mma", "fwd_quantum": quantum, "fwd_handoff": handoff}
    pol = np.linspace(-1, 1, 81)
    return R.rollout_forward(env_c, L.make_mlp(1, 32), flat, K, seed=seed, n_steps_lim=20000, state_f64=f64, want_logw=True,
                             traj_offset=traj_offset, K_global=K_global, policy_opt=pol, grid=(-2.0, 2.0, 0.05),
                             store_path=store_path, ckpt_every=2, kernel="thread", tuning=tuning)


@pytest.mark.gpu
@pytest.mark.parametrize("f64", [False, True])
def test_mma_policy_is_schedule_invariant(f64):
    """Batch size, shard offset, slice length (4 / 8 / 32 passes, run to completion) and hand-off threshold (0 / 4 000 /
    40 000 live trajectories) leave every output of the tensor-core arithmetic bit-identical: float32 state with the path
    checkpoints, float64 state with the l2 error."""
    from rl_sde_is_b200 import _lib as L, rollout as R
    _, flat = _policy(0.6, 21)
    env_c = _env_c(L.HIT_X0_IN_LB_RB if f64 else L.HIT_ALL_GE_LB)
    K = 30000
    base = _run(L, R, env_c, flat, K, f64=f64, quantum=-1, handoff=-1, store_path=not f64)
    T = base.T.cpu().numpy()
    assert (T >= 0).all() and T.max() > 5 * np.median(T)

    def same(o, lo=0, hi=K):
        assert torch.equal(o.G, base.G[lo:hi]) and torch.equal(o.S, base.S[lo:hi]) and torch.equal(o.T, base.T[lo:hi])
        assert torch.equal(o.logw, base.logw[lo:hi]) and torch.equal(o.l2, base.l2[lo:hi])
        if not f64:
            n_ck = T[lo:hi] // 2 + 1
            mask = torch.as_tensor(np.arange(o.path.shape[1])[None, :] < n_ck[:, None], device=o.path.device)
            assert torch.equal(o.path[..., 0][mask], base.path[lo:hi][..., 0][mask])

    for q in (4, 8, 32):
        same(_run(L, R, env_c, flat, K, f64=f64, quantum=q, store_path=not f64))
    for h in (4000, 40000):
        same(_run(L, R, env_c, flat, K, f64=f64, quantum=-1, handoff=h, store_path=not f64))
    # a shard of the same global batch, and a smaller batch
    same(_run(L, R, env_c, flat, 20000, f64=f64, traj_offset=10000, K_global=K, store_path=not f64), 10000, K)
    same(_run(L, R, env_c, flat, 25000, f64=f64, store_path=not f64), 0, 25000)


@pytest.mark.gpu
def test_mma_policy_is_automatic_at_d1_and_rejected_elsewhere():
    """Automatic selection takes the tensor-core arithmetic at d = 1, hidden width 32; forcing it on another shape is an
    error, not a fall-back."""
    from rl_sde_is_b200 import _lib as L, rollout as R
    from rl_sde_is_b200.environments import DoubleWellStoppingTimeND
    from rl_sde_is_b200.models import DeterministicPolicy
    _, flat = _policy(0.5, 3)
    env_c = _env_c(L.HIT_X0_IN_LB_RB)
    K = 50000
    o = {p: R.rollout_forward(env_c, L.make_mlp(1, 32), flat, K, seed=5, n_steps_lim=1000, kernel="thread",
                              tuning={"fwd_policy": p}) for p in ("auto", "mma", "ffma")}
    assert torch.equal(o["auto"].G, o["mma"].G) and torch.equal(o["auto"].T, o["mma"].T)
    assert not torch.equal(o["mma"].G, o["ffma"].G)
    torch.manual_seed(0)
    m2 = DeterministicPolicy(2, 2, [32, 32], nn.Tanh())
    env2 = R.env_struct(DoubleWellStoppingTimeND(2, beta=1.0, alpha=1.0, dt=DT), L.HIT_ALL_GE_LB)
    with pytest.raises(L.RlsdeError):
        R.rollout_forward(env2, L.make_mlp(2, 32), R.flat_parameters(m2).detach().numpy(), K, seed=5, n_steps_lim=100,
                          kernel="thread", tuning={"fwd_policy": "mma"})


# ------------------------------------------------------------------------------ CPU restatement of the packer
def _w2_fragment_map():
    """(p = 0 table of pack_w2_frags) -> for every (hl-independent) register slot [kk][jp][lane][r][half] the element
    (k = input unit, n = output unit) of B[k][n] = W2[n][k] it holds."""
    idx = np.empty((2, 2, 32, 4, 2, 2), dtype=np.int64)
    for kk in range(2):
        for jp in range(2):
            for lane in range(32):
                g, q = lane >> 2, lane & 3
                for jj in range(2):
                    n = 8 * (2 * jp + jj) + g
                    for b in range(2):
                        k = 16 * kk + 2 * q + 8 * b
                        for e in range(2):
                            idx[kk, jp, lane, 2 * jj + b, e] = [k + e, n]
    return idx


def _split(w):
    hi = w.astype(np.float16)
    lo = (w - hi.astype(np.float32)).astype(np.float16)
    return hi, lo


def test_w2_fragments_cover_each_weight_once():
    """The fragment table names every W2 element exactly once, and its hi + lo halves put it back to within the split's
    precision: 2^-22 relative (the lo half carries the 11 bits below the hi half's), 2^-25 absolute where the lo half is
    a float16 subnormal."""
    idx = _w2_fragment_map().reshape(-1, 2)
    flat = idx[:, 0] * 32 + idx[:, 1]
    assert np.array_equal(np.sort(flat), np.arange(32 * 32))
    rng = np.random.default_rng(0)
    W2 = (rng.standard_normal((32, 32)) * 0.5).astype(np.float32)        # [out][in]
    hi, lo = _split(W2[idx[:, 1], idx[:, 0]])
    back = hi.astype(np.float64) + lo.astype(np.float64)
    w = W2[idx[:, 1], idx[:, 0]].astype(np.float64)
    assert np.all(np.abs(back - w) <= 2.0 ** -22 * np.abs(w) + 2.0 ** -25)
    assert np.any(hi.astype(np.float64) != w)


def _policy_split(params, x, lo_terms):
    """Action of the folded precise-tanh policy, float64 except for the float16 split of layer 2's operands."""
    W1, b1 = params["policy.0.weight"].double().numpy(), params["policy.0.bias"].double().numpy()
    W2, b2 = params["policy.2.weight"].double().numpy(), params["policy.2.bias"].double().numpy()
    W3, b3 = params["policy.4.weight"].double().numpy(), params["policy.4.bias"].double().numpy()
    s = 2.0 * np.log2(np.e)
    r1 = 1.0 / (np.exp2(s * (x[:, None] * W1[:, 0] + b1)) + 1.0)                  # (1 - tanh) / 2
    W2f = (-2.0 * s * W2).astype(np.float32)                                        # folded weights
    b2f = s * (b2 + W2.sum(axis=1))
    ah, al = _split(r1.astype(np.float32))
    bh, bl = _split(W2f.T)
    f = lambda a: a.astype(np.float64)
    z2 = f(ah) @ f(bh) + b2f
    if lo_terms:
        z2 += f(al) @ f(bh) + f(ah) @ f(bl)
    r2 = 1.0 / (np.exp2(z2) + 1.0)
    return (b3 + W3.sum(axis=1))[0] + (r2 @ (-2.0 * W3[0]))


def test_dropping_the_lo_terms_is_visible():
    """With the three products the split's action error is ~1e-7 of the action scale, below float32 accumulation; with
    the hi product alone it is ~1e-5, outside what the GPU comparison with the FFMA2 arithmetic allows (1e-6 relative on
    is_mean)."""
    params, _ = _policy(0.5, 17)
    x = np.linspace(-2.0, 2.0, 4001)
    W1, b1 = params["policy.0.weight"].double().numpy(), params["policy.0.bias"].double().numpy()
    W2, b2 = params["policy.2.weight"].double().numpy(), params["policy.2.bias"].double().numpy()
    W3, b3 = params["policy.4.weight"].double().numpy(), params["policy.4.bias"].double().numpy()
    u64 = (np.tanh(np.tanh(x[:, None] * W1[:, 0] + b1) @ W2.T + b2) @ W3.T + b3)[:, 0]
    scale = np.abs(u64).max()
    err3 = np.abs(_policy_split(params, x, True) - u64).max() / scale
    err1 = np.abs(_policy_split(params, x, False) - u64).max() / scale
    assert err3 < 1e-6, err3
    assert err1 > 10 * 1e-6, err1
