"""Pin the float64 reference rollout (oracle/reference_semantics.rollout_reference) before it judges the kernels: on every
recorded rollout of the reference it finds the same hit passes, its returns lie within the reference's own float32
rounding, and so do its gradients; with a constant policy it equals the closed form.  CPU only."""
import math
import os
import sys

import numpy as np
import pytest
import torch

from oracle import reference_semantics as ref

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from readers import wide_case  # noqa: E402

EPS32 = 2.0 ** -24


def _env(npz, p):
    e = npz[p + "env"]
    return int(e[0]), float(e[1]), float(e[2]), float(e[3])


def _fp32_bound(T, value):
    """Per-trajectory scale of float32 accumulation error: one rounding of the result's size per pass executed."""
    return (np.asarray(T) + 1) * EPS32 * (1.0 + np.abs(value))


def _check_torch_case(g, p):
    torch.set_num_threads(1)
    d, alpha, beta, dt = _env(g, p)
    out = ref.rollout_reference(d, alpha, beta, dt, ref.params_from_npz(g, p), g[p + "noise"], keep_margin=True,
                                grad_modes=("reference",))
    T = out["T"].numpy()
    assert np.array_equal(T + 1, g[p + "time_steps"]) and np.array_equal(out["T_own"].numpy(), T)
    m = out["margin"].numpy()
    assert np.all(m[T, np.arange(T.size)] >= 0) and all(np.all(m[:t, i] < 0) for i, t in enumerate(T))
    assert torch.isnan(out["margin_first"]).all()                                  # a free run never disagrees with itself
    G = out["G"].numpy()
    # measured: |G64 - G32| <= 0.20 of the bound (1.8e-5 relative on case b's 2 053-pass paths)
    assert np.all(np.abs(G - g[p + "return_fht"]) <= _fp32_bound(T, G)), np.max(np.abs(G - g[p + "return_fht"]) / _fp32_bound(T, G))
    np.testing.assert_array_equal(out["logw"].numpy(), G - out["S_exact"].numpy())
    # the reference's float32 gradient is within 2.4e-5 of max |g| of the float64 one (tinit_h256_, 4 055 passes): 4x margin
    gs = max(np.abs(g[f"{p}grad.{k}"]).max() for k in ref.PARAM_KEYS)
    for k in ref.PARAM_KEYS:
        np.testing.assert_allclose(out["grads"]["reference"][k], g[f"{p}grad.{k}"], rtol=0, atol=1e-4 * gs, err_msg=k)
    return out


@pytest.mark.parametrize("fixture,prefix", [("rollout_torch_1d", "a_"), ("rollout_torch_1d", "b_"),
                                            ("rollout_torch_1d", "c_"), ("rollout_torch_2d", "a_")])
def test_float64_rollout_matches_torch_fixtures(golden, fixture, prefix):
    g = golden(fixture)
    out = _check_torch_case(g, prefix)
    d, alpha, beta, dt = _env(g, prefix)
    # the stochastic integral of the reference's float32 replay (u . dB on the detecting pass included)
    py = ref.rollout_loss_torch(d, alpha, beta, dt, ref.params_from_npz(g, prefix), g[prefix + "noise"], need_grad=False)
    T = out["T"].numpy()
    S = out["S_ref"].numpy()
    assert np.all(np.abs(S - py["stoch_int_fht"]) <= _fp32_bound(T, S))           # measured <= 2.1e-6 absolute


@pytest.mark.parametrize("prefix", ["th64_", "th128_", "th256_", "t2d_h128_", "tinit_h256_"])
def test_float64_rollout_matches_wide_torch_fixtures(golden, prefix):
    _check_torch_case(wide_case(golden("rollout_wide"), prefix), prefix)


def _check_numpy_case(g, p):
    torch.set_num_threads(1)
    e = g[p + "env"]
    d, alpha, beta, dt, h = int(e[0]), float(e[1]), float(e[2]), float(e[3]), float(e[4])
    params = ref.params_from_npz(g, p)
    out = ref.rollout_reference(d, alpha, beta, dt, params, g[p + "noise"], hit_rule=ref.HIT_X0_IN_LB_RB, f32_policy_input=True,
                                policy_opt=g[p + "policy_opt"], grid=(-2.0, 2.0, h))
    st = ref.rollout_stats_numpy(d, alpha, beta, dt, params, g[p + "noise"], policy_opt=g[p + "policy_opt"], h_state=h)
    assert np.array_equal(out["T"].numpy(), st["ep_lens"])
    # the NumPy path already accumulates in float64; only the first pass's float32 state and the float32 policy differ:
    # measured |dG| <= 2.9e-9, |dl2| <= 4.4e-9
    np.testing.assert_allclose(out["G"].numpy(), st["ep_rets"], rtol=0, atol=5e-8)
    np.testing.assert_allclose(out["l2"].numpy(), st["l2"], rtol=0, atol=5e-8)
    res = g[p + "result"]
    np.testing.assert_allclose([out["G"].numpy().mean(), out["T"].numpy().mean()], [res[0], res[2]], rtol=1e-7)


@pytest.mark.parametrize("prefix", ["a_", "b_"])
def test_float64_rollout_matches_numpy_fixtures(golden, prefix):
    _check_numpy_case(golden("rollout_numpy_1d"), prefix)


@pytest.mark.parametrize("prefix", ["nh64_", "nh128_", "nh256_"])
def test_float64_rollout_matches_wide_numpy_fixtures(golden, prefix):
    _check_numpy_case(wide_case(golden("rollout_wide"), prefix), prefix)


@pytest.mark.parametrize("d,c", [(1, 1.5), (2, 1.75)])         # c exact in float32
def test_float64_rollout_constant_policy_closed_form(d, c):
    """W3 = 0, b3 = c: u = c exactly, so S_exact = c . sum_{j<k*} dB_j and G = -k* (1 + |c|^2 / 2) dt; the hit passes come
    from a separate NumPy Euler-Maruyama loop with the same constant control."""
    torch.manual_seed(3)
    H, K, n, dt = 32, 40, 1500, 0.005
    params = {"policy.0.weight": torch.randn(H, d), "policy.0.bias": torch.randn(H), "policy.2.weight": torch.randn(H, H),
              "policy.2.bias": torch.randn(H), "policy.4.weight": torch.zeros(d, H), "policy.4.bias": torch.full((d,), c)}
    noise = (np.sqrt(dt) * np.random.default_rng(d).standard_normal((n, K, d))).astype(np.float32)
    out = ref.rollout_reference(d, 1.0, 1.0, dt, params, noise)
    T = out["T"].numpy()
    x, want_T = np.full((K, d), -1.0), np.full(K, -1)
    sigma = np.sqrt(2.0)
    for k in range(n):
        fresh = (want_T < 0) & (x >= 1.0).all(axis=1)
        want_T[fresh] = k
        x = x + (-(4.0 * x * (x * x - 1.0)) + sigma * c) * dt + sigma * noise[k].astype(np.float64)
    assert np.array_equal(T, want_T) and (T > 0).sum() > K // 2
    for i in range(K):
        n_i = T[i] if T[i] >= 0 else n                   # unfinished: sums over every pass, S_ref = S_exact
        s = math.fsum(c * float(v) for v in noise[:n_i, i, :].ravel())
        last = c * float(noise[T[i], i, :].astype(np.float64).sum()) if T[i] >= 0 else 0.0
        np.testing.assert_allclose(out["S_exact"][i].item(), s, rtol=1e-12, atol=1e-14)
        np.testing.assert_allclose(out["S_ref"][i].item(), s + last, rtol=1e-12, atol=1e-14)
        np.testing.assert_allclose(out["G"][i].item(), -n_i * (1.0 + 0.5 * d * c * c) * dt, rtol=1e-12)
    np.testing.assert_allclose(out["logw"].numpy(), out["G"].numpy() - out["S_exact"].numpy(), rtol=0, atol=0)


def test_float64_rollout_teacher_forcing_and_budget():
    """hit_index equal to the rollout's own hit passes changes nothing; an earlier forced pass stops the sums there; a
    trajectory forced to -1 (or a budget shorter than its hit pass) is unfinished: G and S over every pass, logw = G - S."""
    torch.manual_seed(5)
    H, K, n, dt = 32, 16, 1200, 0.005
    lin = [torch.nn.Linear(1, H), torch.nn.Linear(H, H), torch.nn.Linear(H, 1)]
    lin[2].bias.data.fill_(1.2)
    params = dict(zip(ref.PARAM_KEYS, [t.detach() for m in lin for t in (m.weight, m.bias)]))
    noise = (np.sqrt(dt) * np.random.default_rng(7).standard_normal((n, K, 1))).astype(np.float32)
    free = ref.rollout_reference(1, 1.0, 1.0, dt, params, noise, keep_path=True, keep_margin=True)
    T = free["T"].numpy()
    assert (T > 10).all()
    same = ref.rollout_reference(1, 1.0, 1.0, dt, params, noise, hit_index=T)
    for key in ("T", "T_own", "G", "S_exact", "S_ref", "logw"):
        assert torch.equal(free[key], same[key]), key
    early = T.copy()
    early[0], early[1] = T[0] - 5, -1
    forced = ref.rollout_reference(1, 1.0, 1.0, dt, params, noise, hit_index=early, keep_path=True, keep_margin=True)
    assert forced["T"][0] == T[0] - 5 and forced["T_own"][0] == -1 and forced["T"][1] == -1
    # the path is the same up to the forced pass; G / S there are the partial sums of the free run's per-pass terms
    x = free["path"][0, :T[0] - 5, 0]
    assert torch.equal(forced["path"][0, :T[0] - 5, 0], x)
    u = ref.policy_torch({k: v.double() for k, v in params.items()}, x[:, None])[:, 0]
    np.testing.assert_allclose(forced["G"][0].item(), float((-(1.0 + 0.5 * u * u) * dt).sum()), rtol=1e-12)
    np.testing.assert_allclose(forced["S_exact"][0].item(), float((u * torch.from_numpy(noise[:T[0] - 5, 0, 0]).double()).sum()),
                               rtol=1e-12)
    assert forced["S_ref"][1] == forced["S_exact"][1] and forced["logw"][1] == forced["G"][1] - forced["S_exact"][1]
    assert forced["margin"].shape[0] == n and not torch.isnan(forced["margin"][:, 1]).any()
    # first disagreement: trajectory 0 at the forced pass (still outside the target set), trajectory 1 at its own hit pass
    mf = forced["margin_first"]
    assert mf[0] == free["margin"][T[0] - 5, 0] and mf[0] < 0
    assert mf[1] == free["margin"][T[1], 1] and mf[1] >= 0 and torch.isnan(mf[2:]).all()
    short = ref.rollout_reference(1, 1.0, 1.0, dt, params, noise, n_steps_lim=int(T.min()), keep_margin=True)
    assert (short["T"] == -1).all() and torch.equal(short["S_ref"], short["S_exact"])
    assert short["margin"].shape[0] == int(T.min()) and short["margin_first"] is not None
    assert ref.rollout_reference(1, 1.0, 1.0, dt, params, noise)["margin"] is None
