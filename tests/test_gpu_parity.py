"""Parity of the CUDA path (through the C ABI) with the oracle and the reference fixtures.

Tolerances (BASELINE.json north_star): injected-noise trajectories within 1e-5 relative on work
functionals, hit indices exact; tables within 1e-6 (we hold 1e-13); in-kernel RNG statistically
indistinguishable (and, against the C restatement of the same Philox stream, per-trajectory close).
"""
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import c_oracle
from oracle import reference_semantics as ref

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from readers import tables_h001_column  # noqa: E402

pytestmark = pytest.mark.gpu


def _env(npz, p):
    e = npz[p + "env"]
    return int(e[0]), float(e[1]), float(e[2]), float(e[3])


def _make_env(d, alpha, beta, dt):
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D, DoubleWellStoppingTimeND
    return DoubleWellStoppingTime1D(beta=beta, alpha=alpha, dt=dt) if d == 1 else DoubleWellStoppingTimeND(d, beta=beta, alpha=alpha, dt=dt)


def _model_from(npz, prefix, d):
    from rl_sde_is_b200.models import DeterministicPolicy
    m = DeterministicPolicy(d, d, [32, 32], nn.Tanh())
    m.load_state_dict({k: torch.from_numpy(np.array(npz[f"{prefix}param.{k}"])) for k in ref.PARAM_KEYS})
    return m


# ------------------------------------------------------------------------------ torch path, injected noise
KERNELS = ["thread", "warp", "tensor"]      # trajectory per thread (CUDA cores) / per warp (latency) / per thread with the hidden layer on tcgen05


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("fixture,prefix", [("rollout_torch_1d", "a_"), ("rollout_torch_1d", "b_"),
                                            ("rollout_torch_1d", "c_"), ("rollout_torch_2d", "a_")])
def test_sample_loss_vectorized_matches_reference(golden, fixture, prefix, kernel):
    from rl_sde_is_b200.reinforce_deterministic_core import sample_loss_vectorized
    g = golden(fixture)
    d, alpha, beta, dt = _env(g, prefix)
    env, model = _make_env(d, alpha, beta, dt), _model_from(g, prefix, d)
    K = g[prefix + "noise"].shape[1]
    loss, ret, steps = sample_loss_vectorized(env, model, K, noise=g[prefix + "noise"], kernel=kernel)
    assert ret.dtype == np.float32 and steps.dtype == np.float64 and loss.dtype == torch.float32 and loss.dim() == 0
    assert np.array_equal(steps, g[prefix + "time_steps"])                               # hit passes: exact
    np.testing.assert_allclose(ret, g[prefix + "return_fht"], rtol=1e-5)
    np.testing.assert_allclose(float(loss), float(g[prefix + "loss"]), rtol=2e-5)
    loss.backward()
    # fp32 sums of ~1e4 cancelling G dB terms: the reference's own gradient is only within 1e-4..1e-3 (of the
    # largest entry) of an fp64 evaluation of the same loss, so entries are compared on the gradient's scale
    gscale = max(np.abs(g[f"{prefix}grad.{k}"]).max() for k, _ in model.named_parameters())
    for k, p in model.named_parameters():
        ref_g = g[f"{prefix}grad.{k}"]
        scale = max(np.abs(ref_g).max(), gscale)
        np.testing.assert_allclose(p.grad.numpy(), ref_g, rtol=2e-4, atol=5e-4 * scale, err_msg=k)  # the reference's own f32 gradient is within ~1e-4..1e-3 of an f64 evaluation here


def test_stochastic_integral_matches_oracle(golden):
    from rl_sde_is_b200 import _lib as L
    from rl_sde_is_b200 import rollout as R
    g = golden("rollout_torch_1d")
    for prefix in ("a_", "c_"):
        d, alpha, beta, dt = _env(g, prefix)
        params = ref.params_from_npz(g, prefix)
        py = ref.rollout_loss_torch(d, alpha, beta, dt, params, g[prefix + "noise"], need_grad=False)
        env = _make_env(d, alpha, beta, dt)
        noise = torch.from_numpy(g[prefix + "noise"]).cuda()
        for kernel in KERNELS:
            out = R.rollout_forward(R.env_struct(env, L.HIT_ALL_GE_LB), L.make_mlp(d, 32), ref.flatten_params(params),
                                    noise.shape[1], noise=noise, kernel=kernel)
            np.testing.assert_allclose(out.S.cpu().numpy(), py["stoch_int_fht"], rtol=1e-5, atol=2e-6)
            assert np.array_equal(out.T.cpu().numpy() + 1, py["time_steps"])


def test_checkpointed_backward_equals_full_path(golden):
    """Gradient with state checkpoints every C passes (+ recompute) == gradient with every state kept."""
    from rl_sde_is_b200.reinforce_deterministic_core import sample_loss_vectorized
    g = golden("rollout_torch_1d")
    d, alpha, beta, dt = _env(g, "a_")
    env = _make_env(d, alpha, beta, dt)
    grads = {}
    for C in (1, 4, 16, 32):
        model = _model_from(g, "a_", d)
        loss, _, _ = sample_loss_vectorized(env, model, 8, noise=g["a_noise"], ckpt_every=C, kernel="thread")
        loss.backward()
        grads[C] = torch.cat([p.grad.reshape(-1) for p in model.parameters()]).numpy()
    for C in (4, 16, 32):
        # only the fp32 summation order over (trajectory, pass) changes with the segment length
        np.testing.assert_allclose(grads[C], grads[1], rtol=1e-4, atol=1e-4 * np.abs(grads[1]).max())


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("d", [3, 10])
def test_loss_and_gradient_higher_dimension_match_oracle(d, kernel):
    """d = 10 is config 4's shape; the reference has no d = 10 env, so the check is against the torch restatement
    (pinned on the reference's 1-D / 2-D fixtures) replaying the kernel's own Philox increments."""
    from rl_sde_is_b200 import rollout as R
    from rl_sde_is_b200.models import DeterministicPolicy
    from rl_sde_is_b200.reinforce_deterministic_core import sample_loss_vectorized
    torch.manual_seed(10 + d)
    model = DeterministicPolicy(d, d, [32, 32], nn.Tanh())
    model.policy[4].bias.data.fill_(2.5)
    env = _make_env(d, 1.0, 1.0, 0.005)
    K, lim = 24, 3000
    noise = R.noise_fill(77, K, d, lim, env.dt).cpu().numpy()
    py = ref.rollout_loss_torch(d, 1.0, 1.0, 0.005, {k: v.detach().clone() for k, v in model.state_dict().items()}, noise)
    assert py["all_hit"]
    loss, ret, steps = sample_loss_vectorized(env, model, K, seed=77, n_steps_lim=lim, kernel=kernel)      # in-kernel Philox
    assert np.array_equal(steps, py["time_steps"].astype(np.float64))
    np.testing.assert_allclose(ret, py["return_fht"], rtol=1e-5)
    np.testing.assert_allclose(float(loss.detach()), float(py["loss"]), rtol=5e-5)
    loss.backward()
    gscale = max(np.abs(v).max() for v in py["grads"].values())
    for k, p in model.named_parameters():
        np.testing.assert_allclose(p.grad.numpy(), py["grads"][k], rtol=2e-4, atol=5e-4 * gscale, err_msg=k)


@pytest.mark.parametrize("kernel", KERNELS)
def test_reinforce_iterations_match_reference(golden, kernel):
    """Three zero_grad -> loss -> backward -> Adam.step iterations on recorded noise follow the reference's parameters."""
    from rl_sde_is_b200.reinforce_deterministic_core import sample_loss_vectorized
    g = golden("reinforce_iters")
    env = _make_env(1, 1.0, 1.0, 0.005)
    model = _model_from(g, "it0_", 1)
    opt = torch.optim.Adam(model.parameters(), lr=1e-2)
    for it in range(3):
        opt.zero_grad()
        loss, ret, steps = sample_loss_vectorized(env, model, 8, noise=g[f"it{it}_noise"], kernel=kernel)
        loss.backward()
        opt.step()
        assert np.array_equal(steps, g[f"it{it}_time_steps"])
        np.testing.assert_allclose(float(loss), float(g[f"it{it}_loss"]), rtol=1e-4)
        for k, v in model.state_dict().items():
            np.testing.assert_allclose(v.numpy(), g[f"it{it + 1}_param.{k}"], rtol=0, atol=2e-4, err_msg=f"it{it} {k}")


# ------------------------------------------------------------------------------ numpy path, injected noise
@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("prefix", ["a_", "b_"])
def test_test_policy_vectorized_matches_reference(golden, prefix, kernel):
    from rl_sde_is_b200.approximate_methods import estimate_fht_vectorized, test_policy_vectorized
    g = golden("rollout_numpy_1d")
    e = g[prefix + "env"]
    env = _make_env(1, float(e[1]), float(e[2]), float(e[3]))
    env.discretize_state_space(float(e[4]))
    model = _model_from(g, prefix, 1)
    res = test_policy_vectorized(env, model, batch_size=g[prefix + "noise"].shape[1], policy_opt=g[prefix + "policy_opt"],
                                 noise=g[prefix + "noise"], kernel=kernel)
    want = g[prefix + "result"]
    assert res[2] == want[2]                                                     # mean hit index: exact
    np.testing.assert_allclose(res[0], want[0], rtol=1e-6)
    np.testing.assert_allclose(res[1], want[1], rtol=1e-5)
    np.testing.assert_allclose(res[3], want[3], rtol=1e-4, atol=1e-9)
    fht = estimate_fht_vectorized(env, model, batch_size=g[prefix + "noise"].shape[1], noise=g[prefix + "noise"], kernel=kernel)
    assert fht == float(g[prefix + "fht"])


@pytest.mark.parametrize("kernel", KERNELS)
def test_estimate_fht_2d_matches_reference(golden, kernel):
    from rl_sde_is_b200.approximate_methods import estimate_fht_vectorized
    g = golden("rollout_numpy_2d")
    d, alpha, beta, dt = _env(g, "a_")
    fht = estimate_fht_vectorized(_make_env(d, alpha, beta, dt), _model_from(g, "a_", d), batch_size=g["a_noise"].shape[1],
                                  noise=g["a_noise"], kernel=kernel)
    assert fht == float(g["a_fht"])


def test_unfinished_rollouts_return_nan(golden):
    from rl_sde_is_b200.approximate_methods import test_policy_vectorized
    g = golden("rollout_numpy_1d")
    env = _make_env(1, 1.0, 1.0, 0.005)
    env.discretize_state_space(0.05)
    res = test_policy_vectorized(env, _model_from(g, "b_", 1), batch_size=64, k_max=5, policy_opt=np.zeros((81, 1)), seed=1)
    assert len(res) == 4 and all(np.isnan(r) for r in res)                       # approximate_methods.py:640-643


# ------------------------------------------------------------------------------ single passes
def test_env_step_matches_reference(golden):
    g = golden("env_step")
    env = _make_env(1, 1.0, 1.0, 0.005)
    for rt in ("state-action", "state-action-next-state"):
        tag = rt.replace("-", "_")
        nxt, r, done, dbt = env.step(g["states1"], g["actions1"], reward_type=rt, dbt=g[f"np1_{tag}_dbt"])
        assert nxt.dtype == np.float64 and np.array_equal(nxt, g[f"np1_{tag}_next"])       # bit-exact
        assert np.array_equal(r, g[f"np1_{tag}_r"]) and np.array_equal(done, g[f"np1_{tag}_done"])
        nxt, r, done, dbt = env.step_torch(torch.from_numpy(g["states1"]), torch.from_numpy(g["actions1"]), reward_type=rt,
                                           dbt=torch.from_numpy(g[f"th1_{tag}_dbt"]))
        assert nxt.dtype == torch.float32 and np.array_equal(nxt.numpy(), g[f"th1_{tag}_next"])
        assert np.array_equal(r.numpy(), g[f"th1_{tag}_r"]) and np.array_equal(done.numpy(), g[f"th1_{tag}_done"])
    env2 = _make_env(2, 1.0, 1.0, 0.005)
    nxt, r, done, _ = env2.step(g["states2"], g["actions2"], dbt=g["np2_dbt"])
    assert np.array_equal(nxt, g["np2_next"]) and np.array_equal(done, g["np2_done"])
    np.testing.assert_allclose(r, g["np2_r"], rtol=1e-7)
    nxt, r, done, _ = env2.step_torch(torch.from_numpy(g["states2"]), torch.from_numpy(g["actions2"]), dbt=torch.from_numpy(g["th2_dbt"]))
    assert np.array_equal(nxt.numpy(), g["th2_next"]) and np.array_equal(done.numpy(), g["th2_done"])
    np.testing.assert_allclose(r.numpy(), g["th2_r"], rtol=3e-7)


def test_env_step_draws_its_own_noise():
    env = _make_env(1, 1.0, 1.0, 0.005)
    env.rng_seed = 11
    x = np.full((20000, 1), -1.0, dtype=np.float32)
    _, _, _, dbt = env.step(x, np.zeros_like(x))
    z = dbt.ravel() / np.sqrt(0.005)
    assert abs(z.mean()) < 0.03 and abs(z.var() - 1) < 0.03
    assert np.allclose(dbt, c_oracle.noise_fill(11, 20000, 1, 1, 0.005)[0], atol=2e-6)


# ------------------------------------------------------------------------------ in-kernel RNG
def test_noise_stream_matches_c_restatement():
    from rl_sde_is_b200 import rollout as R
    for d in (1, 2, 3, 10):
        gpu = R.noise_fill(1234, 257, d, 37, 0.005, traj_offset=5, pass_begin=2).cpu().numpy()
        cpu = c_oracle.noise_fill(1234, 257, d, 37, 0.005, traj_offset=5, pass_begin=2)
        np.testing.assert_allclose(gpu, cpu, rtol=0, atol=3e-6)                   # MUFU log/sqrt/sincos vs libm


def test_rng_rollout_equals_replay_of_its_own_noise():
    """Philox mode == injected mode fed with rlsde_noise_fill output: the in-kernel stream is exactly the exported one."""
    from rl_sde_is_b200 import _lib as L
    from rl_sde_is_b200 import rollout as R
    torch.manual_seed(1)
    from rl_sde_is_b200.models import DeterministicPolicy
    for d in (1, 2, 10):
        m = DeterministicPolicy(d, d, [32, 32], nn.Tanh())
        m.policy[4].bias.data.fill_(1.5 if d > 1 else 0.5)
        env = _make_env(d, 1.0, 1.0, 0.005)
        params = R.flat_parameters(m).detach().numpy()
        K, lim = 300, 1500
        noise = R.noise_fill(99, K, d, lim, 0.005)
        outs = {}
        for kernel in KERNELS:
            a = R.rollout_forward(R.env_struct(env, L.HIT_ALL_GE_LB), L.make_mlp(d, 32), params, K, seed=99, n_steps_lim=lim, kernel=kernel)
            b = R.rollout_forward(R.env_struct(env, L.HIT_ALL_GE_LB), L.make_mlp(d, 32), params, K, noise=noise, n_steps_lim=lim, kernel=kernel)
            assert torch.equal(a.T, b.T) and torch.equal(a.G, b.G) and torch.equal(a.S, b.S)
            outs[kernel] = a
        # the two kernel families sum the dot products in different orders: same trajectories to rounding
        same = outs["thread"].T == outs["warp"].T
        assert same.float().mean() > 0.97
        assert torch.allclose(outs["thread"].G[same], outs["warp"].G[same], rtol=2e-5)


def test_rng_rollout_matches_c_restatement_per_trajectory():
    from rl_sde_is_b200 import _lib as L
    from rl_sde_is_b200 import rollout as R
    from rl_sde_is_b200.models import DeterministicPolicy
    torch.manual_seed(2)
    m = DeterministicPolicy(1, 1, [32, 32], nn.Tanh())
    m.policy[4].bias.data.fill_(0.8)
    env = _make_env(1, 1.0, 1.0, 0.005)
    params = R.flat_parameters(m).detach().numpy()
    K = 4096
    out = R.rollout_forward(R.env_struct(env, L.HIT_ALL_GE_LB), L.make_mlp(1, 32), params, K, seed=7, n_steps_lim=4000,
                            traj_offset=1000)
    c = c_oracle.rollout(1, 32, params, 1.0, 1.0, 0.005, K, seed=7, n_steps_lim=4000, traj_offset=1000)
    T, G = out.T.cpu().numpy(), out.G.cpu().numpy()
    same = T == c["T"]
    assert same.mean() > 0.97          # increments differ by ~1e-6 (MUFU vs libm): a few boundary crossings may move
    np.testing.assert_allclose(G[same], c["G"][same], rtol=2e-5)
    assert abs(G.mean() - c["G"].mean()) < 5e-3 * abs(c["G"].mean())


def test_results_do_not_depend_on_sharding_or_batch_size():
    from rl_sde_is_b200 import _lib as L
    from rl_sde_is_b200 import rollout as R
    from rl_sde_is_b200.models import DeterministicPolicy
    torch.manual_seed(4)
    m = DeterministicPolicy(1, 1, [32, 32], nn.Tanh())
    m.policy[4].bias.data.fill_(1.0)
    env_c, mlp_c = R.env_struct(_make_env(1, 1.0, 1.0, 0.005), L.HIT_ALL_GE_LB), L.make_mlp(1, 32)
    params = R.flat_parameters(m).detach().numpy()
    full = R.rollout_forward(env_c, mlp_c, params, 30000, seed=5, n_steps_lim=3000)
    lo = R.rollout_forward(env_c, mlp_c, params, 12345, seed=5, n_steps_lim=3000, traj_offset=0, K_global=30000)
    hi = R.rollout_forward(env_c, mlp_c, params, 30000 - 12345, seed=5, n_steps_lim=3000, traj_offset=12345, K_global=30000)
    assert torch.equal(full.G, torch.cat([lo.G, hi.G])) and torch.equal(full.T, torch.cat([lo.T, hi.T]))
    again = R.rollout_forward(env_c, mlp_c, params, 30000, seed=5, n_steps_lim=3000)
    assert np.array_equal(full.stats, again.stats)                               # deterministic reduction


def test_importance_sampling_estimator_is_policy_independent():
    """E^u[exp(G - S_exact)] = Psi(x0) for any control: ~0.1565 for beta = 1, dt = 0.005 (SURVEY App. C)."""
    from rl_sde_is_b200.approximate_methods import is_estimate
    from rl_sde_is_b200.models import DeterministicPolicy
    env = _make_env(1, 1.0, 1.0, 0.005)
    vals = []
    for bias in (0.0, 1.0):
        torch.manual_seed(1)
        m = DeterministicPolicy(1, 1, [32, 32], nn.Tanh())
        m.policy[4].bias.data.fill_(bias)
        s = is_estimate(env, m, 400000, n_steps_lim=20000, seed=3)
        assert s["n_unfinished"] == 0
        vals.append(s)
        se = s["is_rel_error"] * s["is_mean"] / np.sqrt(s["n"])
        assert abs(s["is_mean"] - 0.1565) < 5 * se + 0.002
    assert vals[1]["is_rel_error"] < vals[0]["is_rel_error"]                     # a drift towards the target reduces variance
    assert abs(vals[0]["mean_hit_index"] - 731.6) < 10                           # uncontrolled mean hitting pass (BASELINE.md)


def test_fast_tanh_is_statistically_equivalent():
    from rl_sde_is_b200 import _lib as L
    from rl_sde_is_b200 import rollout as R
    from rl_sde_is_b200.models import DeterministicPolicy
    torch.manual_seed(1)
    m = DeterministicPolicy(1, 1, [32, 32], nn.Tanh())
    m.policy[4].bias.data.fill_(0.7)
    env_c, mlp_c = R.env_struct(_make_env(1, 1.0, 1.0, 0.005), L.HIT_ALL_GE_LB), L.make_mlp(1, 32)
    params = R.flat_parameters(m).detach().numpy()
    a = R.summarize(R.rollout_forward(env_c, mlp_c, params, 200000, seed=8, n_steps_lim=20000).stats)
    b = R.summarize(R.rollout_forward(env_c, mlp_c, params, 200000, seed=8, n_steps_lim=20000, tanh="fast").stats)
    assert abs(a["mean_return"] - b["mean_return"]) < 0.01 * abs(a["mean_return"])
    assert abs(a["mean_hit_index"] - b["mean_hit_index"]) < 0.01 * a["mean_hit_index"]


# ------------------------------------------------------------------------------ tables
@pytest.mark.parametrize("tag", ["h01", "b4"])
def test_tables_match_reference(golden, tag):
    from rl_sde_is_b200.dynamic_programming import compute_p_tensor_batch, compute_r_table
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D
    from rl_sde_is_b200.tabular_dp_tables import check_p_tensor
    g = golden("tables")
    alpha, beta, dt, hs, ha = g[tag + "_cfg"]
    env = DoubleWellStoppingTime1D(beta=beta, alpha=alpha, dt=dt)
    env.set_action_space_bounds()
    env.discretize_state_space(hs)
    env.discretize_action_space(ha)
    P, Rt = compute_p_tensor_batch(env), compute_r_table(env)
    assert P.dtype == np.float64 and P.shape == g[tag + "_P"].shape and P.flags["C_CONTIGUOUS"]
    assert np.array_equal(Rt, g[tag + "_R"]) and np.signbit(Rt[env.ts_idx]).all()          # bit-exact, incl. the -0.0 rows
    assert np.abs(P - g[tag + "_P"]).max() < 1e-13                                         # north_star asks for 1e-6
    assert np.array_equal(P[:, env.ts_idx, :], g[tag + "_P"][:, env.ts_idx, :])
    assert check_p_tensor(env, P)


def test_tables_full_size_properties(golden):
    """Config 3 (401 x 401 x 601): sub-sample and the x = -1 column against the reference, column sums, slabs."""
    from rl_sde_is_b200.dynamic_programming import compute_p_tensor_batch
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D
    from rl_sde_is_b200.tabular_dp_tables import check_p_tensor
    g = golden("tables")
    env = DoubleWellStoppingTime1D()
    env.set_action_space_bounds()
    env.discretize_state_space(0.01)
    env.discretize_action_space(0.01)
    P = compute_p_tensor_batch(env, device_out=True)
    assert tuple(P.shape) == (401, 401, 601) and check_p_tensor(env, P)
    st = g["h001_P_stride"]
    sub = P[::int(st[0]), ::int(st[1]), ::int(st[2])].cpu().numpy()
    assert np.abs(sub - g["h001_P_sub"]).max() < 1e-13
    assert np.abs(P[:, 100, :].cpu().numpy() - tables_h001_column(g)).max() < 1e-13
    assert abs(float(P.sum()) - float(g["h001_P_sum"])) < 1e-6 and abs(float((P * P).sum()) - float(g["h001_P_sumsq"])) < 1e-6
    slab = compute_p_tensor_batch(env, device_out=True, sprime_range=(137, 259))
    assert torch.equal(slab, P[137:259])                # a slab holds exactly the entries of the full tensor
    # the erf/erfc path (two CDF evaluations per cell edge, the reference's formula literally) agrees with the
    # quadrature fast path used above
    E = compute_p_tensor_batch(env, device_out=True, exact_cdf=True)
    assert float((E - P).abs().max()) < 2e-14 and check_p_tensor(env, E)
    assert np.abs(E[::int(st[0]), ::int(st[1]), ::int(st[2])].cpu().numpy() - g["h001_P_sub"]).max() < 1e-13
    assert torch.equal(compute_p_tensor_batch(env, device_out=True, exact_cdf=True, sprime_range=(137, 259)), E[137:259])


# ------------------------------------------------------------------------------ DP sweeps (SURVEY 8f-1)
def test_dp_sweeps_match_reference(golden):
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D
    from rl_sde_is_b200.tabular_dp_policy_iteration import policy_update_vect
    from rl_sde_is_b200.tabular_dp_qvalue_iteration import q_table_update_vect
    from rl_sde_is_b200.tabular_dp_sweeps import DeviceTables
    from rl_sde_is_b200.tabular_dp_value_iteration import v_table_update_vect
    g, t = golden("dp_sweeps"), golden("tables")
    env = DoubleWellStoppingTime1D()
    env.set_action_space_bounds(); env.discretize_state_space(0.1); env.discretize_action_space(0.1)
    R, P = t["h01_R"], t["h01_P"]
    for gi, gamma in enumerate(g["gamma"]):
        q = g["q0"].copy()
        for it in range(3):
            q = q_table_update_vect(env, R, P, q, gamma)
            assert isinstance(q, np.ndarray) and np.abs(q - g[f"g{gi}_q{it + 1}"]).max() < 1e-12
        assert np.abs(v_table_update_vect(env, R, P, g["v0"], gamma) - g[f"g{gi}_v1"]).max() < 1e-12
        assert np.array_equal(policy_update_vect(env, R, P, g["v0"], gamma), g[f"g{gi}_pi1"])
    T = DeviceTables(env, R, P)                      # resident tables: 200 sweeps reproduce the reference's fixed point
    q = torch.as_tensor(g["q0"], device="cuda")
    for it in range(200):
        q = q_table_update_vect(env, None, T, q, 1.0)
    assert q.is_cuda and np.abs(q.cpu().numpy() - g["q200"]).max() < 1e-11


def test_qvalue_iteration_full_size_tables():
    """Config 3 tables (773 MB) resident on the device: q-value iteration converges and its fixed point is consistent."""
    from rl_sde_is_b200.dynamic_programming import compute_p_tensor_batch, compute_r_table
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D
    from rl_sde_is_b200.tabular_dp_sweeps import DeviceTables, qvalue_iteration
    env = DoubleWellStoppingTime1D()
    env.set_action_space_bounds(); env.discretize_state_space(0.01); env.discretize_action_space(0.01)
    np.random.seed(0)
    T = DeviceTables(env, compute_r_table(env, device_out=True), compute_p_tensor_batch(env, device_out=True))
    res = qvalue_iteration(env, gamma=1.0, n_iterations=1500, r_table=None, p_tensor=T)
    q, v = res["q_table"], res["v_table"]
    again = T.sweep(torch.as_tensor(v, device="cuda"), 1.0).cpu().numpy()
    assert np.abs(again - q).max() < 1e-4                                    # Bellman residual after 1 500 sweeps (2e-6 measured)
    assert np.all(v[env.ts_idx] == 0.0) and np.all(v[env.not_ts_idx] < 0)    # value = -E[cost to reach the target set]
    v_init = v[env.state_init_idx[0]]
    # -log E[exp(-tau)] = 1.855 is a lower bound on the optimal expected cost (Jensen); the discretised optimum is close
    assert -2.6 < v_init < -1.7


# ------------------------------------------------------------------------------ replay-buffer sampler (SURVEY 8f-4)
@pytest.mark.parametrize("prefix", ["a_", "b_", "c_"])
def test_replay_sampler_matches_reference(golden, prefix):
    """sample_trajectories_buffer_vectorized on the recorded increments fills a ReplayBuffer like the reference does:
    same number of tuples in the same (pass-major) order, done flags and -0.0 rewards exact, float32 values within
    1e-5 relative (the policy is evaluated by FFMA2 dot products in another summation order than torch's)."""
    from rl_sde_is_b200.approximate_methods import sample_trajectories_buffer_vectorized
    from rl_sde_is_b200.replay_buffers import ReplayBuffer
    g = golden("replay")
    d, alpha, beta, dt = _env(g, prefix)
    env, model = _make_env(d, alpha, beta, dt), _model_from(g, prefix, d)
    K, n_max, n, ptr = (int(v) for v in g[prefix + "cfg"])
    buf = ReplayBuffer(size=K * n_max, state_dim=d, action_dim=d)
    stored = sample_trajectories_buffer_vectorized(env, model, buf, K, n_max, noise=g[prefix + "noise"])
    assert stored == n and buf.size == n and buf.ptr == ptr
    assert np.array_equal(buf.done[:n], g[prefix + "done"])
    assert np.array_equal(np.signbit(buf.rewards[:n]), np.signbit(g[prefix + "rewards"]))
    assert np.array_equal(buf.rewards[:n][g[prefix + "done"]], g[prefix + "rewards"][g[prefix + "done"]])
    for name in ("states", "actions", "rewards", "next_states"):
        got, want = getattr(buf, name)[:n], g[prefix + name]
        assert got.dtype == want.dtype and got.shape == want.shape, name
        np.testing.assert_allclose(got, want, rtol=1e-5, atol=2e-6, err_msg=name)
    assert abs(buf.estimate_episode_length() - g[prefix + "done"].sum() / n) < 1e-12
    # a batch that does not fit behind the write pointer raises, as in the reference (replay_buffers.py:61-65)
    small = ReplayBuffer(size=n - 1, state_dim=d, action_dim=d)
    with pytest.raises(ValueError):
        sample_trajectories_buffer_vectorized(env, model, small, K, n_max, noise=g[prefix + "noise"])


def test_replay_sampler_rng_and_device_buffer():
    """In-kernel RNG: the transition stream is consistent with itself (next state of pass k = state of pass k+1, one done
    flag per finished episode, rewards = -(1 + a^2/2) dt), equals the replay of rlsde_noise_fill through the
    injected-noise path bit for bit, and a DeviceReplayBuffer wraps around."""
    from rl_sde_is_b200 import rollout as R
    from rl_sde_is_b200.approximate_methods import sample_transitions, sample_trajectories_buffer_vectorized
    from rl_sde_is_b200.replay_buffers import DeviceReplayBuffer
    env = _make_env(1, 1.0, 1.0, 0.005)
    torch.manual_seed(3)
    from rl_sde_is_b200.models import DeterministicPolicy
    model = DeterministicPolicy(1, 1, [32, 32], nn.Tanh())
    model.policy[4].bias.data.fill_(1.0)
    K, n_max = 3000, 4000
    tr = sample_transitions(env, model, K, n_max, seed=77, order="trajectory")
    counts = tr.counts.cpu().numpy()
    assert len(tr) == counts.sum() and int(tr.done.sum()) == K
    ends = np.cumsum(counts)
    s, a, r, ns, dn = (t.cpu().numpy() for t in (tr.states, tr.actions, tr.rewards, tr.next_states, tr.done))
    assert dn[ends - 1].all() and dn.sum() == K                      # done exactly on the last tuple of every episode
    inner = np.ones(len(tr), dtype=bool)
    inner[ends - 1] = False
    assert np.array_equal(ns[np.nonzero(inner)[0], 0], s[np.nonzero(inner)[0] + 1, 0])      # chained states
    assert np.all(s[ends - counts, 0] == -1.0)
    np.testing.assert_allclose(r[inner], -(1.0 + 0.5 * a[inner, 0].astype(np.float64) ** 2) * 0.005, rtol=1e-6)
    assert np.all(r[~inner] == 0.0) and np.all(np.signbit(r[~inner]))
    # same stream through the injected-noise path
    noise = R.noise_fill(77, K, 1, int(counts.max()), env.dt)
    tr2 = sample_transitions(env, model, K, n_max, noise=noise, order="trajectory")
    for x, y in ((tr.states, tr2.states), (tr.actions, tr2.actions), (tr.rewards, tr2.rewards), (tr.next_states, tr2.next_states)):
        assert torch.equal(x, y)
    # pass-major order = stable sort of the trajectory-major stream by pass index
    tr3 = sample_transitions(env, model, K, n_max, seed=77, order="reference")
    k_idx = np.arange(len(tr)) - np.repeat(ends - counts, counts)
    perm = np.argsort(k_idx, kind="stable")
    assert np.array_equal(tr3.states.cpu().numpy(), s[perm]) and np.array_equal(tr3.done.cpu().numpy(), dn[perm])
    # device-resident ring
    ring = DeviceReplayBuffer(size=len(tr) // 2 + 5, state_dim=1, action_dim=1)
    n_stored = sample_trajectories_buffer_vectorized(env, model, ring, K, n_max, seed=77)
    assert n_stored == len(tr) and ring.size == ring.max_size and ring.ptr == 0
    batch = ring.sample_batch(256)
    assert batch["states"].is_cuda and batch["states"].shape == (256, 1) and batch["done"].dtype == torch.bool


# ------------------------------------------------------------------------------ SURVEY 8f-2 / 8f-3 on the device path
def test_optimal_tables_from_hjb_solution(golden):
    """compute_optimal_{q,v}_table (tabular_dp_tables.py:19-42) with the HJB value function: equal to the reference's NumPy
    expression on the reference's own h = 0.1 tables; and the discrete chain agrees with the continuous solution."""
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D
    from rl_sde_is_b200.tabular_dp_tables import compute_optimal_q_table, compute_optimal_v_table
    from rl_sde_is_b200.tabular_dp_sweeps import qvalue_iteration
    g = golden("tables")
    env = DoubleWellStoppingTime1D(beta=1.0, alpha=1.0, dt=0.005)
    env.set_action_space_bounds()
    env.discretize_state_space(0.1)
    env.discretize_action_space(0.1)
    sol = env.get_hjb_solver()
    assert sol.u_opt.shape == (env.n_states, 1) and sol.value_function.shape == (env.n_states,)
    v_opt, P, R = -sol.value_function, g["h01_P"], g["h01_R"]
    d = np.where(env.is_in_ts, 1, 0)[:, None]
    q_ref = (1 - d) * np.dot(np.moveaxis(P, 0, -1), v_opt) + R                            # tabular_dp_tables.py:35-41
    q = compute_optimal_q_table(env, R, P, v_opt, sol.u_opt)
    np.testing.assert_allclose(q, q_ref, rtol=1e-12, atol=1e-13)
    a_idx = env.get_action_idx(sol.u_opt)
    v = compute_optimal_v_table(env, R, P, v_opt, sol.u_opt)
    np.testing.assert_allclose(v, q_ref[np.arange(env.n_states), a_idx], rtol=1e-12, atol=1e-13)
    # value iteration on the fine tables converges to the time-discretised value: within 5 % of -(-log Psi) at x0 = -1
    env.discretize_state_space(0.01)
    env.discretize_action_space(0.01)
    sol = env.get_hjb_solver()
    out = qvalue_iteration(env, gamma=1.0, n_iterations=1500)
    i0 = int(env.get_state_idx(env.state_init)[0])
    assert abs(out["v_table"][i0] - (-sol.value_function[i0])) < 0.05 * abs(sol.value_function[i0])
    greedy = env.action_space_h[out["greedy_action_idx"]]
    inner = (env.state_space_h > -1.5) & (env.state_space_h < 0.8)
    assert np.abs(greedy[inner] - sol.u_opt[inner, 0]).max() < 0.15                       # greedy action ~ HJB control


def test_reinforce_writes_and_loads_reference_layout(tmp_path):
    """reinforce() leaves agent.npz + model_n-it{i} in the reference's run directory; load=True reads them back;
    load=True, test=True re-tests the stored backups; test_policy_vectorized takes the HJB policy table."""
    from rl_sde_is_b200 import utils_path as up
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D
    from rl_sde_is_b200.reinforce_deterministic_core import reinforce
    up.set_data_dir(tmp_path)
    env = DoubleWellStoppingTime1D(beta=1.0, alpha=1.0, dt=0.005)
    env.discretize_state_space(0.05)
    policy_opt = env.get_hjb_solver().u_opt
    kw = dict(d_hidden_layer=32, batch_size=16, lr=1e-2, n_iterations=4, seed=1, backup_freq_iterations=2, verbose=False)
    data = reinforce(env, test=True, test_batch_size=64, test_freq_iterations=2, policy_opt=policy_opt, **kw)
    rel = data["rel_dir_path"]
    assert rel == "doublewell-1d-st__beta1.0_alpha1.0/reinforce-deterministic/init-state-1.0_gamma1.000_hidden-size32_K2e+01_lr1.0e-02_n-iter4e+00_seed1"
    assert sorted(os.listdir(os.path.join(tmp_path, rel))) == ["agent.npz", "model_n-it0", "model_n-it2", "model_n-it4"]
    assert data["test_policy_l2_errors"].shape == (3,) and np.all(np.isfinite(data["test_policy_l2_errors"]))
    back = reinforce(env, load=True, **kw)
    for key in ("returns", "time_steps", "losses", "exp_returns", "var_returns", "exp_time_steps", "cts", "test_mean_returns"):
        assert np.array_equal(back[key], data[key]), key
    assert back["returns"].dtype == np.float32 and back["time_steps"].dtype == np.float64 and back["seed"] == 1
    assert type(back["model"]).__name__ == "DeterministicPolicy"
    again = reinforce(env, load=True, test=True, test_batch_size=64, test_freq_iterations=2, policy_opt=policy_opt, **kw)
    assert again["test_mean_returns"].shape == (3,) and np.array_equal(again["losses"], data["losses"])


@pytest.mark.parametrize("fixture,prefix", [("rollout_torch_1d", "a_"), ("rollout_torch_2d", "a_")])
def test_fused_training_step_equals_autograd_route(golden, fixture, prefix):
    """reinforce()'s single-synchronisation step (K1 + K2 enqueued back to back, one device-to-host copy) gives exactly
    what sample_loss_vectorized + backward() give: same kernels, same arguments."""
    from rl_sde_is_b200.reinforce_deterministic_core import _loss_and_grads_fused, sample_loss_vectorized
    g = golden(fixture)
    d, alpha, beta, dt = _env(g, prefix)
    env = _make_env(d, alpha, beta, dt)
    K = g[prefix + "noise"].shape[1]
    m1, m2 = _model_from(g, prefix, d), _model_from(g, prefix, d)
    loss1, ret1, steps1 = sample_loss_vectorized(env, m1, K, noise=g[prefix + "noise"])
    loss1.backward()
    loss2, ret2, steps2 = _loss_and_grads_fused(env, m2, K, noise=g[prefix + "noise"])
    assert float(loss1.detach()) == loss2 and np.array_equal(ret1, ret2) and np.array_equal(steps1, steps2)
    for (k, p1), (_, p2) in zip(m1.named_parameters(), m2.named_parameters()):
        assert torch.equal(p1.grad, p2.grad), k
    np.testing.assert_allclose(loss2, float(g[prefix + "loss"]), rtol=2e-5)
    # in-kernel RNG, larger batch (thread-per-trajectory kernels, length-sorted reverse pass)
    torch.manual_seed(5)
    from rl_sde_is_b200.models import DeterministicPolicy
    ma = DeterministicPolicy(d, d, [32, 32], nn.Tanh())
    ma.policy[4].bias.data.fill_(1.5)
    mb = DeterministicPolicy(d, d, [32, 32], nn.Tanh())
    mb.load_state_dict(ma.state_dict())
    la, ra, sa = sample_loss_vectorized(env, ma, 6000, seed=9, n_steps_lim=20000)
    la.backward()
    lb, rb, sb = _loss_and_grads_fused(env, mb, 6000, seed=9, n_steps_lim=20000)
    assert float(la.detach()) == lb and np.array_equal(ra, rb) and np.array_equal(sa, sb)
    for (k, p1), (_, p2) in zip(ma.named_parameters(), mb.named_parameters()):
        assert torch.equal(p1.grad, p2.grad), k


# ------------------------------------------------------------------------------ time-sliced scheduling of K1
@pytest.mark.parametrize("f64", [False, True])
def test_time_sliced_rollout_is_bit_identical(monkeypatch, f64):
    """The forward kernel's FIFO of continuation records (slices of RLSDE_FWD_QUANTUM passes) changes only the schedule:
    every per-trajectory output equals the run-to-completion launch bit for bit, whatever the quantum; so do the state
    checkpoints (hence the gradient) and the transition stream."""
    from rl_sde_is_b200 import _lib as L, rollout as R
    from rl_sde_is_b200.models import DeterministicPolicy
    env = _make_env(1, 1.0, 1.0, 0.005)
    torch.manual_seed(11)
    model = DeterministicPolicy(1, 1, [32, 32], nn.Tanh())
    model.policy[4].bias.data.fill_(0.4)
    params = R.flat_parameters(model).detach().numpy()
    rule = L.HIT_X0_IN_LB_RB if f64 else L.HIT_ALL_GE_LB
    env_c, mlp_c = R.env_struct(env, rule), L.make_mlp(1, 32)
    K, lim = 60000, 700                     # > 148 x 128 lanes' worth: the persistent-grid path; ~15 % never hit within lim
    outs = {}
    for q in ("0", "4", "32", "128"):
        monkeypatch.setenv("RLSDE_FWD_QUANTUM", q)
        o = R.rollout_forward(env_c, mlp_c, params, K, seed=123, n_steps_lim=lim, state_f64=f64, stoch_int="exact", want_logw=True,
                              store_path=not f64, ckpt_every=4)
        outs[q] = (o.G.clone(), o.S.clone(), o.T.clone(), o.logw.clone(), None if f64 else o.path.clone(), o.stats.copy())
        if not f64 and q in ("0", "32"):
            outs[q] += (R.rollout_backward(env_c, mlp_c, params, o, 1.0 / K).clone(),)
    ref_out = outs["0"]
    assert int((ref_out[2] < 0).sum()) > 0.05 * K and int((ref_out[2] >= 0).sum()) > 0.5 * K
    for q in ("4", "32", "128"):
        for a, b in zip(ref_out[:4], outs[q][:4]):
            assert torch.equal(a, b), q
        assert np.array_equal(ref_out[5], outs[q][5]), q
        if not f64:
            # checkpoints: compare what the reverse pass reads (slots up to the hit index)
            T = ref_out[2].cpu().numpy()
            n_ck = np.where(T >= 0, T // 4 + 1, (lim + 3) // 4)
            mask = torch.as_tensor(np.arange(ref_out[4].shape[1])[None, :] < n_ck[:, None], device=ref_out[4].device)
            assert torch.equal(ref_out[4][..., 0][mask], outs[q][4][..., 0][mask]), q
    if not f64:
        assert torch.equal(outs["0"][6], outs["32"][6])


def test_time_sliced_transition_stream(monkeypatch):
    from rl_sde_is_b200.approximate_methods import sample_transitions
    from rl_sde_is_b200.models import DeterministicPolicy
    env = _make_env(1, 1.0, 1.0, 0.005)
    torch.manual_seed(3)
    model = DeterministicPolicy(1, 1, [32, 32], nn.Tanh())
    model.policy[4].bias.data.fill_(1.0)
    res = {}
    for q in ("0", "16"):
        monkeypatch.setenv("RLSDE_FWD_QUANTUM", q)
        tr = sample_transitions(env, model, 30000, 3000, seed=5, order="trajectory")
        res[q] = tr
    for name in ("states", "actions", "rewards", "next_states", "done", "counts"):
        assert torch.equal(getattr(res["0"], name), getattr(res["16"], name)), name


# ------------------------------------------------------------------------------ edge cases
@pytest.mark.parametrize("K", [0, 1, 31, 33, 148 * 128, 148 * 128 + 1])
def test_rollout_ragged_batch_sizes(K):
    """Empty, single, ragged-warp batches and both sides of the small-batch / persistent-grid switch: every trajectory's
    result is a function of (seed, trajectory id) only, so a batch is a prefix of a larger one, bit for bit."""
    from rl_sde_is_b200 import _lib as L, rollout as R
    from rl_sde_is_b200.models import DeterministicPolicy
    env = _make_env(1, 1.0, 1.0, 0.005)
    torch.manual_seed(2)
    model = DeterministicPolicy(1, 1, [32, 32], nn.Tanh())
    model.policy[4].bias.data.fill_(1.2)
    params = R.flat_parameters(model).detach().numpy()
    env_c, mlp_c = R.env_struct(env, L.HIT_ALL_GE_LB), L.make_mlp(1, 32)
    big = R.rollout_forward(env_c, mlp_c, params, 148 * 128 + 64, seed=4, n_steps_lim=3000, kernel="thread")
    out = R.rollout_forward(env_c, mlp_c, params, K, seed=4, n_steps_lim=3000, kernel="thread")
    assert out.G.shape == (K,) and out.T.shape == (K,)
    assert torch.equal(out.G, big.G[:K]) and torch.equal(out.S, big.S[:K]) and torch.equal(out.T, big.T[:K])
    st = out.stats
    assert st[L.ST_N] == K and st[L.ST_N_UNFINISHED] == int((out.T < 0).sum())
    if K:
        assert st[L.ST_USEFUL_STEPS] == float(torch.where(out.T >= 0, out.T + 1, torch.full_like(out.T, 3000)).sum())


def test_rollout_pass_budget_of_one_and_short_noise():
    """n_steps_lim = 1: nothing can be detected (the hit test runs on the current state, x0 is outside the target set);
    injected noise shorter than the budget caps the rollout at the noise length."""
    from rl_sde_is_b200 import _lib as L, rollout as R
    from rl_sde_is_b200.models import DeterministicPolicy
    env = _make_env(1, 1.0, 1.0, 0.005)
    torch.manual_seed(2)
    model = DeterministicPolicy(1, 1, [32, 32], nn.Tanh())
    params = R.flat_parameters(model).detach().numpy()
    env_c, mlp_c = R.env_struct(env, L.HIT_ALL_GE_LB), L.make_mlp(1, 32)
    out = R.rollout_forward(env_c, mlp_c, params, 500, seed=1, n_steps_lim=1)
    assert bool((out.T == -1).all()) and out.stats[L.ST_USEFUL_STEPS] == 500
    u0 = float(model(torch.tensor([[-1.0]])).item())
    np.testing.assert_allclose(out.G.cpu().numpy(), -(1 + 0.5 * u0 * u0) * 0.005, rtol=1e-5)
    noise = R.noise_fill(3, 500, 1, 7, env.dt)
    capped = R.rollout_forward(env_c, mlp_c, params, 500, n_steps_lim=10**6, noise=noise)
    assert bool((capped.T == -1).all()) and capped.stats[L.ST_USEFUL_STEPS] == 500 * 7


@pytest.mark.parametrize("Ns,Na", [(6, 4), (7, 5), (16, 33), (2, 2)])
def test_dp_sweep_even_and_odd_column_counts(Ns, Na):
    """The sweep reads 16-byte pairs; with an even column count all rows share one alignment (one partial array), with
    an odd count they alternate (two).  Random tensors of both kinds against the NumPy contraction."""
    from types import SimpleNamespace
    from rl_sde_is_b200.tabular_dp_sweeps import DeviceTables
    rng = np.random.default_rng(Ns * 100 + Na)
    P = rng.random((Ns, Ns, Na))
    R_ = -rng.random((Ns, Na))
    in_ts = rng.random(Ns) < 0.3
    v = rng.standard_normal(Ns)
    T = DeviceTables(SimpleNamespace(is_in_ts=in_ts), R_, P)
    got = T.sweep(v, 0.9).cpu().numpy()
    want = R_ + (1 - in_ts[:, None].astype(float)) * 0.9 * np.einsum("psa,p->sa", P, v)
    np.testing.assert_allclose(got, want, rtol=1e-13, atol=1e-14)
    vmax, arg = T.rowmax(torch.as_tensor(want, device="cuda"), want_arg=True)
    assert np.array_equal(arg.cpu().numpy(), want.argmax(axis=1)) and np.array_equal(vmax.cpu().numpy(), want.max(axis=1))


# ------------------------------------------------------------------------------ device-resident REINFORCE loop
def test_device_resident_training_loop_matches_host_loop():
    """reinforce(device_loop=True) -- parameters, Adam state and logs on the GPU, one asynchronous C call per iteration --
    follows reinforce(device_loop=False) (torch.optim.Adam on the CPU module after every fused step): same Philox keys,
    same kernels, so losses / returns / hit passes of iteration 0 are identical and the trajectories of the parameters
    stay together to float32 rounding of the Adam update."""
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D
    from rl_sde_is_b200.reinforce_deterministic_core import reinforce
    env = DoubleWellStoppingTime1D(beta=1.0, alpha=1.0, dt=0.005)
    kw = dict(d_hidden_layer=32, batch_size=64, lr=1e-2, n_iterations=6, seed=3, verbose=False, save=False)
    host = reinforce(env, device_loop=False, **kw)
    dev = reinforce(env, device_loop=True, **kw)
    assert np.array_equal(host["returns"][:64], dev["returns"][:64]) and np.array_equal(host["time_steps"][:64], dev["time_steps"][:64])
    assert host["losses"][0] == dev["losses"][0]
    np.testing.assert_allclose(dev["losses"], host["losses"], rtol=2e-3)
    np.testing.assert_allclose(dev["exp_time_steps"], host["exp_time_steps"], rtol=2e-2)
    for (k, a), (_, b) in zip(host["model"].named_parameters(), dev["model"].named_parameters()):
        np.testing.assert_allclose(b.detach().numpy(), a.detach().numpy(), rtol=0, atol=2e-4, err_msg=k)
    assert dev["cts"].shape == (6,) and np.all(dev["cts"] > 0) and dev["returns"].shape == (6 * 64,)
    # one Adam step on the device equals torch.optim.Adam's to float32 rounding
    m0 = reinforce(env, device_loop=False, **{**kw, "n_iterations": 1})["model"]
    m1 = reinforce(env, device_loop=True, **{**kw, "n_iterations": 1})["model"]
    for (k, a), (_, b) in zip(m0.named_parameters(), m1.named_parameters()):
        np.testing.assert_allclose(b.detach().numpy(), a.detach().numpy(), rtol=0, atol=3e-7, err_msg=k)


@pytest.mark.parametrize("d,f64", [(1, False), (1, True), (2, False)])
def test_tail_handoff_to_warp_kernel_is_bit_identical(monkeypatch, d, f64):
    """Run-to-completion launches leave their last live trajectories to the warp-per-trajectory kernel, which continues
    them with K1's summation orders: outputs (incl. the l2 error and the path checkpoints) equal the launch without the
    hand-off bit for bit."""
    from rl_sde_is_b200 import _lib as L, rollout as R
    from rl_sde_is_b200.models import DeterministicPolicy
    env = _make_env(d, 1.0, 1.0, 0.005)
    torch.manual_seed(21)
    model = DeterministicPolicy(d, d, [32, 32], nn.Tanh())
    model.policy[4].bias.data.fill_(0.6 if d == 1 else 1.6)
    params = R.flat_parameters(model).detach().numpy()
    rule = L.HIT_X0_IN_LB_RB if (f64 and d == 1) else L.HIT_ALL_GE_LB
    env_c, mlp_c = R.env_struct(env, rule), L.make_mlp(d, 32)
    K = 30000
    pol = np.linspace(-1, 1, 81) if d == 1 else None
    grid = (-2.0, 2.0, 0.05) if d == 1 else None
    outs = []
    for h in ("0", "4000", "40000"):                 # no hand-off / near the end / almost from the start
        monkeypatch.setenv("RLSDE_FWD_QUANTUM", "0")
        monkeypatch.setenv("RLSDE_FWD_HANDOFF", h)
        o = R.rollout_forward(env_c, mlp_c, params, K, seed=77, n_steps_lim=20000, state_f64=f64, want_logw=True,
                              policy_opt=pol, grid=grid, store_path=not f64, ckpt_every=2)
        outs.append(o)
    T = outs[0].T.cpu().numpy()
    assert (T >= 0).all() and T.max() > 5 * np.median(T)         # a long tail: the hand-off has something to do
    for o in outs[1:]:
        assert torch.equal(o.G, outs[0].G) and torch.equal(o.S, outs[0].S) and torch.equal(o.T, outs[0].T)
        assert torch.equal(o.logw, outs[0].logw)
        if d == 1:
            assert torch.equal(o.l2, outs[0].l2)
        if not f64:
            n_ck = T // 2 + 1
            mask = torch.as_tensor(np.arange(o.path.shape[1])[None, :] < n_ck[:, None], device=o.path.device)
            for i in range(d):
                assert torch.equal(o.path[..., i][mask], outs[0].path[..., i][mask])


def test_reverse_pass_split_between_kernel_families(monkeypatch):
    """Large batches: the longest trajectories of the length-sorted order are differentiated by the warp-per-trajectory
    kernel, the bulk by the thread-per-trajectory kernel, and the two gradients are added.  Any split gives the same
    gradient to float32 summation rounding, and the same split gives the same bits."""
    from rl_sde_is_b200 import _lib as L, rollout as R
    from rl_sde_is_b200.models import DeterministicPolicy
    env = _make_env(1, 1.0, 1.0, 0.005)
    torch.manual_seed(5)
    model = DeterministicPolicy(1, 1, [32, 32], nn.Tanh())
    model.policy[4].bias.data.fill_(0.7)
    params = R.flat_parameters(model).detach().numpy()
    env_c, mlp_c = R.env_struct(env, L.HIT_ALL_GE_LB), L.make_mlp(1, 32)
    K = 40000
    out = R.rollout_forward(env_c, mlp_c, params, K, seed=8, n_steps_lim=20000, store_path=True, ckpt_every=1, want_logw=False)
    grads = {}
    for share in ("0", "1000", "2500", "40000"):
        monkeypatch.setenv("RLSDE_BWD_WARP_SHARE", share)
        grads[share] = R.rollout_backward(env_c, mlp_c, params, out, 1.0 / K).cpu().numpy()
    monkeypatch.delenv("RLSDE_BWD_WARP_SHARE")
    default = R.rollout_backward(env_c, mlp_c, params, out, 1.0 / K).cpu().numpy()        # min(K / 16, 16 x SMs) long trajectories
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    monkeypatch.setenv("RLSDE_BWD_WARP_SHARE", str(min(K // 16, 16 * n_sm)))
    assert np.array_equal(default, R.rollout_backward(env_c, mlp_c, params, out, 1.0 / K).cpu().numpy())
    scale = np.abs(grads["0"]).max()
    for share in ("1000", "2500", "40000"):
        np.testing.assert_allclose(grads[share], grads["0"], rtol=0, atol=2e-5 * scale, err_msg=share)


@pytest.mark.parametrize("d", [1, 2])
def test_step_vectorized_stopped_intended_semantics(golden, d):
    """environments.py:164-199 raises a broadcasting error in the reference for every input; the port implements what its
    body spells out: only lanes ``idx`` move (NumPy arithmetic of ``step``), done on the next state, running-cost rewards."""
    g = golden("env_step")
    env = _make_env(d, 1.0, 1.0, 0.005)
    states, actions = g[f"states{d}"], g[f"actions{d}"]
    idx = np.array([0, 3, 4, 10, 63])
    dbt = (0.07 * np.arange(1, 1 + idx.size * d, dtype=np.float32)).reshape(idx.size, d) * (-1) ** np.arange(idx.size)[:, None]
    nxt, rew, done, db = env.step_vectorized_stopped(states, actions, idx, dbt=dbt.astype(np.float32))
    want_n, want_r, _ = ref.env_step_numpy(d, 1.0, 1.0, 0.005, states[idx], actions[idx], dbt.astype(np.float32),
                                           reward_type="state-action-next-state")
    keep = np.setdiff1d(np.arange(states.shape[0]), idx)
    assert nxt.dtype == np.float64 and nxt.shape == states.shape and rew.shape == (states.shape[0], 1)
    assert np.array_equal(nxt[idx], want_n) and np.array_equal(nxt[keep], states[keep].astype(np.float64))
    assert np.array_equal(rew[idx, 0], want_r) and np.all(rew[keep] == 0.0)
    assert np.array_equal(done, nxt >= 1.0) and np.array_equal(db, dbt.astype(np.float32))
    empty = env.step_vectorized_stopped(states, actions, np.array([], dtype=int))
    assert np.array_equal(empty[0], states.astype(np.float64)) and empty[3].shape == (0, d)


@pytest.mark.parametrize("lim,bias", [(600, 0.3), (20000, 1.0)])
def test_adaptive_tail_strategy_is_bit_identical(monkeypatch, lim, bias):
    """Default launches start running to completion and pick the tail strategy from what they see (time slices once 5 %
    of the completed trajectories have run into the budget, otherwise the hand-off).  Whatever they pick, per-trajectory
    results equal those of the forced schedules bit for bit: one workload with ~25 % capped trajectories, one with none."""
    from rl_sde_is_b200 import _lib as L, rollout as R
    from rl_sde_is_b200.models import DeterministicPolicy
    env = _make_env(1, 1.0, 1.0, 0.005)
    torch.manual_seed(11)
    model = DeterministicPolicy(1, 1, [32, 32], nn.Tanh())
    model.policy[4].bias.data.fill_(bias)
    params = R.flat_parameters(model).detach().numpy()
    env_c, mlp_c = R.env_struct(env, L.HIT_ALL_GE_LB), L.make_mlp(1, 32)
    K = 80000
    monkeypatch.delenv("RLSDE_FWD_QUANTUM", raising=False)
    monkeypatch.delenv("RLSDE_FWD_HANDOFF", raising=False)
    auto = R.rollout_forward(env_c, mlp_c, params, K, seed=31, n_steps_lim=lim, stoch_int="exact", want_logw=True)
    frac_capped = float((auto.T < 0).float().mean())
    assert (frac_capped > 0.1) if lim == 600 else (frac_capped == 0.0)
    for q in ("0", "8"):
        monkeypatch.setenv("RLSDE_FWD_QUANTUM", q)
        forced = R.rollout_forward(env_c, mlp_c, params, K, seed=31, n_steps_lim=lim, stoch_int="exact", want_logw=True)
        assert torch.equal(auto.G, forced.G) and torch.equal(auto.S, forced.S) and torch.equal(auto.T, forced.T)
        assert torch.equal(auto.logw, forced.logw) and np.array_equal(auto.stats, forced.stats)


@pytest.mark.parametrize("alpha,beta,dt,h", [(1.0, 4.0, 0.001, 0.004), (5.0, 1.0, 0.005, 0.016), (1.0, 1.0, 0.001, 0.008)])
def test_table_quadrature_path_against_exact_cdf_path(alpha, beta, dt, h):
    """The Gauss-Legendre / recurrence path of the table builder at cell widths between 0.1 and 0.2 sd, against the
    erf/erfc path (the reference's formula literally) on the same device: |dP| < 1e-13, columns sum to 1."""
    from rl_sde_is_b200.dynamic_programming import compute_p_tensor_batch, p_tensor_column_sums
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D
    env = DoubleWellStoppingTime1D(beta=beta, alpha=alpha, dt=dt)
    env.set_action_space_bounds()
    env.discretize_state_space(h)
    env.discretize_action_space(0.25)
    d_cell = h / (env.sigma * np.sqrt(dt))
    assert 0.1 < d_cell <= 0.2
    fast = compute_p_tensor_batch(env, device_out=True)
    exact = compute_p_tensor_batch(env, device_out=True, exact_cdf=True)
    assert float((fast - exact).abs().max()) < 1e-13
    assert np.abs(p_tensor_column_sums(fast).cpu().numpy() - 1).max() < 1e-12
    # slabs of the fast path are exactly the rows of the full tensor
    slab = compute_p_tensor_batch(env, device_out=True, sprime_range=(37, 211))
    assert torch.equal(slab, fast[37:211])


@pytest.mark.parametrize("na,base_off", [(24, 0), (25, 0), (26, 0), (27, 0), (25, 1), (27, 3), (26, 1)])
def test_table_row_classes_for_every_row_length_and_base_alignment(na, base_off):
    """The quadrature kernel walks rows in residue classes (4 for an odd row length Ns x Na, 2 for 2 mod 4, 1 for 0 mod 4)
    and shifts each class's column tiles so that stores are 32-byte aligned; the shift depends on the row length, on the
    slab's first row and on where the output starts.  Every combination against the erf/erfc kernel (plain column tiles),
    incl. outputs that start 8 and 24 bytes past a 32-byte boundary, and slabs that start inside a class period."""
    from rl_sde_is_b200.dynamic_programming import compute_p_tensor_batch
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D
    env = DoubleWellStoppingTime1D(beta=1.0, alpha=5.0, dt=0.005)
    env.set_action_space_bounds()
    env.discretize_state_space(0.016)                                       # 251 states: cell width 0.16 sd
    env.action_space_h = -3.0 + 0.25 * np.arange(na)
    env.n_actions = na
    env.h_action = 0.25
    ns = env.n_states
    assert ns % 2 == 1 and (ns * na) % 4 == {24: 0, 25: 3, 26: 2, 27: 1}[na]
    exact = compute_p_tensor_batch(env, device_out=True, exact_cdf=True)
    buf = torch.full((ns * ns * na + 8,), float("nan"), dtype=torch.float64, device="cuda")
    out = buf[base_off:base_off + ns * ns * na].view(ns, ns, na)
    fast = compute_p_tensor_batch(env, out=out)
    assert fast.data_ptr() == out.data_ptr() and float((fast - exact).abs().max()) < 1e-13
    assert torch.isnan(buf[:base_off]).all() and torch.isnan(buf[base_off + ns * ns * na:]).all()      # nothing outside
    for lo, hi in ((0, ns), (1, 2), (37, 211), (38, 39), (250, 251), (3, 250)):
        sbuf = torch.full(((hi - lo) * ns * na + 8,), float("nan"), dtype=torch.float64, device="cuda")
        sout = sbuf[base_off:base_off + (hi - lo) * ns * na].view(hi - lo, ns, na)
        slab = compute_p_tensor_batch(env, out=sout, sprime_range=(lo, hi))
        assert torch.equal(slab, fast[lo:hi]), (lo, hi)
        assert torch.isnan(sbuf[:base_off]).all() and torch.isnan(sbuf[base_off + (hi - lo) * ns * na:]).all()


# ------------------------------------------------------------------------------ tensor-core reverse pass
# max |g_kernel - g_f64| / max |g_f64| over the cases below, largest measured on an NVIDIA B200 (1000 W power limit):
# d <= 4 2.8e-7 (d = 1, ckpt 8), 3.6x; d = 10 1.26e-5 (K = 40 000, ckpt 4: float16 x 3 split of the padded d-sized products), 2.4x
K2M_GRAD_TOL = {"d <= 4": 1e-6, "d = 10": 3e-5}


@pytest.mark.parametrize("d,ckpt,K", [(1, 1, 6000), (1, 8, 6000), (2, 1, 6000), (3, 4, 6000), (10, 16, 6000), (10, 4, 40000), (4, 2, 40000)])
def test_reverse_pass_tensor_core_kernel_matches_float64_autograd(d, ckpt, K):
    """K2m (mma.sync, float16 x 3 operand split, fp64 partials) on its in-kernel increments against float64 autograd of the
    reference-mode loss along the kernel's hit passes, where tests/test_gpu_fp64_reference.py does not go: checkpoint
    spacing 2, a budget of 4 000 passes, K = 40 000 (the 128-thread launch shape; d > 4: the d-sized products are
    padded HMMA tiles as well).  The reference runs over chunks of trajectories, each on rollout.noise_fill's bit-exact copy
    of its increments, so that its autograd graph stays within a few GB."""
    from rl_sde_is_b200 import _lib as L, rollout as R
    from rl_sde_is_b200.models import DeterministicPolicy
    torch.manual_seed(4)
    m = DeterministicPolicy(d, d, [32, 32], nn.Tanh())
    m.policy[4].bias.data.fill_(0.8 if d == 1 else 3.0)
    dt = 0.005
    env = _make_env(d, 1.0, 1.0, dt)
    params = R.flat_parameters(m).detach().numpy()
    env_c, mlp_c = R.env_struct(env, L.HIT_ALL_GE_LB), L.make_mlp(d, 32)
    fo = R.rollout_forward(env_c, mlp_c, params, K, seed=21, n_steps_lim=4000, store_path=True, ckpt_every=ckpt, want_logw=False,
                           kernel="thread")
    assert int(fo.stats[L.ST_N_UNFINISHED]) == 0
    lib = L.load()
    ws = R._workspace(fo.G.device, K)
    order = torch.argsort(fo.T, descending=True, stable=True)

    def kernel_grad():
        g = torch.empty(int(lib.rlsde_param_count(mlp_c)), dtype=torch.float32, device=fo.G.device)
        rc = lib.rlsde_rollout_bwd(env_c, mlp_c, params.ctypes.data, fo.cfg, 0, fo.G.data_ptr(), fo.T.data_ptr(), fo.path.data_ptr(),
                                   order.data_ptr(), 1.0 / K, g.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
        L.check(rc, "rlsde_rollout_bwd")
        return g.cpu().numpy().astype(np.float64)

    g = kernel_grad()
    T = fo.T.cpu().numpy()
    sd = {k: v.detach() for k, v in m.state_dict().items()}
    want = np.zeros_like(g)
    chunk = 10000
    for lo in range(0, K, chunk):
        hi = min(K, lo + chunk)
        noise = R.noise_fill(21, hi - lo, d, int(T[lo:hi].max()) + 1, dt, traj_offset=lo)
        r = ref.rollout_reference(d, 1.0, 1.0, dt, sd, noise, hit_index=T[lo:hi], grad_modes=("reference",), device="cuda")
        want += (hi - lo) / K * np.concatenate([r["grads"]["reference"][k].reshape(-1) for k in ref.PARAM_KEYS])
        del noise, r
    err = np.abs(g - want).max() / np.abs(want).max()
    print(f"K2m against float64 autograd: d = {d}, ckpt = {ckpt}, K = {K}, longest {int(T.max()) + 1} passes: {err:.3e}")
    assert np.isfinite(g).all() and err <= K2M_GRAD_TOL["d <= 4" if d <= 4 else "d = 10"], (d, ckpt, K, err)
    # and the tensor-core kernel is deterministic (static assignment, ordered reduction)
    assert np.array_equal(kernel_grad(), g)
