"""The tensor-free Bellman sweep (ImplicitTables, rlsde_dp_sweep_implicit) against the sweep over the dense tensor
(DeviceTables, rlsde_dp_sweep), against the reference's fixtures, and on a grid whose tensor would not fit (770 GB)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _env(hs, ha, alpha=1.0, beta=1.0, dt=0.005, grid=None):
    from rl_sde_is_b200.environments import DoubleWellStoppingTime1D
    env = DoubleWellStoppingTime1D(beta=beta, alpha=alpha, dt=dt)
    env.set_action_space_bounds()
    env.discretize_state_space(hs)
    env.discretize_action_space(ha)
    if grid is not None:                     # a non-uniform state grid with the same cell half-width
        env.state_space_h = grid
        env.n_states = grid.size
        env.get_target_set_idx()
    return env


def _nonuniform():
    x = np.linspace(-2.0, 2.0, 81)
    x[1:-1] += 0.01 * np.sin(np.arange(1, 80))
    return x


# (id, env arguments, path the entries take)
GRIDS = [
    ("h0.1", dict(hs=0.1, ha=0.1), "erf"),
    ("h0.05", dict(hs=0.05, ha=0.05), "erf"),
    ("h0.01", dict(hs=0.01, ha=0.01), "quadrature"),
    ("nonuniform", dict(hs=0.05, ha=0.1, grid=_nonuniform()), "erf"),
    ("alpha0.5_beta0.5", dict(hs=0.01, ha=0.05, alpha=0.5, beta=0.5), "quadrature"),
    ("beta4_dt0.001_h0.005", dict(hs=0.005, ha=0.1, beta=4.0, dt=0.001), "erf"),
    ("beta4_dt0.001_h0.002", dict(hs=0.002, ha=0.1, beta=4.0, dt=0.001), "quadrature"),
]
GRID_PARAMS = [pytest.param(kw, path, id=name) for name, kw, path in GRIDS]


def _dense(env):
    from rl_sde_is_b200.dynamic_programming import compute_p_tensor_batch, compute_r_table
    from rl_sde_is_b200.tabular_dp_sweeps import DeviceTables
    return DeviceTables(env, compute_r_table(env, device_out=True), compute_p_tensor_batch(env, device_out=True))


def _path(env):
    h = env.h_state / 2.0
    uniform = np.abs(np.diff(env.state_space_h) - env.h_state).max() < 1e-9
    return "quadrature" if uniform and 2.0 * h / (env.sigma * np.sqrt(env.dt)) <= 0.2 else "erf"


@pytest.mark.parametrize("kw, path", GRID_PARAMS)
def test_implicit_matches_dense(kw, path):
    """Max |implicit - dense| <= 1e-12 for gamma in {1, 0.97}, v random and v = the HJB solution's V*."""
    from rl_sde_is_b200.tabular_dp_sweeps import ImplicitTables
    env = _env(**kw)
    assert _path(env) == path
    D, I = _dense(env), ImplicitTables(env)
    assert torch.equal(I.R, D.R)
    rng = np.random.default_rng(7)
    vs = {"random": -3.0 * rng.random(env.n_states), "V*": -env.get_hjb_solver().value_function}
    worst = {}
    for vname, v in vs.items():
        for gamma in (1.0, 0.97):
            d, i = D.sweep(v, gamma), I.sweep(v, gamma)
            assert i.is_cuda and i.shape == (env.n_states, env.n_actions)
            worst[f"{vname}, gamma={gamma}"] = err = float((i - d).abs().max())
            assert err <= 1e-12, (vname, gamma, err)
    print(f"\n[implicit vs dense] {path} Ns={env.n_states} Na={env.n_actions}: max|diff| "
          + "; ".join(f"{k}: {e:.2e}" for k, e in worst.items()))


@pytest.mark.parametrize("kw, path", GRID_PARAMS)
def test_column_mass(kw, path):
    """sweep(1, 1) - R = 1 - d[s] in every column (check_p_tensor for the operator), and runs are bitwise repeatable."""
    from rl_sde_is_b200.tabular_dp_sweeps import ImplicitTables
    env = _env(**kw)
    I = ImplicitTables(env)
    ones = torch.ones(env.n_states, dtype=torch.float64, device="cuda")
    out = I.sweep(ones, 1.0)
    live = torch.as_tensor(1.0 - env.is_in_ts.astype(np.float64), device="cuda")[:, None]
    assert float((out - I.R - live).abs().max()) <= 1e-13
    v = torch.as_tensor(-3.0 * np.random.default_rng(3).random(env.n_states), device="cuda")
    a, b = I.sweep(v, 0.97), I.sweep(v, 0.97)
    assert torch.equal(a, b) and torch.equal(a, I.sweep(v, 0.97))


def test_reference_fixtures_through_implicit_tables(golden):
    """q_/v_table_update_vect and policy_update_vect with ImplicitTables on the reference's h = 0.1 fixtures, to the
    tolerances the dense route meets (test_dp_sweeps_match_reference)."""
    from rl_sde_is_b200.tabular_dp_policy_iteration import policy_update_vect
    from rl_sde_is_b200.tabular_dp_qvalue_iteration import q_table_update_vect
    from rl_sde_is_b200.tabular_dp_sweeps import ImplicitTables
    from rl_sde_is_b200.tabular_dp_value_iteration import v_table_update_vect
    g, t = golden("dp_sweeps"), golden("tables")
    env = _env(0.1, 0.1)
    T = ImplicitTables(env, t["h01_R"])
    assert torch.equal(T.R.cpu(), torch.as_tensor(t["h01_R"]))
    for gi, gamma in enumerate(g["gamma"]):
        q = g["q0"].copy()
        for it in range(3):
            q = q_table_update_vect(env, None, T, q, gamma)
            assert isinstance(q, np.ndarray) and np.abs(q - g[f"g{gi}_q{it + 1}"]).max() < 1e-12
        assert np.abs(v_table_update_vect(env, None, T, g["v0"], gamma) - g[f"g{gi}_v1"]).max() < 1e-12
        assert np.array_equal(policy_update_vect(env, None, T, g["v0"], gamma), g[f"g{gi}_pi1"])
    q = torch.as_tensor(g["q0"], device="cuda")
    for it in range(200):
        q = q_table_update_vect(env, None, T, q, 1.0)
    assert q.is_cuda and np.abs(q.cpu().numpy() - g["q200"]).max() < 1e-11


def test_optimal_tables_through_implicit_tables(golden):
    """compute_optimal_{q,v}_table accept the operator and give the dense route's tables (CUDA tensors)."""
    from rl_sde_is_b200.tabular_dp_sweeps import ImplicitTables
    from rl_sde_is_b200.tabular_dp_tables import compute_optimal_q_table, compute_optimal_v_table
    t = golden("tables")
    env = _env(0.1, 0.1)
    sol = env.get_hjb_solver()
    v_opt, P, R = -sol.value_function, t["h01_P"], t["h01_R"]
    T = ImplicitTables(env)
    q, q_dense = compute_optimal_q_table(env, None, T, v_opt), compute_optimal_q_table(env, R, P, v_opt)
    assert q.is_cuda and np.abs(q.cpu().numpy() - q_dense).max() < 1e-12
    v, v_dense = compute_optimal_v_table(env, None, T, v_opt, sol.u_opt), compute_optimal_v_table(env, R, P, v_opt, sol.u_opt)
    assert v.is_cuda and np.abs(v.cpu().numpy() - v_dense).max() < 1e-12


def test_beyond_the_dense_limit():
    """h_s = h_a = 0.001 (4001 x 6001; the dense tensor would take 770 GB): building the operator and sweeping take under
    1 GB of device memory above what was allocated before, every column holds mass 1 - d[s], and sampled columns match the
    reference's formula evaluated in float64 by scipy."""
    from rl_sde_is_b200.tabular_dp_sweeps import ImplicitTables
    env = _env(0.001, 0.001)
    Ns, Na = env.n_states, env.n_actions
    assert (Ns, Na) == (4001, 6001) and 8 * Ns * Ns * Na > 7.6e11
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()            # tensors other tests keep alive
    T = ImplicitTables(env)
    out = T.sweep(torch.ones(Ns, dtype=torch.float64, device="cuda"), 1.0)
    out.sub_(T.R).sub_(torch.as_tensor(1.0 - env.is_in_ts.astype(np.float64), device="cuda")[:, None])
    assert float(out.abs().max()) <= 1e-13
    del out
    v = -3.0 * np.random.default_rng(5).random(Ns)
    q = T.sweep(v, 0.97)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    print(f"\n[h_s = h_a = 0.001] peak device memory of the operator and its sweeps {peak / 1e9:.3f} GB")
    assert peak < 1e9
    R = T.R.cpu().numpy()
    x, a_grid, h = env.state_space_h, env.action_space_h, env.h_state / 2.0
    for s in (0, 7, 1000, 1500, 2001, 2999, 3000, 4000):
        for a in (0, 1, 2999, 3000, 6000):
            want = R[s, a]
            if not env.is_in_ts[s]:
                p = env.state_action_transition_function(x, float(x[s]), float(a_grid[a]), h)
                want = R[s, a] + 0.97 * float(np.dot(p, v))
            assert abs(float(q[s, a]) - want) <= 1e-12, (s, a, float(q[s, a]), want)


def test_qvalue_iteration_implicit_matches_dense():
    """Config 3, 1 500 q-value-iteration sweeps: the implicit route's v is within 1e-9 of the dense route's fixed point,
    and the greedy actions agree wherever the top two q-values differ by more than 1e-9."""
    from rl_sde_is_b200.tabular_dp_sweeps import ImplicitTables, qvalue_iteration
    env = _env(0.01, 0.01)
    np.random.seed(0)
    dense = qvalue_iteration(env, gamma=1.0, n_iterations=1500)
    np.random.seed(0)
    implicit = qvalue_iteration(env, gamma=1.0, n_iterations=1500, p_tensor=ImplicitTables(env))
    dv = np.abs(implicit["v_table"] - dense["v_table"]).max()
    print(f"\n[q-value iteration, 1500 sweeps] max|v_implicit - v_dense| = {dv:.2e}")
    assert dv <= 1e-9
    top2 = np.sort(dense["q_table"], axis=1)[:, -2:]
    clear = top2[:, 1] - top2[:, 0] > 1e-9
    assert clear.sum() > 0.5 * env.n_states
    assert np.array_equal(implicit["greedy_action_idx"][clear], dense["greedy_action_idx"][clear])
