"""Table build + check + the Bellman-expectation tables under the HJB policy: rl_sde_is/tabular_dp_tables.py.

  * ``check_p_tensor`` (:15-17), ``dynamic_programming_tables`` (:44-72) incl. its ``agent.npz`` (utils_path).
  * ``compute_optimal_v_table`` / ``compute_optimal_q_table`` (:19-42): one Bellman-expectation sweep with the value
    function of the HJB reference solution -- the same streaming contraction as the DP sweeps (``rlsde_dp_sweep``),
    ``q[s, a] = r[s, a] + (1 - d[s]) sum_s' P[s', s, a] v_opt[s']``; the v-table reads it at the HJB policy's action indices.
    The reference gets ``value_function_opt`` / ``policy_opt`` from the external sde_hjb_solver; ``env.get_hjb_solver()``
    here provides them from ``hjb_1d`` (SURVEY 8f-3).
"""
import numpy as np
import torch

from .dynamic_programming import compute_p_tensor_batch, compute_r_table, p_tensor_column_sums
from .tabular_dp_sweeps import _like, _tables
from .utils_path import get_dynamic_programming_tables_dir_path, load_data, save_data


def check_p_tensor(env, p_tensor):
    """Every (state, action) column sums to 1 over the next-state axis (np.isclose tolerances)."""
    if torch.is_tensor(p_tensor) and p_tensor.is_cuda:
        sums = p_tensor_column_sums(p_tensor).cpu().numpy()
    else:
        sums = np.sum(np.asarray(p_tensor), axis=0)
    return bool(np.isclose(sums, 1).all())


def compute_optimal_q_table(env, r_table, p_tensor, value_function_opt, policy_opt=None):
    """``(1 - d) P^T v_opt + r`` for every (state, action)  (:32-42).  ``p_tensor`` may also be a ``DeviceTables`` or an
    ``ImplicitTables``; the result is then a CUDA tensor."""
    T = _tables(env, r_table, p_tensor)
    v = np.asarray(value_function_opt, dtype=np.float64).reshape(-1)
    return _like(T.R if T is p_tensor else p_tensor, T.sweep(v, 1.0))


def compute_optimal_v_table(env, r_table, p_tensor, value_function_opt, policy_opt):
    """The optimal q-table read at the HJB policy's discretised actions  (:19-30)."""
    q = compute_optimal_q_table(env, r_table, p_tensor, value_function_opt)
    actions_idx = env.get_action_idx(np.asarray(policy_opt, dtype=np.float64).reshape(-1, 1))
    if torch.is_tensor(q):
        return q[torch.arange(env.n_states, device=q.device), torch.as_tensor(actions_idx, device=q.device)]
    return q[np.arange(env.n_states), actions_idx]


def dynamic_programming_tables(env, value_function_opt=None, policy_opt=None, load=False, *, device=None, device_out=False,
                               save=True):
    """Build ``r_table``, ``p_tensor`` (and ``q_table`` when the HJB value function is given), assert the column-sum
    check and write ``agent.npz`` into the reference's ``dp-tables`` directory (:44-72).  ``load=True`` reads it back.
    ``device_out=True`` keeps the tables as CUDA tensors and skips the 773 MB file."""
    rel_dir_path = get_dynamic_programming_tables_dir_path(env)
    if load:
        return load_data(rel_dir_path)
    r_table = compute_r_table(env, device=device, device_out=True)
    p_tensor = compute_p_tensor_batch(env, device=device, device_out=True)
    assert check_p_tensor(env, p_tensor)
    data = {"r_table": r_table, "p_tensor": p_tensor}
    if value_function_opt is not None:
        data["q_table"] = compute_optimal_q_table(env, r_table, p_tensor, value_function_opt, policy_opt)
    if not device_out:
        data = {k: v.cpu().numpy() for k, v in data.items()}
    data["rel_dir_path"] = rel_dir_path
    if save and not device_out:
        save_data(data, rel_dir_path)
    return data
