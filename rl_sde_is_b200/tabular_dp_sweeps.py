"""Dynamic-programming sweeps on the device-resident transition tensor (SURVEY.md 8f-1).

Reference functions (same names, argument order and return types; re-exported by the modules
``tabular_dp_qvalue_iteration``, ``tabular_dp_value_iteration`` and ``tabular_dp_policy_iteration``):

  * ``q_table_update_vect(env, r_table, p_tensor, q_table, gamma)``   tabular_dp_qvalue_iteration.py:35-43
  * ``v_table_update_vect(env, r_table, p_tensor, v_table, gamma)``   tabular_dp_value_iteration.py:41-52
  * ``policy_update_vect(env, r_table, p_tensor, v_table, gamma)``    tabular_dp_policy_iteration.py:37-49

Each is one streaming pass over ``p_tensor`` (773 MB at h = 0.01): HBM-read bound on the GPU, ~0.3 s in NumPy.
``p_tensor`` / ``r_table`` may be NumPy arrays (uploaded on every call -- only sensible for small tables) or CUDA
tensors as returned by ``compute_p_tensor_batch(env, device_out=True)``; outputs follow the input kind.
``DeviceTables`` + ``qvalue_iteration`` keep everything resident for the 2 000-sweep use of the reference's README.
``ImplicitTables`` is the same operator with no tensor behind it (``rlsde_dp_sweep_implicit`` generates P inside each
sweep): memory O(Ns Na), for grids whose tensor does not fit.  Either is accepted as ``p_tensor`` by every function here.
"""
import numpy as np
import torch

from . import _lib as L
from .dynamic_programming import _device_grids, _state_grid_spacing, compute_r_table
from .rollout import _cuda_device, _ptr


class TransitionOperator:
    """A device-resident Bellman operator: ``sweep(v, gamma)`` and ``rowmax(values, want_arg)`` on (Ns, Na) CUDA tensors,
    with ``Ns``, ``Na``, ``dev``, ``R`` and ``in_ts``."""

    def _dev(self, a):
        if torch.is_tensor(a):
            return a.to(device=self.dev, dtype=torch.float64).contiguous()
        return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device=self.dev)

    def rowmax(self, values, want_arg=False):
        vmax = torch.empty(self.Ns, dtype=torch.float64, device=self.dev)
        arg = torch.empty(self.Ns, dtype=torch.int64, device=self.dev) if want_arg else None
        with torch.cuda.device(self.dev):
            rc = L.load().rlsde_dp_rowmax(_ptr(values), self.Ns, self.Na, _ptr(vmax), _ptr(arg),
                                          torch.cuda.current_stream(self.dev).cuda_stream)
        L.check(rc, "rlsde_dp_rowmax")
        return (vmax, arg) if want_arg else vmax


class DeviceTables(TransitionOperator):
    """r_table, p_tensor and the target-set mask on the GPU, plus the sweep scratch buffer."""

    def __init__(self, env, r_table, p_tensor, device=None):
        dev = p_tensor.device if torch.is_tensor(p_tensor) and p_tensor.is_cuda else _cuda_device(device)
        self.dev = dev
        self.P = self._dev(p_tensor)
        self.R = self._dev(r_table)
        self.Ns, self.Na = int(self.R.shape[0]), int(self.R.shape[1])
        if tuple(self.P.shape) != (self.Ns, self.Ns, self.Na):
            raise L.RlsdeError(f"p_tensor must have shape ({self.Ns}, {self.Ns}, {self.Na}), got {tuple(self.P.shape)}")
        self.in_ts = torch.as_tensor(np.ascontiguousarray(env.is_in_ts, dtype=np.uint8), device=dev)
        self.scratch = torch.empty(L.load().rlsde_dp_scratch_bytes(self.Ns, self.Na), dtype=torch.uint8, device=dev)

    def sweep(self, v, gamma):
        """values[s, a] = R[s, a] + (1 - d[s]) gamma sum_s' P[s', s, a] v[s']   (CUDA tensor)."""
        v = self._dev(v).reshape(-1)
        out = torch.empty((self.Ns, self.Na), dtype=torch.float64, device=self.dev)
        with torch.cuda.device(self.dev):
            rc = L.load().rlsde_dp_sweep(_ptr(self.P), self.Ns, self.Na, _ptr(self.R), _ptr(self.in_ts), _ptr(v), float(gamma),
                                         _ptr(out), _ptr(self.scratch), self.scratch.numel(),
                                         torch.cuda.current_stream(self.dev).cuda_stream)
        L.check(rc, "rlsde_dp_sweep")
        return out


class ImplicitTables(TransitionOperator):
    """The transition operator of ``env``'s own grids with no tensor behind it: each sweep generates P[s', s, a] (as
    ``compute_p_tensor_batch`` defines it) inside the kernel.  ``r_table`` defaults to ``compute_r_table(env)``."""

    def __init__(self, env, r_table=None, device=None):
        if env.d != 1:
            raise L.RlsdeError("the tabular operator covers the 1-D environment (as the reference's does)")
        self.dev = r_table.device if torch.is_tensor(r_table) and r_table.is_cuda else _cuda_device(device)
        self.consts = (float(env.alpha), float(env.sigma), float(env.dt), float(env.h_state) / 2.0)
        self.sgrid, self.agrid, self.in_ts = _device_grids(env, self.dev)     # the un-rounded action grid, as K4 reads it
        self.Ns, self.Na = int(self.sgrid.numel()), int(self.agrid.numel())
        self.R = compute_r_table(env, device=self.dev, device_out=True) if r_table is None else self._dev(r_table)
        if tuple(self.R.shape) != (self.Ns, self.Na):
            raise L.RlsdeError(f"r_table must have shape ({self.Ns}, {self.Na}), got {tuple(self.R.shape)}")
        self.uniform, self.step = _state_grid_spacing(env)

    def sweep(self, v, gamma):
        """values[s, a] = R[s, a] + (1 - d[s]) gamma sum_s' P[s', s, a] v[s']   (CUDA tensor)."""
        v = self._dev(v).reshape(-1)
        if v.numel() != self.Ns:
            raise L.RlsdeError(f"v must have {self.Ns} entries, got {v.numel()}")
        out = torch.empty((self.Ns, self.Na), dtype=torch.float64, device=self.dev)
        with torch.cuda.device(self.dev):
            rc = L.load().rlsde_dp_sweep_implicit(
                _ptr(self.sgrid), self.Ns, _ptr(self.agrid), self.Na, _ptr(self.in_ts), *self.consts, self.uniform, self.step,
                _ptr(self.R), _ptr(v), float(gamma), _ptr(out), torch.cuda.current_stream(self.dev).cuda_stream)
        L.check(rc, "rlsde_dp_sweep_implicit")
        return out


def _tables(env, r_table, p_tensor):
    return p_tensor if isinstance(p_tensor, TransitionOperator) else DeviceTables(env, r_table, p_tensor)


def _like(inp, t):
    return t if torch.is_tensor(inp) and inp.is_cuda else t.cpu().numpy()


def q_table_update_vect(env, r_table, p_tensor, q_table, gamma):
    """q <- r + (1 - d) gamma P^T max_a q   (one q-value-iteration sweep)."""
    T = _tables(env, r_table, p_tensor)
    q = T._dev(q_table)
    return _like(q_table, T.sweep(T.rowmax(q), gamma))


def v_table_update_vect(env, r_table, p_tensor, v_table, gamma):
    """v <- max_a (r + gamma (1 - d) P^T v)   (one value-iteration sweep)."""
    T = _tables(env, r_table, p_tensor)
    return _like(v_table, T.rowmax(T.sweep(v_table, gamma)))


def policy_update_vect(env, r_table, p_tensor, v_table, gamma):
    """Greedy action indices under v; target-set states get the null action (tabular_dp_policy_iteration.py:47-48)."""
    T = _tables(env, r_table, p_tensor)
    _, arg = T.rowmax(T.sweep(v_table, gamma), want_arg=True)
    arg[torch.as_tensor(np.asarray(env.ts_idx), device=T.dev)] = int(np.asarray(env.null_action_idx).reshape(-1)[0])
    return _like(v_table, arg)


def qvalue_iteration(env, gamma=1.0, n_iterations=100, *, r_table=None, p_tensor=None, q_table=None, device=None):
    """n_iterations q-value-iteration sweeps with everything resident on the GPU (tabular_dp_qvalue_iteration.py:45-119
    without the HJB error logging / plotting / file I/O, which are out of the hot path's scope).

    Tables default to a fresh device-side build of the dense tensor; pass ``p_tensor=ImplicitTables(env)`` for grids whose
    tensor does not fit.  ``q_table`` defaults to the reference's ``-np.random.rand`` init.
    Returns ``{'n_iterations', 'q_table' (NumPy), 'v_table', 'greedy_action_idx'}``."""
    from .dynamic_programming import compute_p_tensor_batch
    if p_tensor is None:
        p_tensor = compute_p_tensor_batch(env, device=device, device_out=True)
    if r_table is None:
        r_table = compute_r_table(env, device=device, device_out=True)
    T = _tables(env, r_table, p_tensor)
    q = T._dev(-np.random.rand(env.n_states, env.n_actions) if q_table is None else q_table)
    for _ in range(int(n_iterations)):
        q = T.sweep(T.rowmax(q), gamma)
    v, arg = T.rowmax(q, want_arg=True)
    return {"n_iterations": n_iterations, "q_table": q.cpu().numpy(), "v_table": v.cpu().numpy(),
            "greedy_action_idx": arg.cpu().numpy()}
