"""Tabular reward table and transition tensor on the GPU (drop-in for rl_sde_is/dynamic_programming.py).

Reference: ``compute_r_table(env)`` (:3-16) and ``compute_p_tensor_batch(env)`` (:18-36), which loop over
(state, action) in Python and call ``env.state_action_transition_function`` (environments.py:87-102)
-- 180 300 iterations x 4 scipy ``norm.cdf`` calls at h = 0.01.  Here: one launch of the streaming
table kernel (csrc/tables.cu).  The env's OWN grids are shipped to the device (the action grid is an
un-rounded ``np.arange``; regenerating it on the device would not reproduce the reference's entries).

Return types match the reference (float64 NumPy, ``P[s', s, a]`` C-ordered).  ``device_out=True`` keeps the
result on the GPU as a torch tensor (the 773 MB device-to-host copy costs ~100x the kernel).
"""
import numpy as np
import torch

from . import _lib as L
from .rollout import _cuda_device, _ptr


def _device_grids(env, dev):
    """The env's grids on the device, uploaded once per (env, grids) and kept on the env object: three small pageable
    host-to-device copies per call would otherwise serialise the host with the stream."""
    sg_h = np.ascontiguousarray(env.state_space_h, dtype=np.float64)
    ag_h = np.ascontiguousarray(env.action_space_h, dtype=np.float64)
    ts_h = np.ascontiguousarray(env.is_in_ts, dtype=np.uint8)
    key = (str(dev), sg_h.tobytes(), ag_h.tobytes(), ts_h.tobytes())
    cached = getattr(env, "_rlsde_device_grids", None)
    if cached is not None and cached[0] == key:
        return cached[1]
    grids = tuple(torch.as_tensor(a, device=dev) for a in (sg_h, ag_h, ts_h))
    try:
        env._rlsde_device_grids = (key, grids)
    except AttributeError:
        pass
    return grids


def _state_grid_spacing(env):
    """(uniform, step): whether the state grid is equally spaced to 1e-14, which lets the kernels take the quadrature
    path, and its mean spacing (x_{Ns-1} - x_0) / (Ns - 1)."""
    grid = np.asarray(env.state_space_h, dtype=np.float64)
    Ns = grid.size
    if Ns < 2:
        return 0, 0.0
    uniform = int(np.abs(grid - (grid[0] + np.arange(Ns) * (grid[-1] - grid[0]) / (Ns - 1))).max() <= 1e-14)
    return uniform, float((grid[-1] - grid[0]) / (Ns - 1))


def _tables(env, want_p, want_r, device, sprime_range=None, exact_cdf=False, out=None):
    if env.d != 1:
        raise L.RlsdeError("the tabular builder covers the 1-D environment (as the reference's does)")
    lib = L.load()
    dev = _cuda_device(device)
    sg, ag, ts = _device_grids(env, dev)
    Ns, Na = int(sg.numel()), int(ag.numel())
    lo, hi = (0, Ns) if sprime_range is None else (int(sprime_range[0]), int(sprime_range[1]))
    uniform, step = _state_grid_spacing(env)
    uniform = int(uniform and not exact_cdf)
    P = None
    if want_p:
        P = out if out is not None else torch.empty((hi - lo, Ns, Na), dtype=torch.float64, device=dev)
        if tuple(P.shape) != (hi - lo, Ns, Na) or P.dtype != torch.float64 or P.device != dev or not P.is_contiguous():
            raise L.RlsdeError(f"out must be a contiguous float64 tensor of shape {(hi - lo, Ns, Na)} on {dev}")
    Rt = torch.empty((Ns, Na), dtype=torch.float64, device=dev) if want_r else None
    with torch.cuda.device(dev):
        rc = lib.rlsde_tables(_ptr(sg), Ns, _ptr(ag), Na, _ptr(ts), int(env.is_in_ts.sum()), float(env.alpha),
                              float(env.sigma), float(env.dt), float(env.h_state) / 2.0, float(env.lb), float(env.rb),
                              lo, hi, _ptr(P), _ptr(Rt), uniform, step,
                              torch.cuda.current_stream(dev).cuda_stream)
    L.check(rc, "rlsde_tables")
    return P, Rt


def compute_r_table(env, *, device=None, device_out=False):
    """R[s, a] = -0 on the target set, else -(1 + a^2/2) dt   (float64, shape (n_states, n_actions))."""
    _, Rt = _tables(env, False, True, device)
    return Rt if device_out else Rt.cpu().numpy()


def compute_p_tensor_batch(env, *, device=None, device_out=False, sprime_range=None, exact_cdf=False, out=None):
    """P[s', s, a] (float64, shape (n_states, n_states, n_actions), action innermost).

    ``sprime_range=(begin, end)`` builds only that slab of next-states (multi-GPU sharding, SURVEY 8e).
    ``exact_cdf=True`` forces two erf/erfc evaluations per cell edge (the reference's formula literally) instead of
    the quadrature fast path used on fine uniform grids; both agree with the reference to < 1e-13.
    ``out``: preallocated CUDA tensor to build into (implies ``device_out``)."""
    P, _ = _tables(env, True, False, device, sprime_range, exact_cdf, out)
    return P if (device_out or out is not None) else P.cpu().numpy()


def p_tensor_column_sums(P_dev):
    """sum over s' of a device-resident tensor, in index order (deterministic)."""
    lib = L.load()
    n_sp, Ns, Na = (int(v) for v in P_dev.shape)
    out = torch.zeros((Ns, Na), dtype=torch.float64, device=P_dev.device)
    with torch.cuda.device(P_dev.device):
        rc = lib.rlsde_tables_colsum(_ptr(P_dev), n_sp, Ns, Na, _ptr(out), torch.cuda.current_stream(P_dev.device).cuda_stream)
    L.check(rc, "rlsde_tables_colsum")
    return out
