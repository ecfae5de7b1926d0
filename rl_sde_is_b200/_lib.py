"""ctypes binding of librlsde_b200.so (include/rlsde.h).

The product path has no CPU fallback: if the shared library is missing or a CUDA call fails, the
functions here raise.  Nothing in this module (or anywhere in the package) imports ``oracle/``.
"""
import ctypes as C
import os

import numpy as np

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RLSDE_LIB_PATH") or os.path.join(_PKG_DIR, "librlsde_b200.so")

RLSDE_MAX_D = 16
RLSDE_NSTATS = 16

# hit rules / flags / reward types (include/rlsde.h)
HIT_ALL_GE_LB = 0
HIT_X0_IN_LB_RB = 1
F_NOISE_INJECTED = 1 << 0
F_TANH_FAST = 1 << 1
F_STOCH_INT_EXACT = 1 << 2
F_STATE_F64 = 1 << 3
F_STORE_PATH = 1 << 4
F_GRAD_F32 = 1 << 5
F_HIT_BRIDGE = 1 << 6
F_KERNEL_THREAD = 1 << 8
F_KERNEL_WARP = 1 << 9
F_KERNEL_TENSOR = 1 << 10
REWARD_STATE_ACTION = 0
REWARD_STATE_ACTION_NEXT_STATE = 1

# statistics record
ST_N, ST_N_UNFINISHED, ST_SUM_G, ST_SUM_G2, ST_SUM_T, ST_SUM_T2, ST_SUM_S, ST_SUM_L2, ST_SUM_W, ST_SUM_W2, \
    ST_SUM_LOSS, ST_USEFUL_STEPS, ST_MAX_T = range(13)

# every symbol include/rlsde.h declares (checked by tests/test_abi.py)
EXPORTED_SYMBOLS = [
    "rlsde_version", "rlsde_strerror", "rlsde_last_cuda_error", "rlsde_device_info", "rlsde_supported",
    "rlsde_param_count", "rlsde_workspace_bytes", "rlsde_workspace_bytes_bwd", "rlsde_rollout_fwd", "rlsde_rollout_bwd", "rlsde_reduce_stats",
    "rlsde_tables", "rlsde_tables_colsum", "rlsde_env_step", "rlsde_noise_fill",
    "rlsde_dp_scratch_bytes", "rlsde_dp_sweep", "rlsde_dp_rowmax", "rlsde_rollout_transitions", "rlsde_launch_count", "rlsde_reinforce_step",
    "rlsde_reinforce_rollout", "rlsde_reinforce_apply", "rlsde_fwd_mma_clamp_bounds", "rlsde_rollout_fwd_table",
    "rlsde_rollout_bwd_weighted", "rlsde_rollout_fwd_ragged", "rlsde_rollout_bwd_ragged", "rlsde_dp_sweep_implicit",
]


class RlsdeEnv(C.Structure):
    _fields_ = [
        ("d", C.c_int32), ("hit_rule", C.c_int32),
        ("alpha", C.c_double * RLSDE_MAX_D),
        ("sigma", C.c_double), ("dt", C.c_double), ("lb", C.c_double), ("rb", C.c_double),
        ("x0", C.c_double * RLSDE_MAX_D),
    ]


class RlsdeMlp(C.Structure):
    _fields_ = [("d_in", C.c_int32), ("d_hidden", C.c_int32), ("d_out", C.c_int32), ("n_hidden", C.c_int32)]


class RlsdeRolloutCfg(C.Structure):
    _fields_ = [
        ("K", C.c_int64), ("traj_offset", C.c_int64), ("K_global", C.c_int64), ("seed", C.c_uint64),
        ("n_steps_lim", C.c_int64), ("noise_steps", C.c_int64), ("flags", C.c_uint32), ("ckpt_every", C.c_int32),
        ("ckpt_stride", C.c_int64), ("n_grid", C.c_int64),
        ("grid_lo", C.c_double), ("grid_hi", C.c_double), ("grid_h", C.c_double),
        # scheduling knobs, 0 = automatic (include/rlsde.h)
        ("fwd_quantum", C.c_int32), ("fwd_blocks_per_sm", C.c_int32), ("fwd_handoff", C.c_int64), ("bwd_warp_share", C.c_int64),
        ("bwd_kernel", C.c_int32), ("wide_kernel", C.c_int32), ("fwd_policy", C.c_int32),
    ]


class RlsdeError(RuntimeError):
    pass


_lib = None


def load():
    """Load librlsde_b200.so (once).  Raises if it has not been built: there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RlsdeError(
            f"{LIB_PATH} not found: build it with `python -m rl_sde_is_b200.build` "
            "(or __graft_entry__.build()); the CUDA extension is required, there is no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, u32, u64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_double
    lib.rlsde_version.restype = C.c_int
    lib.rlsde_strerror.restype = C.c_char_p
    lib.rlsde_strerror.argtypes = [C.c_int]
    lib.rlsde_last_cuda_error.restype = C.c_char_p
    lib.rlsde_launch_count.restype = C.c_longlong
    lib.rlsde_device_info.argtypes = [C.POINTER(i32)] * 3
    lib.rlsde_supported.argtypes = [i32, i32, i32]
    lib.rlsde_param_count.restype = i64
    lib.rlsde_param_count.argtypes = [C.POINTER(RlsdeMlp)]
    lib.rlsde_workspace_bytes.restype = C.c_size_t
    lib.rlsde_workspace_bytes.argtypes = [i64]
    lib.rlsde_workspace_bytes_bwd.restype = C.c_size_t
    lib.rlsde_workspace_bytes_bwd.argtypes = [i64, C.c_int32, C.c_int32]
    lib.rlsde_rollout_fwd.argtypes = [C.POINTER(RlsdeEnv), C.POINTER(RlsdeMlp), vp, C.POINTER(RlsdeRolloutCfg),
                                      vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_size_t, vp]
    lib.rlsde_rollout_fwd_table.argtypes = [C.POINTER(RlsdeEnv), vp, C.POINTER(RlsdeRolloutCfg), vp, vp, vp, vp, vp, vp, vp, vp,
                                            vp, C.c_size_t, vp]
    lib.rlsde_rollout_transitions.argtypes = [C.POINTER(RlsdeEnv), C.POINTER(RlsdeMlp), vp, C.POINTER(RlsdeRolloutCfg),
                                              vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_size_t, vp]
    lib.rlsde_reinforce_step.argtypes = [C.POINTER(RlsdeEnv), C.POINTER(RlsdeMlp), vp, vp, vp, C.POINTER(RlsdeRolloutCfg), vp,
                                         dbl, dbl, dbl, dbl, i64, vp, vp, vp, vp, vp, vp, vp, C.c_size_t, vp]
    lib.rlsde_reinforce_rollout.argtypes = [C.POINTER(RlsdeEnv), C.POINTER(RlsdeMlp), vp, C.POINTER(RlsdeRolloutCfg), vp,
                                            vp, vp, vp, vp, vp, vp, vp, vp, C.c_size_t, vp]
    lib.rlsde_reinforce_apply.argtypes = [C.POINTER(RlsdeMlp), vp, vp, vp, vp, i32, dbl, dbl, dbl, dbl, i64, vp, vp, vp]
    lib.rlsde_rollout_bwd.argtypes = [C.POINTER(RlsdeEnv), C.POINTER(RlsdeMlp), vp, C.POINTER(RlsdeRolloutCfg),
                                      vp, vp, vp, vp, vp, dbl, vp, vp, C.c_size_t, vp]
    lib.rlsde_rollout_bwd_weighted.argtypes = [C.POINTER(RlsdeEnv), C.POINTER(RlsdeMlp), vp, C.POINTER(RlsdeRolloutCfg),
                                               vp, vp, vp, vp, vp, vp, dbl, vp, vp, C.c_size_t, vp]
    lib.rlsde_rollout_fwd_ragged.argtypes = [C.POINTER(RlsdeEnv), C.POINTER(RlsdeMlp), vp, C.POINTER(RlsdeRolloutCfg),
                                             vp, vp, vp, vp, vp, vp, vp, vp, C.c_size_t, vp]
    lib.rlsde_rollout_bwd_ragged.argtypes = [C.POINTER(RlsdeEnv), C.POINTER(RlsdeMlp), vp, C.POINTER(RlsdeRolloutCfg),
                                             vp, vp, vp, vp, vp, vp, vp, dbl, vp, vp, C.c_size_t, vp]
    lib.rlsde_reduce_stats.argtypes = [i64, i64, u32, vp, vp, vp, vp, vp, vp, vp, C.c_size_t, vp]
    lib.rlsde_tables.argtypes = [vp, i64, vp, i64, vp, i64, dbl, dbl, dbl, dbl, dbl, dbl, i64, i64, vp, vp, i32, dbl, vp]
    lib.rlsde_tables_colsum.argtypes = [vp, i64, i64, i64, vp, vp]
    lib.rlsde_env_step.argtypes = [C.POINTER(RlsdeEnv), i64, vp, vp, vp, u64, i64, i64, u32, i32, vp, vp, vp, vp, vp]
    lib.rlsde_noise_fill.argtypes = [u64, i64, i64, i32, i64, i64, dbl, vp, vp]
    lib.rlsde_dp_scratch_bytes.restype = C.c_size_t
    lib.rlsde_dp_scratch_bytes.argtypes = [i64, i64]
    lib.rlsde_dp_sweep.argtypes = [vp, i64, i64, vp, vp, vp, dbl, vp, vp, C.c_size_t, vp]
    lib.rlsde_dp_sweep_implicit.argtypes = [vp, i64, vp, i64, vp, dbl, dbl, dbl, dbl, i32, dbl, vp, vp, dbl, vp, vp]
    lib.rlsde_dp_rowmax.argtypes = [vp, i64, i64, vp, vp, vp]
    lib.rlsde_fwd_mma_clamp_bounds.argtypes = [vp, vp]
    for name in ("rlsde_device_info", "rlsde_supported", "rlsde_rollout_fwd", "rlsde_rollout_bwd", "rlsde_reduce_stats",
                 "rlsde_tables", "rlsde_tables_colsum", "rlsde_env_step", "rlsde_noise_fill", "rlsde_dp_sweep", "rlsde_dp_rowmax",
                 "rlsde_rollout_transitions", "rlsde_reinforce_step", "rlsde_reinforce_rollout", "rlsde_reinforce_apply",
                 "rlsde_fwd_mma_clamp_bounds", "rlsde_rollout_fwd_table", "rlsde_rollout_bwd_weighted",
                 "rlsde_rollout_fwd_ragged", "rlsde_rollout_bwd_ragged", "rlsde_dp_sweep_implicit"):
        getattr(lib, name).restype = C.c_int
    _lib = lib
    return lib


def apply_tuning(cfg, tuning=None):
    """Scheduling knobs of a rollout cfg (include/rlsde.h: they change the schedule, never a result).  ``tuning`` is a dict
    with any of ``fwd_quantum`` (passes per time slice, 0 = run to completion), ``fwd_handoff``, ``bwd_warp_share``,
    ``fwd_blocks_per_sm``, ``bwd_kernel`` ('mma'), ``wide_kernel`` ('umma' | 'ffma'), ``fwd_policy`` ('mma' | 'ffma');
    keys that are absent fall back to the environment variables RLSDE_FWD_QUANTUM, RLSDE_FWD_HANDOFF, RLSDE_BWD_WARP_SHARE,
    RLSDE_FWD_BLOCKS_PER_SM, RLSDE_BWD_KERNEL, RLSDE_WIDE_KERNEL, RLSDE_FWD_POLICY (read HERE, in
    Python -- the library reads none), and to "automatic" if those are unset too."""
    tuning = tuning or {}

    def knob(name):
        if name in tuning and tuning[name] is not None:
            return int(tuning[name])
        v = os.environ.get("RLSDE_" + name.upper())
        return int(v) if v not in (None, "") else None

    q = knob("fwd_quantum")
    cfg.fwd_quantum = 0 if q is None else (q if q > 0 else -1)
    h = knob("fwd_handoff")
    cfg.fwd_handoff = 0 if h is None else (h if h > 0 else -1)
    w = knob("bwd_warp_share")
    cfg.bwd_warp_share = 0 if w is None else (w if w > 0 else -1)
    b = knob("fwd_blocks_per_sm")
    cfg.fwd_blocks_per_sm = 0 if b is None or b < 1 else b
    bk = tuning.get("bwd_kernel") or os.environ.get("RLSDE_BWD_KERNEL") or "auto"
    cfg.bwd_kernel = {"auto": 0, "mma": 1}[str(bk).lower()]
    wk = tuning.get("wide_kernel") or os.environ.get("RLSDE_WIDE_KERNEL") or "auto"
    cfg.wide_kernel = {"auto": 0, "umma": 1, "tcgen05": 1, "ffma": 2}[str(wk).lower()]
    fp = tuning.get("fwd_policy") or os.environ.get("RLSDE_FWD_POLICY") or "auto"
    cfg.fwd_policy = {"auto": 0, "mma": 1, "ffma": 2}[str(fp).lower()]
    return cfg


def check(status, what):
    if status != 0:
        lib = load()
        msg = lib.rlsde_strerror(status).decode()
        cuda = lib.rlsde_last_cuda_error().decode()
        raise RlsdeError(f"{what} failed: {msg} (status {status})" + (f" [{cuda}]" if cuda and status == -3 else ""))


def make_env(d, alpha, sigma, dt, lb, rb, x0, hit_rule):
    e = RlsdeEnv()
    e.d, e.hit_rule = int(d), int(hit_rule)
    al = np.broadcast_to(np.asarray(alpha, dtype=np.float64).ravel(), (d,)) if np.ndim(alpha) else np.full(d, float(alpha))
    x0 = np.asarray(x0, dtype=np.float64).ravel()
    for i in range(d):
        e.alpha[i] = float(al[i])
        e.x0[i] = float(x0[i])
    e.sigma, e.dt, e.lb, e.rb = float(sigma), float(dt), float(lb), float(rb)
    return e


def make_mlp(d, hidden, n_hidden=2):
    m = RlsdeMlp()
    m.d_in, m.d_hidden, m.d_out, m.n_hidden = int(d), int(hidden), int(d), int(n_hidden)
    return m
