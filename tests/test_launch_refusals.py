"""Status of every rollout entry point of the C ABI for the arguments it refuses before any device work.

The launch layer decides these statuses from the arguments alone, in a fixed order (shape, pointers, workspace size,
cfg fields, flag combinations), before it asks for a device: so they are the same on a machine without one. The table
holds the cases the other CPU tests do not already check."""
import numpy as np
import pytest

from rl_sde_is_b200 import _lib as L

INVALID, UNSUPPORTED, WORKSPACE = -1, -2, -5
FAKE = 1 << 20                 # never dereferenced: every call below is refused first
DT = 0.005
B, P, F64, NOISE = L.F_HIT_BRIDGE, L.F_STORE_PATH, L.F_STATE_F64, L.F_NOISE_INJECTED

# pointer arguments of each entry point, in order; every one is FAKE unless a case nulls it
PTRS = {
    "fwd": ("params", "cfg", "noise", "policy_opt", "G", "S", "T", "l2", "logw", "path", "stats", "ws"),
    "fwd_ragged": ("params", "cfg", "noise", "base", "G", "S", "T", "path", "stats", "ws"),
    "transitions": ("params", "cfg", "noise", "base", "states", "actions", "rewards", "next", "done", "G", "S", "T",
                    "stats", "ws"),
    "fwd_table": ("table", "cfg", "noise", "policy_opt", "G", "S", "T", "l2", "logw", "stats", "ws"),
    "bwd": ("params", "cfg", "noise", "G", "T", "path", "order", "grad", "ws"),
    "bwd_weighted": ("params", "cfg", "noise", "cG", "cS", "T", "path", "order", "grad", "ws"),
    "bwd_ragged": ("params", "cfg", "noise", "cG", "cS", "T", "base", "path", "order", "grad", "ws"),
    "reinforce_step": ("params", "m", "v", "cfg", "noise", "G", "S", "T", "path", "stats", "grad", "ws"),
    "reinforce_rollout": ("params", "cfg", "noise", "G", "S", "T", "path", "stats", "grad", "packed", "ws"),
}
# pointers that may be NULL (and are, unless a case sets them); the device-resident step always writes the statistics
OPTIONAL = {"noise", "policy_opt", "l2", "logw", "stats", "order"}


def call(entry, d=1, H=32, n_hidden=2, d_in=None, env=True, dt=DT, sigma=np.sqrt(2.0), hit_rule=L.HIT_ALL_GE_LB,
         flags=None, C=1, stride=100, K=64, K_global=None, traj_offset=0, noise_steps=0, n_steps_lim=100, fwd_policy=0,
         bwd_kernel=0, n_grid=401, grid_h=0.01, ws=None, null=(), set_=(), step_t=1):
    lib = L.load()
    if flags is None:              # the reverse passes and the device-resident step need the checkpoint store
        flags = P if entry.startswith("bwd") or entry.startswith("reinforce") else 0
    e = None
    if env:
        e = L.make_env(min(d, 16), 1.0, sigma, dt, 1.0, 2.0, np.full(16, -1.0), hit_rule)
        e.d = d
    mlp = L.make_mlp(d, H, n_hidden)
    if d_in is not None:
        mlp.d_in = d_in
    c = None
    if "cfg" not in null:
        c = L.RlsdeRolloutCfg()
        c.K, c.K_global, c.traj_offset, c.n_steps_lim, c.flags = K, K if K_global is None else K_global, traj_offset, n_steps_lim, flags
        c.noise_steps, c.ckpt_every, c.ckpt_stride, c.fwd_policy, c.bwd_kernel = noise_steps, C, stride, fwd_policy, bwd_kernel
        c.n_grid, c.grid_lo, c.grid_hi, c.grid_h = n_grid, -2.0, 2.0, grid_h
    optional = OPTIONAL - {"stats"} if entry.startswith("reinforce") else OPTIONAL
    p = {name: (0 if name in null or (name in optional and name not in set_) else FAKE) for name in PTRS[entry]}
    p["cfg"] = c
    ws_bytes = int(lib.rlsde_workspace_bytes(K if K > 0 else 0)) if ws is None else ws
    if entry == "fwd":
        return lib.rlsde_rollout_fwd(e, mlp, p["params"], c, p["noise"], p["policy_opt"], p["G"], p["S"], p["T"], p["l2"],
                                     p["logw"], p["path"], p["stats"], p["ws"], ws_bytes, 0)
    if entry == "fwd_ragged":
        return lib.rlsde_rollout_fwd_ragged(e, mlp, p["params"], c, p["noise"], p["base"], p["G"], p["S"], p["T"], p["path"],
                                            p["stats"], p["ws"], ws_bytes, 0)
    if entry == "transitions":
        return lib.rlsde_rollout_transitions(e, mlp, p["params"], c, p["noise"], p["base"], p["states"], p["actions"],
                                             p["rewards"], p["next"], p["done"], p["G"], p["S"], p["T"], p["stats"], p["ws"],
                                             ws_bytes, 0)
    if entry == "fwd_table":
        return lib.rlsde_rollout_fwd_table(e, p["table"], c, p["noise"], p["policy_opt"], p["G"], p["S"], p["T"], p["l2"],
                                           p["logw"], p["stats"], p["ws"], ws_bytes, 0)
    ws_bytes = 1 << 40 if ws is None else ws
    if entry == "bwd":
        return lib.rlsde_rollout_bwd(e, mlp, p["params"], c, p["noise"], p["G"], p["T"], p["path"], p["order"], 1.0, p["grad"],
                                     p["ws"], ws_bytes, 0)
    if entry == "bwd_weighted":
        return lib.rlsde_rollout_bwd_weighted(e, mlp, p["params"], c, p["noise"], p["cG"], p["cS"], p["T"], p["path"],
                                              p["order"], 1.0, p["grad"], p["ws"], ws_bytes, 0)
    if entry == "bwd_ragged":
        return lib.rlsde_rollout_bwd_ragged(e, mlp, p["params"], c, p["noise"], p["cG"], p["cS"], p["T"], p["base"], p["path"],
                                            p["order"], 1.0, p["grad"], p["ws"], ws_bytes, 0)
    if entry == "reinforce_step":
        return lib.rlsde_reinforce_step(e, mlp, p["params"], p["m"], p["v"], c, p["noise"], 1e-3, 0.9, 0.999, 1e-8, step_t,
                                        p["G"], p["S"], p["T"], p["path"], p["stats"], p["grad"], p["ws"], ws_bytes, 0)
    assert entry == "reinforce_rollout"
    return lib.rlsde_reinforce_rollout(e, mlp, p["params"], c, p["noise"], p["G"], p["S"], p["T"], p["path"], p["stats"],
                                       p["grad"], p["packed"], p["ws"], ws_bytes, 0)


MLP_ENTRIES = ("fwd", "fwd_ragged", "transitions", "bwd", "bwd_weighted", "bwd_ragged", "reinforce_step", "reinforce_rollout")
REVERSE = ("bwd", "bwd_weighted", "bwd_ragged")
REINFORCE = ("reinforce_step", "reinforce_rollout")

# (entries, case name, arguments, status)
TABLE = [
    # environment and policy shape
    (MLP_ENTRIES + ("fwd_table",), "env_null", dict(env=False), INVALID),
    (MLP_ENTRIES + ("fwd_table",), "dt_zero", dict(dt=0.0), INVALID),
    (MLP_ENTRIES + ("fwd_table",), "sigma_nan", dict(sigma=float("nan")), INVALID),
    (MLP_ENTRIES + ("fwd_table",), "hit_rule_unknown", dict(hit_rule=2), INVALID),
    (MLP_ENTRIES, "d_above_max", dict(d=17), INVALID),
    (MLP_ENTRIES, "mlp_d_in_mismatch", dict(d_in=2), INVALID),
    (MLP_ENTRIES, "depth_3", dict(n_hidden=3), UNSUPPORTED),
    (MLP_ENTRIES, "d5_h32", dict(d=5), UNSUPPORTED),
    (MLP_ENTRIES, "d3_h64", dict(d=3, H=64), UNSUPPORTED),
    (MLP_ENTRIES, "d1_h512", dict(H=512), UNSUPPORTED),
    # NULL pointers, a small workspace, and which of the two is found first
    (MLP_ENTRIES, "params_null", dict(null=("params",)), INVALID),
    (MLP_ENTRIES + ("fwd_table",), "cfg_null", dict(null=("cfg",)), INVALID),
    (MLP_ENTRIES + ("fwd_table",), "workspace_null", dict(null=("ws",)), INVALID),
    (MLP_ENTRIES + ("fwd_table",), "T_null", dict(null=("T",)), INVALID),
    (("fwd", "fwd_ragged", "transitions", "fwd_table") + REINFORCE, "G_null", dict(null=("G",)), INVALID),
    (("fwd", "fwd_ragged", "transitions", "fwd_table") + REINFORCE, "S_null", dict(null=("S",)), INVALID),
    (REVERSE + REINFORCE, "grad_null", dict(null=("grad",)), INVALID),
    (("bwd", "bwd_weighted") + REINFORCE, "path_null", dict(null=("path",)), INVALID),
    (("bwd_weighted", "bwd_ragged"), "cS_null", dict(null=("cS",)), INVALID),
    (("bwd_ragged",), "cG_null", dict(null=("cG",)), INVALID),
    (REINFORCE, "stats_null", dict(null=("stats",)), INVALID),
    (("reinforce_step",), "adam_m_null", dict(null=("m",)), INVALID),
    (("reinforce_step",), "adam_v_null", dict(null=("v",)), INVALID),
    (("reinforce_step",), "step_t_zero", dict(step_t=0), INVALID),
    (("reinforce_rollout",), "packed_null", dict(null=("packed",)), INVALID),
    (("transitions",), "states_null", dict(null=("states",)), INVALID),
    (("transitions",), "done_null", dict(null=("done",)), INVALID),
    (("transitions",), "slot_base_null", dict(null=("base",)), INVALID),
    (MLP_ENTRIES + ("fwd_table",), "workspace_1k", dict(ws=1024), WORKSPACE),
    (MLP_ENTRIES, "workspace_1k_cfg_null", dict(ws=1024, null=("cfg",)), WORKSPACE),
    (("fwd_table",), "workspace_1k_cfg_null", dict(ws=1024, null=("cfg",)), INVALID),
    (MLP_ENTRIES, "workspace_1k_d5", dict(ws=1024, d=5), UNSUPPORTED),
    (REVERSE + REINFORCE, "workspace_1k_grad_null", dict(ws=1024, null=("grad",)), INVALID),
    # cfg fields
    (MLP_ENTRIES + ("fwd_table",), "K_negative", dict(K=-1, K_global=1), INVALID),
    (MLP_ENTRIES + ("fwd_table",), "budget_zero", dict(n_steps_lim=0), INVALID),
    (MLP_ENTRIES + ("fwd_table",), "budget_above_2e9", dict(n_steps_lim=2000000001), INVALID),
    (MLP_ENTRIES + ("fwd_table",), "traj_offset_negative", dict(traj_offset=-1), INVALID),
    (MLP_ENTRIES + ("fwd_table",), "noise_steps_zero", dict(flags=NOISE, noise_steps=0), INVALID),
    (MLP_ENTRIES + ("fwd_table",), "shard_outside_batch", dict(flags=NOISE, noise_steps=100, traj_offset=8, K_global=64), INVALID),
    (MLP_ENTRIES + ("fwd_table",), "fwd_policy_3", dict(fwd_policy=3), INVALID),
    (REVERSE, "bwd_kernel_2", dict(bwd_kernel=2), UNSUPPORTED),
    (("fwd", "fwd_ragged", "transitions", "fwd_table"), "noise_null", dict(flags=NOISE, noise_steps=100), INVALID),
    (REVERSE + REINFORCE, "noise_null", dict(flags=NOISE | P, noise_steps=100), INVALID),
    (("fwd", "bwd", "bwd_weighted", "reinforce_step", "reinforce_rollout"), "stride_below_budget",
     dict(flags=P, stride=99), INVALID),
    (("fwd", "bwd", "bwd_weighted"), "stride_fits_injected_noise_only",
     dict(flags=P | NOISE, noise_steps=40, stride=39), INVALID),
    (("fwd", "bwd", "bwd_weighted"), "spacing_zero", dict(flags=P, C=0), INVALID),
    (("fwd",), "path_null", dict(flags=P, null=("path",)), INVALID),
    (("fwd_table",), "table_null_d2", dict(d=2, null=("table",)), UNSUPPORTED),
    (("fwd_table",), "store_path", dict(flags=P), INVALID),
    (("fwd",), "table_policy_without_grid", dict(set_=("policy_opt",), n_grid=0), INVALID),
    (("fwd",), "table_policy_grid_h_zero", dict(set_=("policy_opt",), grid_h=0.0), INVALID),
    (("fwd",), "table_policy_at_d2", dict(d=2, set_=("policy_opt",)), INVALID),
    (REINFORCE, "K_zero", dict(K=0, K_global=1), INVALID),
    (REINFORCE, "spacing_2", dict(flags=P, C=2, stride=50), INVALID),
    (REINFORCE, "no_store", dict(flags=0), INVALID),
    # flag conflicts: the Brownian-bridge test, the ragged store, the float64 state, the spacing
    (("fwd",), "bridge_store_path_d2", dict(d=2, flags=B | P), INVALID),
    (("fwd",), "bridge_d10", dict(d=10, flags=B), UNSUPPORTED),
    (("fwd",), "bridge_h256_d2", dict(d=2, H=256, flags=B), UNSUPPORTED),
    (("transitions",), "store_path", dict(flags=P), INVALID),
    (("transitions",), "store_path_slot_base_null", dict(flags=P, null=("base",)), INVALID),
    (("transitions",), "bridge_d2", dict(d=2, flags=B), INVALID),
    (("fwd_ragged",), "bridge_f64", dict(flags=B | F64), INVALID),
    (("fwd_ragged",), "f64_h256", dict(H=256, flags=F64), UNSUPPORTED),
    (("fwd_ragged",), "f64_d10", dict(d=10, flags=F64), UNSUPPORTED),
    (("fwd_ragged",), "spacing_33_f64", dict(C=33, flags=F64), INVALID),
    (("fwd_ragged",), "f64_noise_null", dict(flags=F64 | NOISE, noise_steps=100), UNSUPPORTED),
    (("fwd_ragged",), "bridge_d2", dict(d=2, flags=B), INVALID),
    (REVERSE, "bridge_f64", dict(flags=P | B | F64), INVALID),
    (REVERSE, "f64_without_store", dict(flags=F64), UNSUPPORTED),
    (REVERSE, "spacing_33", dict(flags=P, C=33, stride=4), INVALID),
    (REVERSE, "spacing_64_h256", dict(H=256, flags=P, C=64, stride=2), INVALID),
    (("bwd", "bwd_weighted"), "f64_h256", dict(H=256, flags=P | F64), UNSUPPORTED),
    (("bwd_ragged",), "bridge_d2", dict(d=2, flags=B), INVALID),
    (REINFORCE, "f64", dict(flags=P | F64), INVALID),
    (REINFORCE, "bridge", dict(flags=P | B), INVALID),
]


@pytest.mark.parametrize("entry, kw, status", [pytest.param(entry, kw, status, id=f"{entry}-{name}")
                                               for entries, name, kw, status in TABLE for entry in entries])
def test_refused_before_device_work(entry, kw, status):
    assert call(entry, **kw) == status
