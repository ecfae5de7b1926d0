"""The ragged checkpoint store on the CPU: the layout of its base, the choice between the dense and the ragged store, and
the C ABI's refusals (rlsde_rollout_fwd_ragged / rlsde_rollout_bwd_ragged).  tests/test_gpu_ragged_store.py runs it."""
import numpy as np
import pytest
import torch

from rl_sde_is_b200 import _lib as L
from rl_sde_is_b200 import rollout as R

DT = 0.005


@pytest.mark.parametrize("C", R.RAGGED_SPACINGS)
def test_base_layout(C):
    """Restated in plain Python: every slot is covered exactly once, each trajectory's slots are contiguous and hold
    checkpoints 0 .. floor(T / C), an unfinished trajectory has none, and the total is sum (floor(T / C) + 1)."""
    rng = np.random.default_rng(C)
    T = rng.integers(0, 3000, size=257)
    T[rng.random(T.size) < 0.1] = -1
    T[:3] = [0, C - 1, C]
    base, total = R.slot_offsets(R.ragged_ckpt_counts(torch.as_tensor(T, dtype=torch.int32), C))
    base = base.numpy()
    want = sum(t // C + 1 for t in T if t >= 0)
    assert base.shape == (T.size + 1,) and base[0] == 0 and int(total) == base[-1] == want
    owner = np.full(want, -1)
    for t, k in enumerate(T):
        n = k // C + 1 if k >= 0 else 0
        assert base[t + 1] - base[t] == n
        assert (owner[base[t]:base[t + 1]] == -1).all()
        owner[base[t]:base[t + 1]] = t
    assert (owner >= 0).all()


def test_slot_offsets_of_the_transition_stream():
    """rollout_transitions' slot base is the same prefix sum: exclusive, with the total in the last entry."""
    counts = torch.tensor([3, 0, 5, 1], dtype=torch.int64)
    base, total = R.slot_offsets(counts)
    assert base.tolist() == [0, 3, 3, 8, 9] and int(total) == 9


def test_chooser_keeps_the_dense_store_where_it_fits():
    """choose_path_store returns choose_ckpt_every's spacing wherever it succeeds and None (the ragged store) exactly where
    it raises."""
    n_dense = n_ragged = 0
    for H in (32, 64, 256):
        for d in (1, 2, 10):
            for K in (100, 10**4, 7 * 10**4, 4 * 10**5, 10**6):
                for lim in (1000, 10**5, 10**6):
                    try:
                        want = R.choose_ckpt_every(K, d, lim, hidden=H)
                    except L.RlsdeError:
                        want = None
                    assert R.choose_path_store(K, d, lim, hidden=H) == want, (H, d, K, lim)
                    n_dense += want is not None
                    n_ragged += want is None
    assert n_dense > 0 and n_ragged > 0
    assert R.choose_path_store(7 * 10**4, 1, 10**6, hidden=32) is None          # the default budget at K = 7e4
    assert R.choose_path_store(6 * 10**4, 1, 10**6, hidden=256) is None         # the README's wide training row


def test_ragged_spacing():
    """The smallest spacing whose ragged store fits at width 32, spacing 1 above it, an error when even that does not fit;
    the budget is the module-level PATH_BUDGET_BYTES."""
    b = R.PATH_BUDGET_BYTES
    totals = lambda s: [s // c for c in R.RAGGED_SPACINGS]
    assert R.choose_ragged_ckpt_every(totals(b // 4), 1) == 1
    assert R.choose_ragged_ckpt_every(totals(b // 4 + 1), 1) == 2
    assert R.choose_ragged_ckpt_every(totals(b // 2), 2) == 4
    assert R.choose_ragged_ckpt_every(totals(8 * b), 1) == 32
    with pytest.raises(L.RlsdeError):
        R.choose_ragged_ckpt_every(totals(40 * b), 1)
    wide = max(b, 32 << 30) // 4
    assert R.choose_ragged_ckpt_every([wide], 1, hidden=256) == 1
    with pytest.raises(L.RlsdeError):
        R.choose_ragged_ckpt_every([wide + 1], 1, hidden=256)


def test_budget_can_be_lowered(monkeypatch):
    """Lowering PATH_BUDGET_BYTES moves both choosers: a store that fits today goes ragged, then raises."""
    assert R.choose_path_store(1000, 1, 1000) == 1
    monkeypatch.setattr(R, "PATH_BUDGET_BYTES", 1000 * 1000 * 4 // 64)
    assert R.choose_path_store(1000, 1, 1000) is None
    assert R.choose_ragged_ckpt_every([10**5 // c for c in R.RAGGED_SPACINGS], 1) == 8
    with pytest.raises(L.RlsdeError):
        R.choose_ragged_ckpt_every([10**7 // c for c in R.RAGGED_SPACINGS], 1)


def test_c_abi_refusals():
    """Both entry points refuse before any device work: RLSDE_F_HIT_BRIDGE, a spacing above 32, a NULL base or store
    (RLSDE_ERR_INVALID_ARG), the float64 state (RLSDE_ERR_UNSUPPORTED)."""
    lib = L.load()
    fake = 1 << 20                             # never dereferenced: every call below fails its argument checks first
    ws_bytes = int(lib.rlsde_workspace_bytes(64))
    params = np.zeros(1 + 32 + 32 * 32 + 32 + 32 + 1 + 64, dtype=np.float32)
    RLSDE_ERR_INVALID_ARG, RLSDE_ERR_UNSUPPORTED = -1, -2
    env = L.make_env(1, 1.0, np.sqrt(2.0), DT, 1.0, 2.0, np.full(1, -1.0), L.HIT_ALL_GE_LB)

    def cfg(flags, C):
        c = L.RlsdeRolloutCfg()
        c.K, c.K_global, c.n_steps_lim, c.flags = 64, 64, 100, flags
        c.ckpt_every, c.ckpt_stride = C, 0      # the stride is not read: 0 would be refused by the dense store
        return c

    def fwd(flags=0, C=1, base=fake, path=fake):
        return lib.rlsde_rollout_fwd_ragged(env, L.make_mlp(1, 32), params.ctypes.data, cfg(flags, C), 0, base, fake, fake,
                                            fake, path, 0, fake, ws_bytes, 0)

    def bwd(flags=0, C=1, base=fake, path=fake):
        return lib.rlsde_rollout_bwd_ragged(env, L.make_mlp(1, 32), params.ctypes.data, cfg(flags, C), 0, fake, fake, fake,
                                            base, path, 0, 1.0, fake, fake, 1 << 40, 0)

    for call in (fwd, bwd):
        assert call(L.F_HIT_BRIDGE) == RLSDE_ERR_INVALID_ARG
        assert call(L.F_STORE_PATH | L.F_HIT_BRIDGE) == RLSDE_ERR_INVALID_ARG
        assert call(C=33) == RLSDE_ERR_INVALID_ARG
        assert call(base=0) == RLSDE_ERR_INVALID_ARG
        assert call(path=0) == RLSDE_ERR_INVALID_ARG
        assert call(L.F_STATE_F64) == RLSDE_ERR_UNSUPPORTED
    assert fwd(C=0) == RLSDE_ERR_INVALID_ARG
    # the dense entry point keeps refusing a stride that cannot hold the budget
    assert lib.rlsde_rollout_fwd(env, L.make_mlp(1, 32), params.ctypes.data, cfg(L.F_STORE_PATH, 1), 0, 0, fake, fake, fake,
                                 0, 0, fake, 0, fake, ws_bytes, 0) == RLSDE_ERR_INVALID_ARG
