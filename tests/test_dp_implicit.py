"""The tensor-free Bellman sweep (rlsde_dp_sweep_implicit) without a GPU: the band rule it uses to skip cells, restated
here, keeps every column's skipped mass at or below 2^-60; and the arguments it refuses before any device work."""
import numpy as np
import pytest
from scipy.special import ndtr

from rl_sde_is_b200 import _lib as L

BAND_Z = 9.0                     # csrc/dp_implicit.cu
INVALID = -1
FAKE = 1 << 20                   # never dereferenced: every call below is refused first


def band(x, h, mu, sd):
    """Rows the kernel visits: cell s' spans [L(s'), U(s')] with U(s') = x[s'+1] - h, U(Ns-1) = +inf, L(s') = U(s'-1),
    L(0) = -inf; the band is [first s' with U >= mu - z sd, last s' with L <= mu + z sd]."""
    reach = BAND_Z * sd
    inner = x[1:] - h                                               # U(0 .. Ns-2) = L(1 .. Ns-1)
    lo = int(np.searchsorted(inner, mu - reach, side="left"))
    hi = int(np.searchsorted(inner, mu + reach, side="right"))
    return lo, hi


def skipped_mass(x, h, mu, sd):
    lo, hi = band(x, h, mu, sd)
    assert 0 <= lo <= hi < len(x)
    below = ndtr((x[lo] - h - mu) / sd) if lo > 0 else 0.0         # cells 0 .. lo-1 and the left tail
    above = ndtr(-(x[hi + 1] - h - mu) / sd) if hi < len(x) - 1 else 0.0
    return below + above, hi - lo + 1


def grids():
    for ns in (1, 2, 41, 401, 4001):
        yield f"uniform{ns}", np.linspace(-2.0, 2.0, ns) if ns > 1 else np.array([-1.0]), 2.0 / max(ns - 1, 1)
    x = np.linspace(-2.0, 2.0, 81)
    x[1:-1] += 0.01 * np.sin(np.arange(1, 80))
    yield "nonuniform81", x, 0.025


def test_band_skips_at_most_2_pow_minus_60():
    worst, cut = 0.0, 0
    for name, x, h in grids():
        span = x[-1] - x[0]
        means = np.concatenate([x[0] + np.array([-3.0, -0.5, -1e-3, 0.0, 1e-3, 0.3]) * max(span, 1.0),
                                x[-1] + np.array([-0.3, -1e-3, 0.0, 1e-3, 0.5, 3.0]) * max(span, 1.0),
                                np.linspace(x[0], x[-1], 17)])
        for sd in (0.5, 0.1, 0.0224, 0.003):
            for mu in means:
                mass, rows = skipped_mass(x, h, mu, sd)
                assert mass <= 2.0 ** -60, (name, mu, sd, mass)
                worst = max(worst, mass)
                cut += rows < len(x)
    assert cut > 100                 # the rule does skip rows in most cases, so the bound above is not vacuous
    assert worst > 2.0 ** -70        # ... and it is close to what the rule allows


def test_band_of_narrow_transition_is_narrow():
    """Config 5's environment (beta = 4, dt = 1e-3) on a grid of h_s = 1e-3: the band spans about 2 x 9 sd."""
    x = np.round(np.arange(-2.0, 2.0 + 1e-3, 1e-3), 3)
    sd = np.sqrt(2.0 / 4.0) * np.sqrt(1e-3)
    lo, hi = band(x, 5e-4, -1.0, sd)
    assert abs((hi - lo + 1) - 2 * BAND_Z * sd / 1e-3) <= 3


def call(null=(), Ns=401, Na=601, alpha=1.0, sigma=np.sqrt(2.0), dt=0.005, h=0.005, uniform=1, step=0.01):
    p = {n: (0 if n in null else FAKE) for n in ("sgrid", "agrid", "ts", "R", "v", "values")}
    return L.load().rlsde_dp_sweep_implicit(p["sgrid"], Ns, p["agrid"], Na, p["ts"], alpha, sigma, dt, h, uniform, step,
                                            p["R"], p["v"], 1.0, p["values"], None)


CASES = [(f"{n}_null", dict(null=(n,))) for n in ("sgrid", "agrid", "ts", "R", "v", "values")] + [
    ("Ns_zero", dict(Ns=0)), ("Ns_negative", dict(Ns=-1)), ("Na_zero", dict(Na=0)), ("Na_negative", dict(Na=-5)),
    ("sigma_zero", dict(sigma=0.0)), ("sigma_negative", dict(sigma=-1.0)), ("sigma_nan", dict(sigma=float("nan"))),
    ("dt_zero", dict(dt=0.0)), ("dt_negative", dict(dt=-0.005)), ("dt_nan", dict(dt=float("nan"))),
    ("h_zero", dict(h=0.0)), ("h_negative", dict(h=-0.005)),
    ("uniform_step_zero", dict(step=0.0)), ("uniform_step_negative", dict(step=-0.01)),
    ("uniform_step_nan", dict(step=float("nan"))),
    ("grid_above_2_pow_31_blocks", dict(Ns=1 << 30, Na=601)), ("Na_above_int32", dict(Na=1 << 31)),
]


@pytest.mark.parametrize("kw", [pytest.param(kw, id=name) for name, kw in CASES])
def test_refused_before_device_work(kw):
    assert call(**kw) == INVALID
