"""NAFF tunes without a GPU: the NumPy definition (tests/naff_oracle.py) on pure tones, edge cases,
octupole detuning and the PS Booster's linear tunes through the tracking oracle; the header
constants; the argument checks that run before anything is launched."""
import os
import re

import numpy as np
import pytest
import torch

from tests import helpers as H
from tests import naff_oracle as NO

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "xline_b200.h")


def _tones(T, m, seed):
    rng = np.random.default_rng(seed)
    nu = rng.uniform(0.05, 0.45, m)
    ph = rng.uniform(0.0, 2 * np.pi, m)
    t = np.arange(T)[:, None]
    return nu, np.cos(2 * np.pi * nu * t + ph), -np.sin(2 * np.pi * nu * t + ph)


@pytest.mark.parametrize("T", [1000, 1024, 2048])
def test_oracle_recovers_pure_tones(T):
    """x - i·px of a unit circle is e^{+i(2πνt + φ)}: the tune is ν, the amplitude 1 (1/2 for the
    real signal x, whose power splits between ±ν).  The error left is mostly leakage of the
    subtracted mean into the peak."""
    nu, x, px = _tones(T, 50, seed=1)
    q, a, near = NO.naff(x, px)
    assert np.abs(q - nu).max() <= 1e-11
    assert np.abs(a - 1.0).max() <= 1e-7
    qr, ar, _ = NO.naff(x)
    assert np.abs(qr - nu).max() <= 1e-9
    assert np.abs(ar - 0.5).max() <= 1e-6
    assert not near.any()


def test_oracle_normalises_with_beta_alpha():
    """u = √β·cos φ, pu = -(sin φ + α cos φ)/√β is a linear particle at (β, α): the complex signal
    recovers ν and √(2J) = 1."""
    beta, alpha, T = 7.5, -1.3, 1024
    nu, c, s = _tones(T, 8, seed=2)
    u = np.sqrt(beta) * c
    pu = (s - alpha * c) / np.sqrt(beta)  # s = -sin φ
    q, a, _ = NO.naff(u, pu, beta, alpha)
    assert np.abs(q - nu).max() <= 1e-11
    assert np.abs(a - 1.0).max() <= 1e-7


def test_oracle_invalid_signals():
    T = 256
    _, x, px = _tones(T, 4, seed=3)
    x[17, 0] = np.nan
    px[200, 1] = np.inf
    x[:, 2] = 0.0
    px[:, 2] = 0.0
    q, a, _ = NO.naff(x, px)
    assert np.isnan(q[:3]).all()
    assert np.isnan(a[:2]).all() and a[2] == 0.0
    assert np.isfinite(q[3]) and np.isfinite(a[3])
    qr, ar, _ = NO.naff(x)
    # the real signal reads x only: column 1's inf sits in px
    assert np.isnan(qr[[0, 2]]).all() and np.isnan(ar[0]) and ar[2] == 0.0
    assert np.isfinite(qr[1]) and ar[1] > 0


def test_coarse_peak_ties_go_to_the_lowest_bin():
    mag = np.zeros((16, 3))
    mag[[3, 7], 0] = 2.0          # tie inside the complex range
    mag[[5, 12], 1] = 1.0         # 12 > M/2: outside the real range
    mag[[0, 4, 9], 2] = [9.0, 1.0, 1.0]  # k = 0 (the mean) is never a candidate
    k, near = NO.coarse_bin(mag, real=False)
    assert list(k) == [3, 5, 4] and near.all()
    k, _ = NO.coarse_bin(mag, real=True)
    assert list(k) == [3, 5, 4]


# Real signals whose largest peak, seen from the coarse bin k = M/2, is the mirror line just above
# 1/2: (offset of line 1, of line 2 in units of 1/T from 1/2, amplitude of line 2, phases), T = 256.
MIRROR_CASES = ((0.155, -1.438, 0.83, 3.78, 1.31), (-0.887, -0.253, 0.67, 1.35, 3.82))


def mirror_signals(T=256):
    c = np.array(MIRROR_CASES).T
    t = np.arange(T)[:, None]
    return (np.cos(2 * np.pi * (0.5 + c[0] / T) * t + c[3])
            + c[2] * np.cos(2 * np.pi * (0.5 + c[1] / T) * t + c[4]))


def test_oracle_folds_tunes_into_range():
    """The bracket of k = M/2 reaches past 1/2: a real signal whose root lands there is folded to
    1 - ν (the same line seen from the other side), so every real tune is in [0, 1/2] and every
    complex one in [0, 1)."""
    x = mirror_signals()
    q, a, near = NO.naff(x)
    assert (q <= 0.5).all() and (q > 0.497).all() and not near.any()
    rng = np.random.default_rng(7)
    T = 512
    nu = np.concatenate([rng.uniform(-3, 3, 200) / T, 0.5 + rng.uniform(-3, 3, 200) / T])
    t = np.arange(T)[:, None]
    qc, _, _ = NO.naff(np.cos(2 * np.pi * nu * t), -np.sin(2 * np.pi * nu * t))
    qr, _, _ = NO.naff(np.cos(2 * np.pi * nu * t + 1.0))
    assert ((qc >= 0) & (qc < 1)).all()
    assert ((qr >= 0) & (qr <= 0.5)).all()


def octupole_fodo(k3l, num_stores=2048, ids=1, qx=0.18):
    """One thin-lens FODO cell (drifts of 1 m, tune ``qx`` in both planes: 0.07 from the nearest
    fourth-order resonance) with a thin octupole at the centre of the focusing quadrupole and a
    BeamMonitor in front of it (element 0)."""
    import xline_b200 as xl

    k = 2 * np.sin(np.pi * qx)  # thin FODO: sin(μ/2) = L·k/2, L = 1 m
    els = [xl.BeamMonitor(num_stores=num_stores, start=0, skip=1, min_particle_id=0, max_particle_id=ids - 1),
           xl.Multipole(knl=[0, 0, 0, k3l]), xl.Multipole(knl=[0, k / 2]), xl.Drift(length=1.0),
           xl.Multipole(knl=[0, -k]), xl.Drift(length=1.0), xl.Multipole(knl=[0, k / 2])]
    return xl.Line(elements=els)


def detuning_errors(q, a, tw, k3l):
    """Relative deviation of ν - qx from the first-order k3l·β²·A²/(32π) (A = the NAFF amplitude
    √(2J); dpx = -k3l·x³/6 comes from H = k3l·x⁴/24 and <x⁴> = (3/2)·β²·J²)."""
    beta = tw["betx"][1]
    pred = k3l * beta ** 2 * a ** 2 / (32 * np.pi)
    return (q - tw["qx"] % 1) / pred - 1.0


DETUNING_AMPLITUDES = np.array([2e-3, 4e-3, 6e-3, 8e-3])  # √(2J): ν - qx from 5e-5 to 7e-4


def detuning_columns(tw):
    n = len(DETUNING_AMPLITUDES)
    z = np.zeros(n)
    return dict(x=DETUNING_AMPLITUDES * np.sqrt(tw["betx"][0]), px=z.copy(), y=z.copy(), py=z.copy(),
                zeta=z.copy(), delta=z.copy())


def test_octupole_detuning_through_the_tracking_oracle():
    from xline_b200 import optics

    k3l = 100.0
    line = octupole_fodo(k3l, ids=len(DETUNING_AMPLITUDES))
    tw = optics.twiss(line)
    assert min(abs(4 * tw["qx"] % 1 - r) for r in (0.0, 1.0)) >= 0.2  # qx at least 0.05 from any p/4
    mons = {}
    H.run_oracle(line.to_specs(), detuning_columns(tw), 1e9, 938.272e6, num_turns=2048, monitors=mons)
    st = list(mons.values())[0]
    x, px = (np.asarray(st[k]).reshape(2048, -1) for k in ("x", "px"))
    q, a, _ = NO.naff(x, px, tw["betx"][0], tw["alfx"][0])
    assert (q - tw["qx"] % 1).max() <= 1e-3
    assert np.abs(detuning_errors(q, a, tw, k3l)).max() <= 0.01


def test_psb_linear_tunes_through_the_tracking_oracle():
    """A small-amplitude particle of the bare PS Booster, tracked 1024 turns by the NumPy oracle:
    its NAFF tunes are the tunes of optics.twiss to 1e-10."""
    import xline_b200 as xl
    from xline_b200 import configs, optics

    line, meta = configs.load_lattice("psb")
    p0c, m0 = configs.p0c_of(meta)
    tw = optics.twiss(line)
    turns = 1024
    line.insert_element(0, xl.BeamMonitor(num_stores=turns, start=0, skip=1, min_particle_id=0,
                                          max_particle_id=0), "monitor")
    cols = dict(x=np.array([1e-5]), px=np.zeros(1), y=np.array([1e-5]), py=np.zeros(1), zeta=np.zeros(1),
                delta=np.zeros(1))
    mons = {}
    H.run_oracle(line.to_specs(), cols, p0c, m0, num_turns=turns, monitors=mons)
    st = list(mons.values())[0]
    x, px, y, py = (np.asarray(st[k]).reshape(turns, -1)[:, 0] for k in ("x", "px", "y", "py"))
    qx, _, _ = NO.naff(x, px, tw["betx"][0], tw["alfx"][0])
    qy, _, _ = NO.naff(y, py, tw["bety"][0], tw["alfy"][0])
    assert abs(qx[0] - tw["qx"] % 1) <= 1e-10
    assert abs(qy[0] - tw["qy"] % 1) <= 1e-10
    qxr, _, _ = NO.naff(x)
    assert abs(qxr[0] - tw["qx"] % 1) <= 1e-10


def test_turn_limits_match_the_header():
    from xline_b200 import _cabi, tunes

    text = open(HEADER).read()
    defs = dict(re.findall(r"#define (XLB_NAFF_\w+) (\d+)", text))
    assert int(defs["XLB_NAFF_MIN_TURNS"]) == _cabi.NAFF_MIN_TURNS == tunes.MIN_TURNS == NO.MIN_TURNS
    assert int(defs["XLB_NAFF_MAX_TURNS"]) == _cabi.NAFF_MAX_TURNS == tunes.MAX_TURNS == NO.MAX_TURNS
    assert "int xlb_naff_device(" in text
    assert "xlb_naff_device" in _cabi.EXPORTS


def test_naff_checks_arguments_before_the_device():
    """Shapes, dtypes, strides, T and (β, α) are checked first (ValueError); a CPU tensor that
    passes them is refused with RuntimeError -- there is no CPU path."""
    from xline_b200.tunes import naff

    u = torch.zeros(128, 8, dtype=torch.float64)
    for bad in (torch.zeros(63, 8, dtype=torch.float64), torch.zeros(8193, 2, dtype=torch.float64),
                u.float(), u[:, ::2], u.t().contiguous().t(), u[0]):
        with pytest.raises(ValueError):
            naff(bad)
    with pytest.raises(ValueError):
        naff(u, u[:, :4])
    with pytest.raises(ValueError):
        naff(u, torch.zeros(128, 16, dtype=torch.float64)[:, :8])  # same shape, other strides
    for beta, alpha in ((0.0, 0.0), (-1.0, 0.0), (float("nan"), 0.0), (1.0, float("inf"))):
        with pytest.raises(ValueError):
            naff(u, u, beta=beta, alpha=alpha)
    with pytest.raises(RuntimeError):
        naff(u)
    with pytest.raises(RuntimeError):
        naff(u, u, beta=2.0)


def _monitor(**kw):
    import xline_b200 as xl

    mon = xl.BeamMonitor(**dict(dict(num_stores=200, start=0, skip=1, min_particle_id=0, max_particle_id=3), **kw))
    mon.data = {k: torch.zeros(mon.num_stores, 4, dtype=torch.float64) for k in ("x", "px", "y", "py")}
    return mon


def test_monitor_tunes_refusals():
    from xline_b200.tunes import monitor_tunes

    with pytest.raises(ValueError, match="run past"):
        monitor_tunes(_monitor(), num_turns=128, windows=2)
    with pytest.raises(ValueError, match="run past"):
        monitor_tunes(_monitor(), num_turns=128, start=100)
    with pytest.raises(ValueError, match="rolling"):
        monitor_tunes(_monitor(is_rolling=True), num_turns=64)
    with pytest.raises(ValueError, match="skip"):
        monitor_tunes(_monitor(skip=2), num_turns=64)
    import xline_b200 as xl

    with pytest.raises(ValueError, match="no data"):
        monitor_tunes(xl.BeamMonitor(num_stores=100), num_turns=64)
    # windows that fit get as far as the device check
    with pytest.raises(RuntimeError):
        monitor_tunes(_monitor(), windows=2)
