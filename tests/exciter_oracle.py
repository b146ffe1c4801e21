"""TEST INFRASTRUCTURE -- the CPU oracle of ``Exciter`` and a ``Line.track`` loop over the oracle's
element maps (``oracle/xline_oracle.py``, with ``LimitPolygon`` from ``tests/polygon_oracle.py``) that
includes it.

The map is the project's own (include/xline_b200.h, DESIGN.md §4.11), restated here from the element's
fields: the sample index with the header's roundings in NumPy float64 (NumPy never fuses a multiply-add),
the kick as the reference's multipole polynomial (xline/elements.py:120-136) times the sample.  Nothing
is shared with the product package.
"""
import numpy as np
from scipy.constants import c as clight

from oracle import xline_oracle as xo
from tests import polygon_oracle as PO
from tests import radiation_oracle as RO


def sample_index(f, at_turn, zeta, beta0):
    """The sample each particle reads, -1 for none: t = T - start_turn as float64,
    u = t*A - (zeta*B)/beta0 with A = fs/frev, B = fs/c, v = floor(u + 0.5), in range iff
    0 <= v < len(samples) (never for a NaN or infinite zeta)."""
    fs, frev = float(f["sampling_frequency"]), float(f["frev"])
    a, b = fs / frev, fs / clight
    n = len(np.atleast_1d(np.asarray(f["samples"], dtype=np.float64))) if len(f["samples"]) else 0
    t = (np.asarray(at_turn, dtype=np.int64) - np.int64(int(f["start_turn"]))).astype(np.float64)
    with np.errstate(invalid="ignore"):
        v = np.floor((t * a - (np.asarray(zeta, dtype=np.float64) * b) / beta0) + 0.5)
        ok = (v >= 0) & (v < n)
    return np.where(ok, v, -1.0).astype(np.int64)


def polynomial(f, x, y):
    """(Px, Py): the reference's Horner loop of knl/ksl with its division by ii at every step."""
    knl_in, ksl_in = list(f.get("knl", [0])), list(f.get("ksl", [0]))
    order = max(len(knl_in), len(ksl_in)) - 1
    knl = np.concatenate([np.asarray(knl_in, dtype=np.float64), np.zeros(order + 1 - len(knl_in))])
    ksl = np.concatenate([np.asarray(ksl_in, dtype=np.float64), np.zeros(order + 1 - len(ksl_in))])
    dpx, dpy = knl[order] * np.ones_like(x), ksl[order] * np.ones_like(x)
    for ii in range(order, 0, -1):
        zre = (dpx * x - dpy * y) / ii
        zim = (dpx * y + dpy * x) / ii
        dpx = knl[ii - 1] + zre
        dpy = ksl[ii - 1] + zim
    return dpx, dpy


def sample_values(f, idx):
    samples = np.asarray(f["samples"], dtype=np.float64).reshape(-1)
    if len(samples) == 0:
        return np.zeros(len(idx))
    return np.where(idx >= 0, samples[np.maximum(idx, 0)], 0.0)


def track_exciter(p, f):
    s = sample_values(f, sample_index(f, p.at_turn, p.zeta, p.beta0))
    dpx, dpy = polynomial(f, p.x, p.y)
    p.px = p.px + (-p.chi * (s * dpx))
    p.py = p.py + p.chi * (s * dpy)


TRACKERS = dict(PO.TRACKERS, Exciter=track_exciter)


def line_track(specs, p, num_turns=1, radiation=None, seed=0):
    """``xline_oracle.line_track`` (no monitors) with Exciter and LimitPolygon among the element maps;
    ``p.at_turn`` counts the turns, as the exciter's waveform does.  ``radiation`` ("mean" or
    "quantum"): every Multipole of length > 0 radiates through ``tests/radiation_oracle.py``."""
    for _ in range(num_turns):
        if len(p) == 0:
            break
        for iel, (name, f) in enumerate(specs):
            if name == "BeamMonitor":
                continue
            if radiation is not None and RO.radiates(name, f):
                RO.track_multipole_rad(p, f, radiation, seed, iel)
                continue
            rec = TRACKERS[name](p, f)
            if rec is not None:
                rec["at_element"][:] = iel
                rec["state"][:] = 0
                if len(p) == 0:
                    break
        p.at_turn = p.at_turn + 1
    return p


def run_oracle(specs, cols, p0c, mass0, num_turns=1, radiation=None, seed=0):
    """Full-length result columns by particle id (``tests/helpers.run_oracle`` for these lines)."""
    n = len(cols["x"])
    p = xo.OracleParticles(n, p0c=p0c, mass0=mass0, **cols)
    line_track(specs, p, num_turns=num_turns, radiation=radiation, seed=seed)
    return xo.gather_full(p, n)


def algorithmic_ops(specs):
    """``polygon_oracle.algorithmic_ops`` plus, per Exciter, a straight multipole of its order and 8
    (the sample index: two products, a quotient, a difference, the half and the floor; the two
    scalings by the sample)."""
    total = PO.algorithmic_ops([s for s in specs if s[0] != "Exciter"])
    for name, f in specs:
        if name == "Exciter":
            order = max(len(f.get("knl", [0])), len(f.get("ksl", [0]))) - 1
            total += 10 * order + 4 + 8
    return total
