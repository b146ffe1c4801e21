"""Shared helpers for the parity tests (golden fixtures, oracle drivers)."""
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
COORDS = ("x", "px", "y", "py", "zeta", "delta")


def manifest():
    with open(os.path.join(GOLDEN, "manifest.json")) as fh:
        return json.load(fh)


def load_case(case):
    m = manifest()[case]
    data = dict(np.load(os.path.join(GOLDEN, ("element_%s.npz" % case) if m["type"] != "Line"
                                     else "%s.npz" % case)))
    cols = {k[3:]: v for k, v in data.items() if k.startswith("in_")}
    out = {k[4:]: v for k, v in data.items() if k.startswith("out_")}
    if m["type"] == "Line":
        specs = [(n, f) for n, f in m["elements"]]
    else:
        specs = [(m["type"], m["fields"])]
    return m, specs, cols, out


def run_oracle(specs, cols, p0c, mass0, num_turns=1, monitors=None):
    from oracle import xline_oracle as xo

    n = len(cols["x"])
    p = xo.OracleParticles(n, p0c=p0c, mass0=mass0, **cols)
    xo.line_track(specs, p, num_turns=num_turns, monitors=monitors)
    return xo.gather_full(p, n)


def rel_err(a, b):
    """max |a-b| / max(|a|,|b|), 0 where both are 0 -- the 1e-12 metric of north_star."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    den = np.maximum(np.abs(a), np.abs(b))
    with np.errstate(invalid="ignore", divide="ignore"):
        r = np.where(den > 0, np.abs(a - b) / den, 0.0)
    both_nan = np.isnan(a) & np.isnan(b)
    r = np.where(both_nan, 0.0, r)
    return float(np.max(r)) if r.size else 0.0


def _finite_pairs(a, b):
    """The mask of entries finite on both sides, or None when the two finite masks differ."""
    fa, fb = np.broadcast_arrays(np.isfinite(a), np.isfinite(b))
    if not np.array_equal(fa, fb):
        return None
    return fa


def scaled_err(a, b):
    """max |a-b| / rms(b): error relative to the beam scale of the coordinate.  Entries that are
    non-finite on both sides are skipped; an entry non-finite on one side only is an infinite
    error."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    ok = _finite_pairs(a, b)
    if ok is None:
        return float("inf")
    a, b = np.broadcast_arrays(a, b)
    if not ok.any():
        return 0.0
    scale = np.sqrt(np.mean(b[ok] ** 2))
    if scale == 0:
        return float(np.max(np.abs(a[ok] - b[ok])))
    return float(np.max(np.abs(a[ok] - b[ok])) / scale)


def floor_rel_err(a, b, floor=1e-3):
    """max |a-b| / max(|a|, |b|, floor * rms(b)): elementwise relative error with the
    denominator floored at ``floor`` x the beam's r.m.s. of that coordinate, so that values
    passing through zero are judged against the coordinate's scale, not against themselves.
    Non-finite entries as in ``scaled_err``."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    ok = _finite_pairs(a, b)
    if ok is None:
        return float("inf")
    a, b = np.broadcast_arrays(a, b)
    if not ok.any():
        return 0.0
    rms = np.sqrt(np.mean(b[ok] ** 2))
    den = np.maximum(np.maximum(np.abs(a[ok]), np.abs(b[ok])), floor * rms)
    den = np.where(den > 0, den, 1.0)
    return float(np.max(np.abs(a[ok] - b[ok]) / den))
