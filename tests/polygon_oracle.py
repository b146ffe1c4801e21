"""TEST INFRASTRUCTURE -- the CPU oracle of ``LimitPolygon`` and a ``Line.track`` loop over the
oracle's element maps (``oracle/xline_oracle.py``) that includes it.

The reference's ``LimitPolygon.track`` raises ``NotImplementedError`` (xline/elements.py:483), so
nothing there pins this map: it is the project's own definition (include/xline_b200.h,
DESIGN.md §4.5), restated here from the element's vertex lists.  Nothing is shared with the
product package.
"""
import numpy as np

from oracle import xline_oracle as xo


def track_limit_polygon(p, f):
    """Even-odd rule over the closed polygon V_0 .. V_(n-1); an edge with distinct end ordinates,
    taken from its lower end (x0, y0) to (x1, y1), is crossed by the particle at (x, y) when
    y0 <= y < y1 and x < x0 + (y - y0) * ((x1 - x0) / (y1 - y0)), each operation rounded once
    (NumPy never fuses a multiply-add).  NaN and inf coordinates cross an even number of edges
    and are lost."""
    xv = np.asarray(f["x_vertices"], dtype=np.float64)
    yv = np.asarray(f["y_vertices"], dtype=np.float64)
    x, y = p.x, p.y
    inside = np.zeros(len(x), dtype=bool)
    for k in range(len(xv)):
        xa, ya, xb, yb = xv[k], yv[k], xv[(k + 1) % len(xv)], yv[(k + 1) % len(xv)]
        if ya == yb:
            continue
        if yb < ya:
            xa, ya, xb, yb = xb, yb, xa, ya
        slope = (xb - xa) / (yb - ya)
        with np.errstate(invalid="ignore"):  # inf * 0 for an infinite y at a vertical edge
            inside ^= (y >= ya) & (y < yb) & (x < xa + (y - ya) * slope)
    p.state = np.int64(1) * inside
    return p.remove_lost_particles()


TRACKERS = dict(xo.TRACKERS, LimitPolygon=track_limit_polygon)


def line_track(specs, p, num_turns=1):
    """``xline_oracle.line_track`` (no monitors) with LimitPolygon among the element maps."""
    for _ in range(num_turns):
        if len(p) == 0:
            break
        for iel, (name, f) in enumerate(specs):
            if name == "BeamMonitor":
                continue
            rec = TRACKERS[name](p, f)
            if rec is not None:
                rec["at_element"][:] = iel
                rec["state"][:] = 0
                if len(p) == 0:
                    break
        p.at_turn = p.at_turn + 1
    return p


def run_oracle(specs, cols, p0c, mass0, num_turns=1):
    """``tests/helpers.run_oracle`` for lines with polygons: full-length columns by particle id."""
    n = len(cols["x"])
    p = xo.OracleParticles(n, p0c=p0c, mass0=mass0, **cols)
    line_track(specs, p, num_turns=num_turns)
    return xo.gather_full(p, n)


def inside(x_vertices, y_vertices, x, y):
    """The predicate alone: which of the points (x, y) are inside."""
    p = xo.OracleParticles(len(x), x=x, y=y)
    track_limit_polygon(p, {"x_vertices": list(x_vertices), "y_vertices": list(y_vertices)})
    return xo.gather_full(p, len(x))["state"] == 1


def algorithmic_ops(specs):
    """``xline_oracle.algorithmic_ops`` plus 6 per stored polygon edge (two compares for the y slab,
    sub, mul, add, one compare)."""
    total = xo.algorithmic_ops([s for s in specs if s[0] != "LimitPolygon"])
    for name, f in specs:
        if name == "LimitPolygon":
            yv = list(f["y_vertices"])
            total += 6 * sum(1 for k in range(len(yv)) if yv[k] != yv[(k + 1) % len(yv)])
    return total
