"""Polygons, beams and lines shared by the LimitPolygon tests (CPU and GPU)."""
import math
from fractions import Fraction

import numpy as np

P0C, MASS0 = 26e9, 938.27208816e6


def octagon(ap=(0.02, 0.018, 0.5, 1.0)):
    """The vertex lists of the MAD-X ``octagon`` mapping (xline/loader_mad.py:229-242) for
    ``aperture = [x-half-width, y-half-width, angle 1, angle 2]``."""
    v1 = (ap[0], ap[0] * math.tan(ap[2]))
    v2 = (ap[1] / math.tan(ap[3]), ap[1])
    return ([v1[0], v2[0], -v2[0], -v1[0], -v1[0], -v2[0], v2[0], v1[0]],
            [v1[1], v2[1], v2[1], v1[1], -v1[1], -v2[1], -v2[1], -v1[1]])


def _star(tips=10, r_out=0.02, r_in=0.008):
    th = np.arange(2 * tips) * (math.pi / tips) + 0.1
    r = np.where(np.arange(2 * tips) % 2 == 0, r_out, r_in)
    return (r * np.cos(th)).tolist(), (r * np.sin(th)).tolist()


def _ngon600():
    rng = np.random.default_rng(600)
    th = np.arange(600) * (2 * math.pi / 600)
    r = 0.015 * (1 + 0.15 * np.sin(7 * th)) * (1 + 0.02 * rng.uniform(-1, 1, 600))
    return (r * np.cos(th)).tolist(), (r * np.sin(th)).tolist()


POLYGONS = {
    "octagon": octagon(),
    # concave L, corner at the lower left
    "concave_l": ([-0.01, 0.012, 0.012, 0.002, 0.002, -0.01], [-0.01, -0.01, 0.0, 0.0, 0.015, 0.015]),
    "star10": _star(),
    # self-intersecting: even-odd gives the two triangles that touch at the origin
    "bowtie": ([-0.01, 0.01, 0.01, -0.01], [-0.008, 0.008, -0.008, 0.008]),
    "triangle_off_origin": ([0.004, 0.02, 0.009], [0.003, 0.006, 0.018]),
    "ngon600": _ngon600(),
}


def _segments(xv, yv):
    xv, yv = np.asarray(xv), np.asarray(yv)
    return xv, yv, np.roll(xv, -1), np.roll(yv, -1)


def distance_to_boundary(xv, yv, x, y):
    """Smallest distance from each point to the polygon's edges (float64, an estimate)."""
    x0, y0, x1, y1 = _segments(xv, yv)
    dx, dy = x1 - x0, y1 - y0
    best = np.full(len(x), np.inf)
    for k in range(len(x0)):
        t = np.clip(((x - x0[k]) * dx[k] + (y - y0[k]) * dy[k]) / (dx[k] ** 2 + dy[k] ** 2), 0.0, 1.0)
        best = np.minimum(best, np.hypot(x - (x0[k] + t * dx[k]), y - (y0[k] + t * dy[k])))
    return best


def exact_inside(xv, yv, x, y):
    """The even-odd crossing test of the definition in exact rational arithmetic (the edges'
    slopes unrounded): reference for points that are not within rounding of an edge."""
    x0, y0, x1, y1 = _segments(xv, yv)
    out = np.zeros(len(x), dtype=bool)
    for i in range(len(x)):
        px, py = Fraction(float(x[i])), Fraction(float(y[i]))
        odd = False
        for k in range(len(x0)):
            ya, yb, xa, xb = y0[k], y1[k], x0[k], x1[k]
            if ya == yb:
                continue
            if yb < ya:
                xa, ya, xb, yb = xb, yb, xa, ya
            if not (ya <= y[i] < yb):  # float comparisons are exact
                continue
            # x < xa + (y - ya) (xb - xa) / (yb - ya), times yb - ya > 0
            fa, fya = Fraction(float(xa)), Fraction(float(ya))
            if (px - fa) * (Fraction(float(yb)) - fya) < (py - fya) * (Fraction(float(xb)) - fa):
                odd = not odd
        out[i] = odd
    return out


def random_points(xv, yv, n, rng, margin=0.2):
    xv, yv = np.asarray(xv), np.asarray(yv)
    wx, wy = np.ptp(xv), np.ptp(yv)
    x = rng.uniform(xv.min() - margin * wx, xv.max() + margin * wx, n)
    y = rng.uniform(yv.min() - margin * wy, yv.max() + margin * wy, n)
    return x, y


def boundary_points(xv, yv, rng, per_edge=8):
    """Exact vertices and points on the edges (rounded onto the float grid, so on either side)."""
    x0, y0, x1, y1 = _segments(xv, yv)
    xs, ys = [np.asarray(xv, dtype=float)], [np.asarray(yv, dtype=float)]
    for k in range(len(x0)):
        t = rng.uniform(0, 1, per_edge)
        xs.append(x0[k] + t * (x1[k] - x0[k]))
        ys.append(y0[k] + t * (y1[k] - y0[k]))
        if y0[k] == y1[k]:  # horizontal: exactly on it
            ys[-1] = np.full(per_edge, y0[k])
        if x0[k] == x1[k]:  # vertical: exactly on it
            xs[-1] = np.full(per_edge, x0[k])
    return np.concatenate(xs), np.concatenate(ys)


def mixed_beam(xv, yv, n, rng):
    """``n`` particles at the aperture: random points, exact vertices, boundary points, NaN and
    +-inf in either coordinate; small momenta so that a following drift moves them a little."""
    bx, by = boundary_points(xv, yv, rng)
    special = np.array([np.nan, np.inf, -np.inf, 0.0])
    sx = np.concatenate([special, np.zeros(4), special[:3], special[:3]])
    sy = np.concatenate([np.zeros(4), special, special[:3], special[::-1][:3]])
    rx, ry = random_points(xv, yv, n, rng)
    x = np.concatenate([bx, sx, rx])[:n]
    y = np.concatenate([by, sy, ry])[:n]
    perm = rng.permutation(n)
    return dict(x=x[perm], y=y[perm], px=rng.normal(0, 1e-5, n), py=rng.normal(0, 1e-5, n),
                zeta=rng.normal(0, 0.05, n), delta=rng.normal(0, 1e-4, n))


def random_polygon_line(rng, polygons=POLYGONS):
    """A random thin-lens line with polygon apertures among the other elements: polygon -> drift
    (fused) and polygon -> DriftExact, polygons next to multipoles, boxes and shifts."""
    import xline_b200 as xl

    names = sorted(polygons)
    els = []
    for _ in range(int(rng.integers(6, 20))):
        u = rng.random()
        if u < 0.35:
            xv, yv = polygons[names[int(rng.integers(len(names)))]]
            s = float(rng.choice([0.15, 0.2, 0.3]))  # the polygons span ~ 2-4 cm: scale to mm
            els.append(xl.LimitPolygon(x_vertices=[v * s for v in xv], y_vertices=[v * s for v in yv]))
            if rng.random() < 0.6:
                L = float(rng.choice([0.3, 1.1]))
                els.append(xl.DriftExact(length=L) if rng.random() < 0.4 else xl.Drift(length=L))
        elif u < 0.6:
            els.append(xl.Multipole(knl=[0.0, rng.normal(0, 0.05), rng.normal(0, 0.5)],
                                    ksl=[0.0, rng.normal(0, 0.02)]))
            if rng.random() < 0.3:
                els.append(xl.LimitRect(min_x=-3e-3, max_x=3e-3, min_y=-2.5e-3, max_y=2.5e-3))
            els.append(xl.Drift(length=float(rng.choice([0.5, 1.5]))))
        elif u < 0.8:
            els.append(xl.XYShift(dx=rng.normal(0, 2e-4), dy=rng.normal(0, 2e-4)))
        else:
            els.append(xl.SRotation(angle=rng.normal(0, 10)))
    if not any(type(e).__name__ == "LimitPolygon" for e in els):
        xv, yv = polygons["octagon"]
        els.append(xl.LimitPolygon(x_vertices=[v * 0.15 for v in xv], y_vertices=[v * 0.15 for v in yv]))
    line = xl.Line(els)
    line.polygon_apertures = True
    return line


def octagon_madx_sequence():
    """A thin MAD-X sequence whose quadrupole carries an octagon aperture."""
    from types import SimpleNamespace

    from xline_b200.madx_input import MadElement, MadSequence

    els = [
        MadElement("mqf", "multipole", dict(knl=[0.0, 2e-2], ksl=[0.0, 0.0], lrad=0.5, apertype="octagon",
                                            aperture=[0.004, 0.0035, 0.5, 1.0]), 1.0),
        MadElement("mqd", "multipole", dict(knl=[0.0, -2e-2], ksl=[0.0, 0.0], lrad=0.5, apertype="rectangle",
                                            aperture=[0.01, 0.01]), 4.0),
    ]
    return MadSequence("oct", 6.0, els, SimpleNamespace(pc=26.0))
