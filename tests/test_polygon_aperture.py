"""LimitPolygon apertures without a GPU: the packed record, the pack-time and C-ABI validation,
the oracle's predicate against an exact rational crossing test, the half-open boundary rule, and
packed lines with polygons interpreted against the oracle."""
import ctypes as C
import math

import numpy as np
import pytest

import xline_b200 as xl
from oracle import xline_oracle as xo
from tests import helpers as H
from tests import polygon_cases as PC
from tests import packed_interpreter as PI
from tests import polygon_oracle as PO
from xline_b200 import _cabi, lattice

ELATTICE = -3  # XLB_ELATTICE


def _poly(xv, yv):
    return xl.LimitPolygon(x_vertices=list(xv), y_vertices=list(yv))


def _polygon_record(packed):
    """(first word index, words) of the one LIMIT_POLYGON record of a packed lattice."""
    w = packed.words
    pos = 0
    while True:
        hdr = int(w[pos])
        tag, size = hdr & 0xFF, (hdr >> 16) & 0x3FFF
        if tag == lattice.T_LIMIT_POLYGON:
            return pos, w[pos: pos + 2 * size]
        assert tag not in (lattice.T_END_TURN, lattice.T_END_CHUNK), "no polygon record"
        pos += 2 * size


def _validate(packed, words=None):
    words = packed.words if words is None else words
    lat = _cabi.Lattice(words.ctypes.data, words.size, packed.chunk_words, packed.n_chunks,
                        packed.n_elements, packed.flags)
    return _cabi.lib().xlb_lattice_validate(C.byref(lat))


def _oracle_inside(xv, yv, x, y):
    return PO.inside(xv, yv, x, y)


# ---------------------------------------------------------------- the packed record
def test_record_layout_edges_slopes_path_length_and_fused_drift():
    # pentagon with a horizontal top edge, vertices listed clockwise
    xv, yv = [-1e-3, 0.5e-3, 2e-3, 1e-3, -2e-3], [2e-3, 2e-3, 0.3e-3, -1.7e-3, -0.4e-3]
    for strict in (False, True):
        line = xl.Line([xl.Drift(length=1.5), _poly(xv, yv), xl.DriftExact(length=2.25), xl.Drift(length=0.5)])
        line.polygon_apertures = True
        packed = line.pack(strict=strict)
        pos, rec = _polygon_record(packed)
        f64, i64 = rec.view(np.float64), rec.view(np.int64)
        hdr = int(rec[0])
        assert hdr >> 32 == 1  # element index
        assert (hdr >> 8) & 0xFF == lattice.AUX_DRIFT | lattice.AUX_DRIFT_EXACT
        assert i64[1] == 4 and len(rec) == 2 * (2 + 2 * 4)  # the horizontal edge is dropped
        assert f64[2] == 1.5 and f64[3] == 2.25  # s_here, the fused DriftExact
        edges = f64[4:].reshape(-1, 4)
        want = []
        for k in range(5):
            x0, y0, x1, y1 = xv[k], yv[k], xv[(k + 1) % 5], yv[(k + 1) % 5]
            if y0 == y1:
                continue
            if y1 < y0:
                x0, y0, x1, y1 = x1, y1, x0, y0
            want.append((y0, y1, x0, (x1 - x0) / (y1 - y0)))
        assert np.array_equal(edges.view(np.uint64), np.array(want).view(np.uint64))
        assert all(e[0] < e[1] for e in edges)
        assert _validate(packed) == 0
    # same words in both encodings; unfused: aux 0, drift word 0
    fast, strict = line.pack(strict=False), line.pack(strict=True)
    assert np.array_equal(_polygon_record(fast)[1], _polygon_record(strict)[1])
    line.fuse_records = False
    rec = _polygon_record(line.pack())[1]
    assert (int(rec[0]) >> 8) & 0xFF == 0 and rec.view(np.float64)[3] == 0.0


def test_madx_octagon_packs_to_six_edges():
    from xline_b200.madx_input import iter_from_madx_sequence

    seq = PC.octagon_madx_sequence()
    out = dict(iter_from_madx_sequence(seq, xl.elements.element_classes(), install_apertures=True))
    poly = out["mqf_aperture"]
    assert type(poly).__name__ == "LimitPolygon" and len(poly.x_vertices) == 8
    packed = lattice.pack_line([poly], polygons=True)
    rec = _polygon_record(packed)[1]
    assert rec.view(np.int64)[1] == 6
    assert _validate(packed) == 0


def test_polygon_apertures_off_still_refuses():
    poly = _poly(*PC.POLYGONS["octagon"])
    with pytest.raises(NotImplementedError, match="polygon_apertures"):
        lattice.pack_line([poly])
    with pytest.raises(NotImplementedError):
        lattice.pack_line([poly, xl.Drift(length=1.0)])  # the aperture -> drift peephole too
    line = xl.Line([xl.Drift(length=1.0), poly])
    assert line.polygon_apertures is False
    with pytest.raises(NotImplementedError):
        line.pack()
    with pytest.raises(NotImplementedError):
        xl.Line.from_madx_sequence(PC.octagon_madx_sequence(), install_apertures=True).pack()


@pytest.mark.parametrize("xv, yv, what", [
    ([0.0, 1.0, 0.0], [0.0, 0.0], "same length"),
    ([0.0, 1.0], [0.0, 1.0], "same length"),
    ([0.0, 1.0, float("nan")], [0.0, 0.0, 1.0], "non-finite vertex"),
    ([0.0, 1.0, 0.5], [0.0, 0.0, float("inf")], "non-finite vertex"),
    ([0.0, 1.0, 2.0, 3.0], [1.0, 1.0, 1.0, 1.0], "no edge"),
    ([-1e308, 1e308, 0.0], [0.0, 1e-300, 1.0], "non-finite slope"),
])
def test_malformed_polygons_raise_value_error(xv, yv, what):
    with pytest.raises(ValueError, match=what):
        lattice.pack_line([_poly(xv, yv)], polygons=True)


def test_validator_rejects_malformed_polygon_records():
    packed = lattice.pack_line([_poly(*PC.POLYGONS["star10"]), xl.Drift(length=1.0)], polygons=True)
    assert _validate(packed) == 0
    pos, rec = _polygon_record(packed)
    n_edges = int(rec.view(np.int64)[1])

    def broken(fn):
        w = packed.words.copy()
        fn(w)
        return _validate(packed, w)

    assert broken(lambda w: w.__setitem__(pos + 1, np.uint64(n_edges - 1))) == ELATTICE  # wrong length
    assert broken(lambda w: w.__setitem__(pos + 1, np.uint64(0))) == ELATTICE  # n_edges = 0

    def size_zero_edges(w):
        w[pos] = np.uint64((int(w[pos]) & ~(0x3FFF << 16)) | (2 << 16))
        w[pos + 1] = np.uint64(0)
    assert broken(size_zero_edges) == ELATTICE  # n_edges = 0 with a matching size
    f = packed.words.view(np.float64)
    e3 = pos + 4 + 4 * 3  # the fourth edge
    assert broken(lambda w: w.view(np.float64).__setitem__(e3 + 1, f[e3])) == ELATTICE  # y_lo == y_hi
    assert broken(lambda w: w.view(np.float64).__setitem__(e3, f[e3 + 1] + 1.0)) == ELATTICE  # y_lo > y_hi
    assert broken(lambda w: w.view(np.float64).__setitem__(e3 + 3, np.nan)) == ELATTICE  # NaN slope
    assert "polygon" in _cabi.lib().xlb_last_error().decode()


# ---------------------------------------------------------------- the predicate
@pytest.mark.parametrize("name", sorted(PC.POLYGONS))
def test_oracle_predicate_is_the_exact_crossing_test(name):
    """Away from the boundary (> 1 nm from every edge) the rounded predicate is the exact
    even-odd rule."""
    xv, yv = PC.POLYGONS[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    n = 2000 if name == "ngon600" else 20000
    x, y = PC.random_points(xv, yv, int(n * 1.02) + 50, rng)
    keep = PC.distance_to_boundary(xv, yv, x, y) > 1e-9
    x, y = x[keep][:n], y[keep][:n]
    assert len(x) == n
    got = _oracle_inside(xv, yv, x, y)
    want = PC.exact_inside(xv, yv, x, y)
    assert np.array_equal(got, want)
    assert 0.05 < got.mean() < 0.95  # both sides are sampled
    if name == "triangle_off_origin":
        assert not _oracle_inside(xv, yv, np.zeros(1), np.zeros(1))[0]
    if name == "bowtie":  # even-odd: the crossing point itself is the boundary; the lobes are inside
        assert list(_oracle_inside(xv, yv, np.array([-0.008, 0.008, 0.0, 0.0]),
                                   np.array([0.0, 0.0, 0.005, -0.005]))) == [True, True, False, False]


def test_half_open_boundary_rule():
    a = 0.01
    xv, yv = [-a, a, a, -a], [-a, -a, a, a]  # the box [-a, a]^2 as a polygon
    t = np.array([-0.75, -0.25, 0.0, 0.4, 0.9]) * a
    one = np.ones_like(t)
    cases = [  # (x, y, inside?)
        (-a * one, t, True),    # left edge
        (a * one, t, False),    # right edge
        (t, -a * one, True),    # bottom edge
        (t, a * one, False),    # top edge
        (np.array([-a]), np.array([-a]), True),  # lower left vertex: on the left and bottom edges
        (np.array([a, a, -a]), np.array([-a, a, a]), False),  # the other three vertices
        (np.array([np.nan, 0.0, np.inf, -np.inf, 0.0, 0.0]), np.array([0.0, np.nan, 0.0, 0.0, np.inf, -np.inf]), False),
    ]
    line = xl.Line([_poly(xv, yv)])
    line.polygon_apertures = True
    for x, y, inside in cases:
        assert np.all(_oracle_inside(xv, yv, x, y) == inside), (x, y)
        for strict in (True, False):
            res = PI.track(line.pack(strict=strict), dict(x=x, y=y), PC.P0C, PC.MASS0)
            assert np.all((res["state"] == 1) == inside), (x, y, strict)
    # LimitRect is inclusive on all four sides: the two differ on the right and top edges only
    rect = xo.OracleParticles(2, p0c=PC.P0C, mass0=PC.MASS0, x=np.array([a, 0.0]), y=np.array([0.0, a]))
    xo.track_limit_rect(rect, dict(min_x=-a, max_x=a, min_y=-a, max_y=a))
    assert len(rect) == 2


@pytest.mark.parametrize("name", sorted(PC.POLYGONS))
def test_interpreter_and_oracle_agree_on_boundary_points(name):
    xv, yv = PC.POLYGONS[name]
    rng = np.random.default_rng(7)
    cols = PC.mixed_beam(xv, yv, 3000, rng)
    ref = _oracle_inside(xv, yv, cols["x"], cols["y"])
    line = xl.Line([_poly(xv, yv)])
    line.polygon_apertures = True
    for strict in (True, False):
        res = PI.track(line.pack(strict=strict), cols, PC.P0C, PC.MASS0)
        assert np.array_equal(res["state"] == 1, ref)
    assert not ref[~np.isfinite(cols["x"]) | ~np.isfinite(cols["y"])].any()


# ---------------------------------------------------------------- lines with polygons
@pytest.mark.parametrize("seed", range(12))
def test_random_polygon_lines_strict_bitwise_and_fast_close(seed):
    rng = np.random.default_rng(5000 + seed)
    line = PC.random_polygon_line(rng)
    line.chunk_words = int(rng.choice([64, 256, 2048]))
    n = 400
    cols = dict(x=rng.normal(0, 1.2e-3, n), px=rng.normal(0, 1e-4, n), y=rng.normal(0, 1.2e-3, n),
                py=rng.normal(0, 1e-4, n), zeta=rng.normal(0, 0.05, n), delta=rng.normal(0, 3e-4, n))
    with np.errstate(all="ignore"):
        ref = PO.run_oracle(line.to_specs(), cols, PC.P0C, PC.MASS0, num_turns=3)
        strict = PI.track(line.pack(strict=True), cols, PC.P0C, PC.MASS0, num_turns=3)
        fast = PI.track(line.pack(strict=False), cols, PC.P0C, PC.MASS0, num_turns=3)
    assert (ref["state"] == 0).any()
    polys = {i for i, e in enumerate(line.elements) if type(e).__name__ == "LimitPolygon"}
    assert set(ref["at_element"][ref["state"] == 0]) & polys, "some losses at the polygons"
    for k in ("state", "at_element", "at_turn"):
        assert np.array_equal(strict[k], ref[k]), k
        assert np.array_equal(fast[k], ref[k]), k
    for k in H.COORDS:
        assert np.array_equal(strict[k], ref[k], equal_nan=True), k
        assert H.scaled_err(fast[k], ref[k]) <= 1e-10, k


def test_toggling_polygon_apertures_repacks():
    line = xl.Line([xl.Drift(length=1.0), _poly(*PC.POLYGONS["concave_l"]), xl.Drift(length=1.0)])
    with pytest.raises(NotImplementedError):
        line.pack()
    line.polygon_apertures = True
    first = line.pack()
    assert first.record_counts.get(lattice.T_LIMIT_POLYGON) == 1
    assert line.pack() is first  # cached
    line.polygon_apertures = False
    with pytest.raises(NotImplementedError):
        line.pack()
    line.polygon_apertures = True
    again = line.pack()
    assert again is not first and np.array_equal(again.words, first.words)


def test_algorithmic_ops_count_six_per_stored_edge():
    line = xl.Line([_poly(*PC.octagon()), _poly(*PC.POLYGONS["ngon600"]), xl.LimitRect()])
    assert line.algorithmic_ops_per_turn() == 6 * 6 + 6 * 600 + 4
    assert PO.algorithmic_ops(line.to_specs()) == line.algorithmic_ops_per_turn()


def test_octagon_vertices_follow_the_madx_angles():
    xv, yv = PC.octagon((0.02, 0.018, 0.5, 1.0))
    assert xv[0] == 0.02 and yv[0] == 0.02 * math.tan(0.5) and yv[1] == 0.018
