"""LimitPolygon apertures on the GPU: every kernel path against the oracle, bit for bit where the
definition says so (loss flags always; coordinates in the strict kernels)."""
import numpy as np
import pytest
import torch

import xline_b200 as xl
from tests import helpers as H
from tests import polygon_cases as PC
from tests import polygon_oracle as PO
from xline_b200 import lattice

pytestmark = pytest.mark.gpu

FAST_TOL = 1e-14
COLUMNS = H.COORDS + ("rpp", "rvv", "s", "state", "at_element", "at_turn")


def _poly(xv, yv, scale=1.0):
    return xl.LimitPolygon(x_vertices=[v * scale for v in xv], y_vertices=[v * scale for v in yv])


def _line(els, **opts):
    line = xl.Line(els)
    line.polygon_apertures = True
    for k, v in opts.items():
        setattr(line, k, v)
    return line


def _track(line, cols, num_turns=1, p0c=PC.P0C, m0=PC.MASS0, **kw):
    p = xl.Particles(p0c=p0c, mass0=m0, device="cuda", **cols)
    line.track(p, num_turns=num_turns, **kw)
    torch.cuda.synchronize()
    return p.to_numpy()


def _close(a, b, tol=FAST_TOL):
    """Equal (NaN == NaN, inf == inf), or |a - b| <= tol * max(1, |b|) where both are finite: the
    coordinates here are millimetres and centimetres, so tol is absolute for them (zeta passes
    through zero), relative for s."""
    same = (a == b) | (np.isnan(a) & np.isnan(b))
    fin = np.isfinite(a) & np.isfinite(b)
    with np.errstate(invalid="ignore"):
        near = np.abs(a - b) <= tol * np.maximum(1.0, np.abs(b))
    return bool(np.all(same | (fin & near)))


def _assert_like_oracle(got, ref, strict, tol=FAST_TOL):
    for k in ("state", "at_element", "at_turn"):
        assert np.array_equal(got[k], ref[k]), k
    for k in H.COORDS + ("s",):
        if strict:
            assert np.array_equal(got[k], ref[k], equal_nan=True), k
        else:
            assert _close(got[k], ref[k], tol), k


def _assert_bitwise(a, b, keys=COLUMNS):
    for k in keys:
        assert np.array_equal(a[k], b[k], equal_nan=True), k


@pytest.mark.parametrize("strict", [False, True])
@pytest.mark.parametrize("ppt", [1, 2, 3, 4])
@pytest.mark.parametrize("name", sorted(PC.POLYGONS))
def test_polygon_matches_oracle(name, ppt, strict):
    """4 099 particles (idle lanes in the last warp) at the polygon: random points, exact
    vertices, points on the edges, NaN and +-inf; two turns through polygon -> drift -> quadrupole
    -> polygon -> DriftExact."""
    xv, yv = PC.POLYGONS[name]
    rng = np.random.default_rng(ppt + 10 * len(name))
    n = 4099
    cols = PC.mixed_beam(xv, yv, n, rng)
    line = _line([_poly(xv, yv), xl.Drift(length=1.2), xl.Multipole(knl=[0.0, 0.02]), _poly(xv, yv),
                  xl.DriftExact(length=0.7)])
    with np.errstate(all="ignore"):
        ref = PO.run_oracle(line.to_specs(), cols, PC.P0C, PC.MASS0, num_turns=2)
    got = _track(line, cols, 2, strict=strict, particles_per_thread=ppt)
    assert 0 < (ref["state"] == 0).sum() < n
    _assert_like_oracle(got, ref, strict)


@pytest.mark.parametrize("strict", [False, True])
@pytest.mark.parametrize("exact", [False, True])
def test_fused_and_unfused_polygon_drift_are_bitwise_equal(exact, strict):
    xv, yv = PC.POLYGONS["star10"]
    rng = np.random.default_rng(3)
    cols = PC.mixed_beam(xv, yv, 5000, rng)
    drift = xl.DriftExact(length=2.0) if exact else xl.Drift(length=2.0)
    els = [xl.Drift(length=1.5), _poly(xv, yv), drift, xl.Multipole(knl=[0.0, 0.01])]
    fused = _line(els)
    unfused = _line(els, fuse_records=False)
    drifts = lambda ln: sum(ln.pack(strict).record_counts.get(t, 0) for t in (lattice.T_DRIFT, lattice.T_DRIFT_EXACT))  # noqa: E731
    assert (drifts(fused), drifts(unfused)) == (1, 2)
    a = _track(fused, cols, strict=strict)
    b = _track(unfused, cols, strict=strict)
    _assert_bitwise(a, b)
    lost = a["state"] == 0
    assert lost.any() and np.all(a["at_element"][lost] == 1)
    assert np.all(a["s"][lost] == 1.5)  # s_here: the drifts before the aperture


@pytest.mark.parametrize("strict", [False, True])
def test_c2_rectangles_as_polygons_are_bitwise_the_same(strict):
    """The C2 geometry with every LimitRect replaced by its 4-vertex polygon: the two rules differ
    only on the right and top edges, which no particle of this beam hits."""
    from xline_b200 import configs

    line, cols, p0c, m0 = configs.config_lhc(20_000)
    line.merge_multipoles = False
    poly = xl.Line([_poly([e.min_x, e.max_x, e.max_x, e.min_x], [e.min_y, e.min_y, e.max_y, e.max_y])
                    if type(e).__name__ == "LimitRect" else e for e in line.elements], line.element_names)
    poly.merge_multipoles = False
    poly.polygon_apertures = True
    a = _track(line, cols, 2, p0c, m0, strict=strict)
    tally_rect = line.loss_tally.cpu().numpy()
    b = _track(poly, cols, 2, p0c, m0, strict=strict)
    _assert_bitwise(a, b)
    assert np.array_equal(tally_rect, poly.loss_tally.cpu().numpy())
    at_poly = np.array([type(e).__name__ == "LimitPolygon" for e in poly.elements])
    lost = b["state"] == 0
    assert at_poly[b["at_element"][lost]].sum() > 100  # the polygons take part


def _fodo_with_polygons(n):
    from xline_b200 import configs

    line, cols, p0c, m0 = configs.config_fodo(n)
    els = list(line.elements)
    els.insert(len(els) // 2, _poly(*PC.POLYGONS["concave_l"], scale=0.35))
    els.append(_poly(*PC.octagon((0.004, 0.0035, 0.5, 1.0))))
    return _line(els), cols, p0c, m0


@pytest.mark.parametrize("strict", [False, True])
def test_compaction_launches_equal_one_launch(strict):
    line, cols, p0c, m0 = _fodo_with_polygons(20_000)
    a = _track(line, cols, 200, p0c, m0, strict=strict, turns_per_launch=-1)
    tally = line.loss_tally.cpu().numpy()
    line.invalidate()
    b = _track(line, cols, 200, p0c, m0, strict=strict, turns_per_launch=20)
    assert line.last_stats["kernel_launches"] == 10
    # the fast kernels add s once per launch: the grouping of that sum follows the launches
    _assert_bitwise(a, b, [k for k in COLUMNS if strict or k != "s"])
    if not strict:
        assert np.allclose(a["s"], b["s"], rtol=1e-11, atol=0)
    assert np.array_equal(tally, line.loss_tally.cpu().numpy())
    lost = a["state"] == 0
    polys = [i for i, e in enumerate(line.elements) if type(e).__name__ == "LimitPolygon"]
    for i in polys:
        assert tally[i] == int((a["at_element"][lost] == i).sum()) > 0, i
    assert int(tally.sum()) == int(lost.sum())


def test_general_kernels_with_chi_column_equal_specialised_ones():
    line, cols, p0c, m0 = _fodo_with_polygons(6_000)
    a = _track(line, cols, 30, p0c, m0)
    b = _track(line, cols, 30, p0c, m0, particles_per_thread=3, threads_per_block=128, _general_kernels=True)
    _assert_bitwise(a, b)
    assert (a["state"] == 0).any()


@pytest.mark.parametrize("strict", [False, True])
def test_beam_field_kernels_with_polygons(strict):
    xv, yv = PC.POLYGONS["octagon"]
    rng = np.random.default_rng(11)
    cols = PC.mixed_beam(xv, yv, 3000, rng)
    sc = xl.SCCoasting(number_of_particles=2e11, circumference=100.0, sigma_x=4e-3, sigma_y=3e-3,
                       length=1.0, x_co=1e-4, y_co=-1e-4)
    line = _line([_poly(xv, yv), xl.Drift(length=0.8), sc, xl.Drift(length=0.5), _poly(xv, yv, 0.9)])
    with np.errstate(all="ignore"):
        ref = PO.run_oracle(line.to_specs(), cols, PC.P0C, PC.MASS0, num_turns=2)
    got = _track(line, cols, 2, strict=strict)
    assert line.pack(strict).flags & lattice.F_BEAMFIELDS
    for k in ("state", "at_element", "at_turn"):
        assert np.array_equal(got[k], ref[k]), k
    for k in H.COORDS:
        assert H.scaled_err(got[k], ref[k]) <= 1e-12, k  # the space-charge kick: libm vs CUDA exp


def test_unsplit_6d_lens_family_with_polygons():
    """The kernels that carry the 6D lens in the record loop (split_lenses = False) have the
    polygon case too: the same losses as the segmented lattice."""
    from xline_b200 import configs

    line, cols, p0c, m0 = configs.config_lhc_beambeam(2_000)
    els = [_poly(*PC.octagon((0.0006, 0.0005, 0.5, 1.0)))] + list(line.elements)
    split = _line(els)
    fused = _line(els, split_lenses=False)
    assert fused.pack().segments is None and split.pack().segments is not None
    a = _track(split, cols, 1, p0c, m0)
    b = _track(fused, cols, 1, p0c, m0, particles_per_thread=1)
    for k in ("state", "at_element", "at_turn"):
        assert np.array_equal(a[k], b[k]), k
    assert (a["at_element"][a["state"] == 0] == 0).any()


def test_polygon_kernel_shapes_agree_bitwise():
    """Every launch shape of the kernels with the polygon case gives the same bits."""
    line, cols, p0c, m0 = _fodo_with_polygons(30_000)
    ref = None
    for ppt, thr in ((3, 128), (1, 128), (1, 256), (1, 512), (2, 128), (2, 256), (4, 128)):
        cur = _track(line, cols, 20, p0c, m0, particles_per_thread=ppt, threads_per_block=thr)
        if ref is None:
            ref = cur
            assert (ref["state"] == 0).any()
            continue
        _assert_bitwise(ref, cur)


def test_trace_elem_by_elem_rows_end_at_the_polygon():
    from oracle import xline_oracle as xo

    xv, yv = PC.POLYGONS["triangle_off_origin"]
    rng = np.random.default_rng(5)
    n = 1000
    cols = PC.mixed_beam(xv, yv, n, rng)
    line = _line([xl.Drift(length=0.0), _poly(xv, yv), xl.Drift(length=1.0), xl.Multipole(knl=[0.0, 0.01])])
    for strict in (False, True):
        p = xl.Particles(p0c=PC.P0C, mass0=PC.MASS0, device="cuda", **cols)
        trace = line.trace_elem_by_elem(p, strict=strict).cpu().numpy()
        o = xo.OracleParticles(n, p0c=PC.P0C, mass0=PC.MASS0, **cols)
        for i, (name, f) in enumerate(line.to_specs()):
            with np.errstate(all="ignore"):
                PO.TRACKERS[name](o, f)
            gone = np.ones(n, dtype=bool)
            gone[o.particle_id] = False
            assert np.isnan(trace[i + 1][:, gone]).all(), i
            for fi, k in enumerate(H.COORDS):
                assert _close(trace[i + 1][fi, o.particle_id], getattr(o, k)), (i, k)
        lost_at_poly = ~np.isin(np.arange(n), o.particle_id)
        assert lost_at_poly.any() and np.isnan(trace[2:, :, lost_at_poly]).all()


def test_track_elem_by_elem_passes_the_option():
    xv, yv = PC.POLYGONS["bowtie"]
    rng = np.random.default_rng(9)
    cols = PC.mixed_beam(xv, yv, 2000, rng)
    line = _line([xl.Drift(length=0.0), xl.Multipole(knl=[0.0, 0.0]), _poly(xv, yv), xl.Drift(length=1.0)])
    p = xl.Particles(p0c=PC.P0C, mass0=PC.MASS0, device="cuda", **cols)
    out = line.track_elem_by_elem(p)
    assert len(out) == len(line) + 1
    got = p.to_numpy()
    lost = got["state"] == 0
    assert lost.any() and np.all(got["at_element"][lost] == 2) and np.all(got["at_turn"] == 0)
    with np.errstate(all="ignore"):
        ref = PO.run_oracle(line.to_specs(), cols, PC.P0C, PC.MASS0)
    assert np.array_equal(got["state"], ref["state"])
    line.polygon_apertures = False
    with pytest.raises(NotImplementedError):
        line.track_elem_by_elem(xl.Particles(p0c=PC.P0C, mass0=PC.MASS0, device="cuda", **cols))


@pytest.mark.parametrize("strict", [False, True])
def test_madx_octagon_line_refuses_by_default_and_tracks_on_request(strict):
    seq = PC.octagon_madx_sequence()
    line = xl.Line.from_madx_sequence(seq, install_apertures=True)
    assert "mqf_aperture" in line.element_names
    rng = np.random.default_rng(21)
    n = 8000
    cols = dict(x=rng.normal(0, 2.5e-3, n), px=rng.normal(0, 2e-4, n), y=rng.normal(0, 2.5e-3, n),
                py=rng.normal(0, 2e-4, n), zeta=rng.normal(0, 0.05, n), delta=rng.normal(0, 1e-4, n))
    p = xl.Particles(p0c=PC.P0C, mass0=PC.MASS0, device="cuda", **cols)
    with pytest.raises(NotImplementedError):
        line.track(p)
    line.polygon_apertures = True
    got = _track(line, cols, 3, strict=strict)
    ref = PO.run_oracle(line.to_specs(), cols, PC.P0C, PC.MASS0, num_turns=3)
    _assert_like_oracle(got, ref, strict, tol=1e-12)
    at_oct = line.element_names.index("mqf_aperture")
    assert (got["at_element"][got["state"] == 0] == at_oct).sum() > 0
