"""Tangent map without a GPU: the NumPy statement of the recursion (tests/tangent_oracle.py)
against Richardson-extrapolated central differences of the packed interpreter's element maps, exact
closed forms, the header constants and the argument checks of the C entry point."""
import math
import os
import re

import numpy as np
import pytest

from tests import tangent_oracle as TO
import xline_b200 as xl
from xline_b200 import _cabi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("case", TO.element_cases(), ids=lambda c: c[0])
def test_oracle_jacobian_matches_finite_differences(case):
    name, el, p0c, z = case
    J = TO.oracle_jacobian(el, z, p0c)
    fd = TO.fd_jacobian(TO.pack_one(el), z, p0c)
    # per column: the error of a Richardson-extrapolated difference is relative to the column's size
    scale = np.maximum(np.max(np.abs(J), axis=0), 1e-300)
    err = np.max(np.abs(J - fd) / scale)
    assert err <= 1e-8, (name, err, J, fd)


def _one(el, z, p0c=TO.P0C):
    return TO.oracle_jacobian(el, np.asarray(z, dtype=float), p0c)


def test_closed_forms():
    z = np.array([1e-3, 2e-4, -1e-3, 1e-4, 0.0, 0.0])
    J = _one(xl.Drift(length=3.0), z)
    ref = np.eye(6)
    ref[0, 1] = ref[2, 3] = 3.0
    ref[0, 5], ref[2, 5] = -2e-4 * 3.0, -1e-4 * 3.0
    ref[4, 1], ref[4, 3] = -3.0 * 2e-4, -3.0 * 1e-4
    rv1 = TO.MASS0 ** 2 / (TO.P0C ** 2 + TO.MASS0 ** 2)  # d rvv / d delta at delta = 0: 1 - beta0^2
    ref[4, 5] = 3.0 * (rv1 + 5e-8)
    assert np.allclose(J, ref, rtol=1e-12, atol=1e-15)  # 1 - beta0^2 of the LHC carries ~1e-8 relative rounding
    J = _one(xl.Multipole(knl=[0.0, 0.02]), z)
    ref = np.eye(6)
    ref[1, 0], ref[3, 2] = -0.02, 0.02
    assert np.array_equal(J, ref)
    J = _one(xl.SRotation(angle=30.0), z)
    c, s = math.cos(math.radians(30.0)), math.sin(math.radians(30.0))
    ref = np.eye(6)
    ref[0, 0] = ref[1, 1] = ref[2, 2] = ref[3, 3] = c
    ref[0, 2] = ref[1, 3] = s
    ref[2, 0] = ref[3, 1] = -s
    assert np.allclose(J, ref, rtol=0, atol=2e-16)
    el = xl.DipoleEdge(h=0.05, e1=0.1, hgap=0.03, fint=0.5)
    J = _one(el, z)
    corr = 2 * el.h * el.hgap * el.fint
    ref = np.eye(6)
    ref[1, 0] = el.h * np.tan(el.e1)
    ref[3, 2] = -el.h * np.tan(el.e1 - corr / np.cos(el.e1) * (1 + np.sin(el.e1) ** 2))
    assert np.array_equal(J, ref)


def test_header_constants_and_binding():
    text = open(os.path.join(ROOT, "include", "xline_b200.h")).read()
    assert int(re.search(r"#define XLB_TANGENT_SCALE_LOG2 (\d+)", text).group(1)) == _cabi.TANGENT_SCALE_LOG2
    assert int(re.search(r"#define XLB_TANGENT_MAX_THREADS (\d+)", text).group(1)) == _cabi.TANGENT_MAX_THREADS
    assert "int xlb_track_tangent_device(" in text
    assert "xlb_track_tangent_device" in _cabi.EXPORTS
    assert int(re.search(r"#define XLB_ABI_VERSION (\d+)", text).group(1)) == 4


def test_tangent_map_container():
    t = xl.TangentMap(3, "cpu")
    assert t.jacobian.shape == (3, 6, 6)
    assert np.array_equal(t.jacobian[1].numpy(), np.eye(6))
    assert np.allclose(t.fli.numpy(), math.log10(math.sqrt(6)))
    assert np.allclose(t.lyapunov(10).numpy(), math.log(math.sqrt(6)) / 10)
    t.log2_scale[0] = 600
    m = t.matrix()
    assert float(m[0, 0, 0]) == 2.0 ** 600 and float(m[1, 0, 0]) == 1.0
    t.log2_scale[0] = 2000
    assert math.isinf(float(t.matrix()[0, 0, 0]))


def test_closed_orbit_argument_checks():
    line = xl.Line([xl.Drift(length=1.0)])
    p = xl.Particles(p0c=1e9, x=[0.0], device="cpu")
    with pytest.raises(ValueError):
        xl.closed_orbit(line, p, mode="5d")
    with pytest.raises(ValueError):
        xl.closed_orbit(line, p, mode="6d")  # no RF


def test_packing_is_one_record_per_element():
    from xline_b200.lattice import pack_line

    els = [xl.Multipole(knl=[0, 0.01]), xl.LimitRect(min_x=-1, max_x=1, min_y=-1, max_y=1), xl.Drift(length=1.0),
           xl.Multipole(knl=[0, -0.01]), xl.Drift(length=0.0)]
    packed = pack_line(els, strict=False, fuse=False, merge=False, split_lenses=False, drop_noops=False)
    words = packed.words.view(np.uint64)
    tags, w = [], 0
    while True:
        hdr = int(words[w])
        if hdr & 0xFF in (0, 1):
            break
        tags.append(hdr & 0xFF)
        w += 2 * ((hdr >> 16) & 0x3FFF)
    assert tags == [4, 11, 2, 4, 2] and all(t < 0x80 for t in tags)
