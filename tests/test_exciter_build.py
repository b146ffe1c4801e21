"""What the compiler made of the twins that carry the EXCITER case (CPU-only, from `ptxas -v` of the
in-tree build): no spill where the twin had none before the case existed, and the figures DESIGN.md
records for the one-species thin-lens twins."""
import re

import pytest

from tests.test_build_artifacts import _ptxas

TWINS = ("track_kernel_polygons", "track_kernel_radiation")
UNITS = ("track_fast", "track_fast_nc", "track_fast_nc_lo", "track_fast_bf", "track_fast_bf_nc_lo", "track_fast_bf6")
# (unit, twin, particles per thread, threads, min blocks, trace) that spilled before the EXCITER case
SPILLED_BEFORE = {
    ("track_fast", "track_kernel_polygons", 1, 256, 3, 0), ("track_fast", "track_kernel_polygons", 1, 512, 2, 0),
    ("track_fast_bf", "track_kernel_polygons", 3, 128, 3, 0),
    ("track_fast_bf6", "track_kernel_polygons", 1, 256, 2, 0), ("track_fast_bf6", "track_kernel_polygons", 2, 256, 2, 0),
    ("track_fast_bf6", "track_kernel_polygons", 3, 128, 3, 0),
    ("track_fast_bf_nc_lo", "track_kernel_polygons", 3, 128, 3, 0),
    ("track_fast_bf_nc_lo", "track_kernel_polygons", 4, 128, 3, 0),
    ("track_fast_nc", "track_kernel_polygons", 1, 256, 3, 0), ("track_fast_nc", "track_kernel_polygons", 1, 512, 2, 0),
    ("track_fast_nc", "track_kernel_polygons", 4, 128, 3, 0),
    ("track_fast_nc", "track_kernel_radiation", 1, 128, 5, 0), ("track_fast_nc", "track_kernel_radiation", 1, 256, 3, 0),
    ("track_fast_nc", "track_kernel_radiation", 1, 512, 2, 0), ("track_fast_nc", "track_kernel_radiation", 2, 256, 2, 0),
    ("track_fast_nc", "track_kernel_radiation", 4, 128, 3, 0),
    ("track_fast_nc_lo", "track_kernel_polygons", 3, 128, 4, 0), ("track_fast_nc_lo", "track_kernel_polygons", 4, 128, 3, 0),
    ("track_fast_nc_lo", "track_kernel_radiation", 1, 128, 5, 0),
    ("track_fast_nc_lo", "track_kernel_radiation", 3, 128, 4, 0),
    ("track_fast_nc_lo", "track_kernel_radiation", 4, 128, 3, 0),
}
# DESIGN.md §4.9: spill stores of the one-species thin-lens twins in the tightest shapes, and registers
RECORDED = {
    ("track_fast_nc", "track_kernel_polygons", 4, 128, 3, 0): dict(spill_st=52, regs=168),
    ("track_fast_nc", "track_kernel_polygons", 1, 512, 2, 0): dict(spill_st=232, regs=64),
    ("track_fast_nc", "track_kernel_radiation", 4, 128, 3, 0): dict(spill_st=132, regs=168),
    ("track_fast_nc", "track_kernel_radiation", 1, 512, 2, 0): dict(spill_st=512, regs=64),
}


def _twins(unit):
    out = {}
    for name, k in _ptxas(unit).items():
        m = re.search(r"(track_kernel_\w+?)ILi(\d+)ELi(\d+)ELi(\d+)ELb(\d)E", name)
        if m and m.group(1) in TWINS:
            out[(unit, m.group(1)) + tuple(int(v) for v in m.groups()[1:])] = k
    return out


@pytest.mark.parametrize("unit", UNITS)
def test_twins_spill_nowhere_new(unit):
    twins = _twins(unit)
    assert twins
    for key, k in twins.items():
        if key not in SPILLED_BEFORE:
            assert k["spill_st"] == 0 and k["spill_ld"] == 0 and k["stack"] <= 48, (key, k)


def test_recorded_figures_hold():
    twins = _twins("track_fast_nc")
    for key, want in RECORDED.items():
        assert twins[key]["spill_st"] <= want["spill_st"], (key, twins[key])
        assert twins[key]["regs"] <= want["regs"], (key, twins[key])
