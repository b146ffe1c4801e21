"""Exciter without a GPU: the element, the packed record and its data region, pack-time and C-ABI
validation, the refusals, and packed lines with exciters interpreted against the exciter oracle."""
import copy
import ctypes as C
import hashlib
import math

import numpy as np
import pytest
import torch
from scipy.constants import c as clight

import xline_b200 as xl
from oracle import xline_oracle as xo
from tests import exciter_oracle as EO
from tests import exciter_interpreter as EI
from xline_b200 import _cabi, configs, lattice

ELATTICE = -3  # XLB_ELATTICE
P0C, M0 = 450e9, xo.PROTON_MASS_EV


def _validate(packed, words=None, flags=None):
    words = packed.words if words is None else words
    lat = _cabi.Lattice(words.ctypes.data, words.size, packed.chunk_words, packed.n_chunks, packed.n_elements,
                        packed.flags if flags is None else flags)
    return _cabi.lib().xlb_lattice_validate(C.byref(lat))


def _record(packed, tag=lattice.T_EXCITER):
    """(first word index, words) of the first record with ``tag``."""
    w = packed.words
    pos = 0
    while True:
        hdr = int(w[pos])
        t, size = hdr & 0xFF, (hdr >> 16) & 0x3FFF
        if t == tag:
            return pos, w[pos: pos + 2 * size]
        if t == lattice.T_END_CHUNK:
            pos = (pos // packed.chunk_words + 1) * packed.chunk_words
            continue
        assert t != lattice.T_END_TURN, "no such record"
        pos += 2 * size


def _exciter(**kw):
    f = dict(knl=[1e-6, 2e-5], ksl=[3e-7], samples=[0.5, -1.0, 2.0], sampling_frequency=11245.5 * 2,
             frev=11245.5, start_turn=3)
    f.update(kw)
    return xl.Exciter(**f)


# ---------------------------------------------------------------- the element
def test_fields_defaults_and_not_a_multipole():
    e = xl.Exciter()
    assert (list(e.knl), list(e.ksl), tuple(e.samples), e.sampling_frequency, e.frev, e.start_turn) == \
        ([0], [0], (), 0, 0, 0)
    assert e.get_fields() == ["knl", "ksl", "samples", "sampling_frequency", "frev", "start_turn"]
    assert not isinstance(e, xl.Multipole) and "Exciter" in xl.element_classes()
    assert _exciter(knl=[0, 0, 1.0]).order == 2


def test_edits_of_samples_repack_and_json_round_trip(tmp_path):
    ex = _exciter(samples=np.arange(5.0))
    line = xl.Line([xl.Drift(length=1.0), ex])
    first = line.pack()
    assert line.pack() is first
    ex.samples[2] = 7.5  # item assignment on the array field
    second = line.pack()
    assert second is not first and second.words.view(np.float64)[-3] == 7.5
    ex.samples = [1.0, 2.0]
    assert line.pack().words.view(np.float64)[-2:].tolist() == [1.0, 2.0]
    ex.start_turn = 9
    assert int(_record(line.pack())[1].view(np.int64)[3]) == 9
    path = tmp_path / "line.json"
    line.to_json(str(path))
    back = xl.Line.from_json(str(path))
    assert back.elements[1] == ex and back.elements[1] is not ex
    assert np.array_equal(back.pack().words, line.pack().words)
    assert ex.copy() == ex and copy.deepcopy(line).pack().words.tobytes() == line.pack().words.tobytes()
    assert xl.Line.from_dict(line.to_dict()).elements[1] == ex


# ---------------------------------------------------------------- the record and the data region
def test_record_words_and_data_region():
    ex1 = _exciter()
    ex2 = _exciter(knl=[4e-6], ksl=[], samples=np.linspace(-1, 1, 7), sampling_frequency=3.0, frev=1.5,
                   start_turn=-2)
    packed = lattice.pack_line([xl.Drift(length=2.0), ex1, xl.Drift(length=1.0), ex2, xl.Multipole(knl=[1e-3])])
    assert packed.flags & lattice.F_EXCITER and packed.flags & lattice.F_LOW_ORDER
    region = packed.chunk_words * packed.n_chunks
    assert packed.words.size == region + 3 + 7
    f64, i64 = packed.words.view(np.float64), packed.words.view(np.int64)
    assert f64[region:].tolist() == [0.5, -1.0, 2.0] + np.linspace(-1, 1, 7).tolist()
    pos, rec = _record(packed)
    hdr = int(rec[0])
    assert (hdr & 0xFF, (hdr >> 8) & 0xFF, (hdr >> 16) & 0x3FFF, hdr >> 32) == (0x40, 1, 5, 1)
    rf, ri = rec.view(np.float64), rec.view(np.int64)
    assert rf[1] == (11245.5 * 2) / 11245.5 and rf[2] == (11245.5 * 2) / clight
    assert ri[3:6].tolist() == [3, 3, region]
    assert rf[6:10].tolist() == [2e-5, 0.0, 1e-6, 3e-7]  # (kn_1, ks_1), (kn_0, ks_0), kn_i = knl[i]/i!
    pos2, rec2 = _record(packed.__class__(packed.words[pos + 10:], 0, 0, 0, 0, dict(layout=[], words=0), {}))
    ri2, rf2 = rec2.view(np.int64), rec2.view(np.float64)
    assert (int(rec2[0]) >> 32, ri2[3], ri2[4], ri2[5]) == (3, -2, 7, region + 3)
    assert rf2[1] == 2.0 and rf2[6:8].tolist() == [4e-6, 0.0]
    assert _validate(packed) == 0
    # an order above 3 takes the lattice out of the low-order family
    assert not lattice.pack_line([_exciter(knl=[0, 0, 0, 0, 1.0])]).flags & lattice.F_LOW_ORDER


def test_exciter_is_never_fused_merged_or_dropped():
    els = [xl.Multipole(knl=[1e-4]), _exciter(knl=[0.0], samples=[]), xl.Multipole(knl=[2e-4]),
           xl.LimitRect(), xl.Drift(length=1.0)]
    packed = lattice.pack_line(els)
    assert packed.record_counts[lattice.T_EXCITER] == 1
    assert packed.record_counts.get(lattice.T_MERGED_BLOCK | lattice.AP_RECT_SYM | lattice.TB_DRIFT, 0) == 0
    assert _validate(packed) == 0


def test_validator_accepts_the_data_region_only_with_the_flag_and_checks_the_record():
    packed = lattice.pack_line([xl.Drift(length=1.0), _exciter(), xl.Drift(length=1.0)])
    assert _validate(packed) == 0
    pos, _ = _record(packed)
    region = packed.chunk_words * packed.n_chunks

    def broken(fn, flags=None):
        w = packed.words.copy()
        fn(w)
        return _validate(packed, w, flags)

    i64 = lambda w: w.view(np.int64)  # noqa: E731
    assert broken(lambda w: i64(w).__setitem__(pos + 5, region - 2)) == ELATTICE  # offset inside the chunks
    assert broken(lambda w: i64(w).__setitem__(pos + 5, region + 1)) == ELATTICE  # runs past n_words
    assert broken(lambda w: i64(w).__setitem__(pos + 5, 1 << 62)) == ELATTICE
    assert broken(lambda w: i64(w).__setitem__(pos + 4, -1)) == ELATTICE  # n_samples < 0
    assert broken(lambda w: i64(w).__setitem__(pos + 4, 4)) == ELATTICE
    assert broken(lambda w: w.view(np.float64).__setitem__(region + 1, np.nan)) == ELATTICE
    assert "sample" in _cabi.lib().xlb_last_error().decode()
    assert broken(lambda w: w.view(np.float64).__setitem__(pos + 1, np.inf)) == ELATTICE  # A
    assert broken(lambda w: w.view(np.float64).__setitem__(pos + 2, np.nan)) == ELATTICE  # B
    assert broken(lambda w: None, packed.flags & ~lattice.F_EXCITER) == ELATTICE  # record and region, no flag
    assert broken(lambda w: None, packed.flags | lattice.F_STRICT) == ELATTICE
    # a data region without the flag: refused even when no record points into it
    plain = lattice.pack_line([xl.Drift(length=1.0)])
    padded = np.concatenate([plain.words, np.zeros(2, dtype=np.uint64)])
    assert _validate(plain, padded) == ELATTICE and "n_words" in _cabi.lib().xlb_last_error().decode()
    assert _validate(plain, padded, plain.flags | lattice.F_EXCITER) == 0
    # every other tag of 0x40 .. 0x7f is an unknown tag
    for tag in range(0x41, 0x80):
        assert broken(lambda w: w.__setitem__(pos, np.uint64((int(w[pos]) & ~0xFF) | tag))) == ELATTICE, tag
        assert "unknown tag" in _cabi.lib().xlb_last_error().decode()


class _Huge:
    def __len__(self):
        return lattice.EXCITER_MAX_SAMPLES + 1


@pytest.mark.parametrize("fields, what", [
    (dict(sampling_frequency=0.0), "sampling_frequency"),
    (dict(sampling_frequency=-1.0), "sampling_frequency"),
    (dict(sampling_frequency=np.inf), "sampling_frequency"),
    (dict(frev=0.0), "frev"),
    (dict(frev=np.nan), "frev"),
    (dict(samples=[1.0, np.nan]), "sample"),
    (dict(samples=[np.inf]), "sample"),
    (dict(knl=[np.nan]), "knl"),
    (dict(ksl=[0.0, -np.inf]), "ksl"),
    (dict(start_turn=1.5), "start_turn"),
    (dict(start_turn=2.0), "start_turn"),
    (dict(start_turn=True), "start_turn"),
    (dict(samples=_Huge()), "samples"),
    (dict(knl=[0.0] * 65), "order"),
])
def test_pack_time_refusals(fields, what):
    with pytest.raises(ValueError, match=what):
        lattice.pack_line([_exciter(**fields)])


def test_refusals_name_the_exciter():
    line = xl.Line([xl.Drift(length=1.0), _exciter(), xl.Cavity(voltage=1e6, frequency=400e6)])
    with pytest.raises(ValueError, match="Exciter"):
        line.pack(strict=True)
    with pytest.raises(ValueError, match="Exciter"):
        lattice.pack_line(line.elements, strict=True)
    p = xl.Particles(p0c=P0C, mass0=M0, x=[0.0], device="cpu")
    with pytest.raises(ValueError, match="Exciter"):
        line.track_tangent(p, xl.TangentMap(1, "cpu"))
    with pytest.raises(ValueError, match="Exciter"):
        line.track_envelope(p, xl.Envelope(1, "cpu"))
    with pytest.raises(ValueError, match="Exciter"):
        xl.closed_orbit(line, p)
    line.radiation = "mean"
    with pytest.raises(ValueError, match="Exciter"):
        xl.radiation_equilibrium(line, p)


def test_exciter_lines_keep_beambeam6d_lenses_in_the_tracking_kernel():
    line = configs.config_lhc_beambeam(16)[0]
    assert line.pack().segments is not None
    packed = lattice.pack_line(list(line.elements) + [_exciter()])
    assert packed.segments is None and packed.flags & lattice.F_BB6D and packed.flags & lattice.F_EXCITER
    assert _validate(packed) == 0


# ---------------------------------------------------------------- existing lines are unchanged
# sha256 of the packed words of the configurations (16 particles), fast / strict, at the commit
# before exciters existed
PARENT_WORDS = {
    ("C2", False): "5c73ee221a67d3668ccd51b15a5f1601e4e8bf8a936cbeefb631718ac5a918c1",
    ("C2", True): "c261b114c8e4a5a6fea43ff9c5368c084a05ca554ebdbdf329bfee64557bb529",
    ("C3", False): "f79d38a19377e2f2842e3b3243ce8632abf8fc24a746ed043022a0d78ac8669d",
    ("C3", True): "5dd6d494a92855878501eeb2f360c5a5596ac65a39fdf789bb436a717f4a7dbc",
    ("C4", False): "09acc7d7366987430a9d00325b338e6fb50c21b115c6417aac7204c1e7b96656",
    ("C4", True): "e535e6c4d400d82deff6380fa167ab911e55d7a964ac1150af25ebd009539dea",
    ("C5", False): "5c4904d860d289bd8f17cc42255a42a0becab734d0d52717f8dd80584f544a5d",
    ("C5", True): "3f070407d97b5a84976fdd8df8c97a8552a82aee04ac2918ff5eb9a34326fac2",
}
CONFIGS = {"C2": configs.config_lhc, "C3": configs.config_lhc_beambeam, "C4": configs.config_petra4,
           "C5": configs.config_psb}


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_existing_lines_pack_to_the_same_words(name):
    line = CONFIGS[name](16)[0]
    for strict in (False, True):
        words = np.ascontiguousarray(line.pack(strict=strict).words)
        assert hashlib.sha256(words.tobytes()).hexdigest() == PARENT_WORDS[(name, strict)], (name, strict)


# ---------------------------------------------------------------- interpreter == oracle, bit for bit
def _half_sample_zetas(ex, turns, beta0, rng, n):
    """zeta values whose u + 0.5 lands on (or one ulp either side of) an integer, for turns ``turns``."""
    a, b = ex.sampling_frequency / ex.frev, ex.sampling_frequency / clight
    t = rng.choice(turns, n).astype(np.float64) - ex.start_turn
    k = rng.integers(-2, len(ex.samples) + 2, n).astype(np.float64)
    z = (t * a - (k - 0.5)) * beta0 / b
    return np.nextafter(z, rng.choice([-np.inf, np.inf], n)) if rng.random() < 0.5 else z


def _random_line(rng):
    """Elements whose fast encoding the interpreter evaluates in the oracle's operation order (drifts,
    straight multipoles of order <= 2, rectangles, shifts) and exciters of order <= 2."""
    els = []
    for _ in range(rng.integers(6, 14)):
        kind = rng.integers(0, 5)
        if kind == 0:
            els.append(xl.Drift(length=float(rng.uniform(0.1, 3.0))))
        elif kind == 1:
            order = int(rng.integers(0, 3))
            els.append(xl.Multipole(knl=list(rng.normal(0, 1e-3, order + 1)), ksl=list(rng.normal(0, 1e-4, order + 1))))
        elif kind == 2:
            els.append(xl.LimitRect(min_x=-0.01, max_x=0.012, min_y=-0.011, max_y=0.01))
        elif kind == 3:
            els.append(xl.XYShift(dx=float(rng.normal(0, 1e-4)), dy=float(rng.normal(0, 1e-4))))
        else:
            order = int(rng.integers(0, 3))
            h = float(rng.choice([1.0, 2.0, 0.37, 35640.0]))
            els.append(xl.Exciter(knl=list(rng.normal(0, 1e-4, order + 1)), ksl=list(rng.normal(0, 1e-5, order)),
                                  samples=list(rng.normal(0, 1, int(rng.integers(0, 9)))),
                                  sampling_frequency=11245.5 * h, frev=11245.5, start_turn=int(rng.integers(-2, 3))))
    els.append(_exciter(samples=[2.0 ** k for k in range(6)], sampling_frequency=11245.5, start_turn=0, knl=[1e-5]))
    return els


@pytest.mark.parametrize("seed", range(12))
def test_interpreter_equals_the_oracle_bit_for_bit(seed):
    rng = np.random.default_rng(seed)
    els = _random_line(rng)
    n, turns = 400, 4
    beta0 = P0C / math.sqrt(P0C * P0C + M0 * M0)
    ex = els[-1]
    zeta = _half_sample_zetas(ex, np.arange(turns), beta0, rng, n)
    zeta[:8] = [np.nan, np.inf, -np.inf, 0.0, -0.0, 1e-300, -1e-300, 5e-324]
    cols = dict(x=rng.normal(0, 1e-3, n), px=rng.normal(0, 1e-5, n), y=rng.normal(0, 1e-3, n),
                py=rng.normal(0, 1e-5, n), zeta=zeta, delta=rng.normal(0, 1e-4, n),
                at_turn=rng.integers(0, 3, n))
    packed = lattice.pack_line(els, merge=False)
    assert _validate(packed) == 0
    got = EI.track(packed, cols, P0C, M0, num_turns=turns)
    want = EO.run_oracle(xl.Line(els).to_specs(), cols, P0C, M0, num_turns=turns)
    for k in ("state", "at_element", "at_turn"):
        assert np.array_equal(got[k], want[k]), k
    for k in ("x", "px", "y", "py", "zeta", "delta"):
        assert np.array_equal(got[k].view(np.int64), want[k].view(np.int64)), k


def test_sample_index_rounds_to_nearest_and_matches_the_record():
    """With sampling_frequency == frev a particle with |zeta| < C/2 reads the sample of its own turn; the
    interpreter's index from the record words equals the oracle's from the fields at half-sample
    boundaries, one ulp either side and for non-finite zeta."""
    frev = 11245.5
    circumference = 299792458.0 * (P0C / math.sqrt(P0C * P0C + M0 * M0)) / frev
    beta0 = P0C / math.sqrt(P0C * P0C + M0 * M0)
    ex = _exciter(samples=np.arange(10.0), sampling_frequency=frev, frev=frev, start_turn=2)
    f = ex.to_dict()
    turns = np.array([0, 1, 2, 3, 11, 12, 13])
    z = np.linspace(-0.499, 0.499, 11) * circumference
    T, Z = np.meshgrid(turns, z)
    idx = EO.sample_index(f, T.ravel(), Z.ravel(), beta0)
    own = T.ravel() - 2
    assert np.array_equal(idx, np.where((own >= 0) & (own < 10), own, -1))
    packed = lattice.pack_line([ex])
    pos, _ = _record(packed)
    rng = np.random.default_rng(7)
    for h in (1.0, 2.0, 35640.0):
        ex.sampling_frequency = frev * h
        ex.samples = np.arange(50.0)
        packed = lattice.pack_line([ex])
        pos, _ = _record(packed)
        zeta = np.concatenate([_half_sample_zetas(ex, np.arange(40), beta0, rng, 4000),
                               [np.nan, np.inf, -np.inf, 0.0]])
        at_turn = rng.integers(0, 40, len(zeta))
        want = EO.sample_index(ex.to_dict(), at_turn, zeta, beta0)
        got = EI.exciter_index(packed.words.view(np.float64), packed.words.view(np.int64), pos, at_turn, zeta, beta0)
        assert np.array_equal(got, want)
        assert (want >= 0).any() and (want < 0).any()


def test_algorithmic_ops():
    els = [xl.Drift(length=1.0), _exciter(), _exciter(knl=[1.0], ksl=[])]
    assert lattice.algorithmic_ops(els) == EO.algorithmic_ops(xl.Line(els).to_specs()) == 15 + (14 + 8) + (4 + 8)


def test_particles_on_cpu_do_not_track():
    line = xl.Line([_exciter()])
    p = xl.Particles(p0c=P0C, mass0=M0, x=[0.0], device="cpu")
    with pytest.raises(RuntimeError):
        line.track(p)
    assert torch.equal(p.x, torch.zeros(1, dtype=torch.float64))
