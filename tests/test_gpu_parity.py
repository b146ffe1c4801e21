"""GPU parity tests proper: the CUDA path (through the C ABI) against

* the committed outputs of the reference's own element code (tests/golden), and
* the CPU oracle on the same seeded inputs,

for the fast (FMA, pre-folded constants) and strict (reference operation order) kernels.
Tolerances, from BASELINE.json's north_star: coordinates within 1e-12 relative after one
turn; state / at_element / at_turn bit-exact except for particles within EDGE_EPS of an
aperture edge (none of the cases below has one unless stated).
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from tests import helpers as H

pytestmark = pytest.mark.gpu

REL_TOL_ONE_TURN = 1e-12   # north_star tolerance, fast kernel vs reference
STRICT_TOL = 4e-16         # strict kernel: <= 2 ulp (libm-vs-CUDA sin/cos/exp only)
FAST_FULL_TURN_TOL = 1e-11  # fast kernel, worst particle, one full LHC turn (see DESIGN.md)
EDGE_EPS = 1e-9            # aperture margin [m] inside which loss flags may differ

BEAMFIELD_TYPES = ("BeamBeam4D", "BeamBeam6D", "SCCoasting", "SCQGaussProfile", "SCInterpolatedProfile")
LEAN_CASES = sorted(k for k, m in H.manifest().items() if m["type"] not in BEAMFIELD_TYPES)


def build_line(specs):
    import xline_b200 as xl

    els = []
    for name, f in specs:
        cls = getattr(xl, name)
        base = {k: v for k, v in f.items() if k in cls().get_fields(keepextra=True)}
        els.append(cls(**base))
    return xl.Line(els)


def make_particles(cols, p0c, mass0, device="cuda"):
    import xline_b200 as xl

    return xl.Particles(p0c=p0c, mass0=mass0, device=device, **cols)


def run_gpu(specs, cols, p0c, mass0, num_turns=1, **kw):
    line = build_line(specs)
    p = make_particles(cols, p0c, mass0)
    line.track(p, num_turns=num_turns, **kw)
    torch.cuda.synchronize()
    return p.to_numpy(), line


@pytest.mark.parametrize("ppt", [1, 2, 3, 4])
@pytest.mark.parametrize("case", LEAN_CASES)
def test_fast_kernel_matches_reference_outputs(case, ppt):
    m, specs, cols, ref = H.load_case(case)
    got, _ = run_gpu(specs, cols, m["p0c"], m["mass0"], num_turns=m.get("num_turns", 1),
                     particles_per_thread=ppt)
    assert np.array_equal(got["state"], ref["state"]), case
    assert np.array_equal(got["at_element"], ref["at_element"]), case
    assert np.array_equal(got["at_turn"], ref["at_turn"]), case
    for k in H.COORDS + ("rpp", "rvv", "s"):
        err = H.rel_err(got[k], ref[k])
        tol = REL_TOL_ONE_TURN * m.get("num_turns", 1)
        assert err <= tol, (case, k, err)


@pytest.mark.parametrize("ppt", [1, 2])
@pytest.mark.parametrize("case", LEAN_CASES)
def test_strict_kernel_matches_reference_outputs(case, ppt):
    m, specs, cols, ref = H.load_case(case)
    got, _ = run_gpu(specs, cols, m["p0c"], m["mass0"], num_turns=m.get("num_turns", 1),
                     strict=True, particles_per_thread=ppt)
    for k in ("state", "at_element", "at_turn"):
        assert np.array_equal(got[k], ref[k]), (case, k)
    transcendental = any(t in case for t in ("cavity", "rfmult", "line"))  # sin/cos differ in the last ulp
    for k in H.COORDS + ("rpp", "rvv", "s"):
        err = H.rel_err(got[k], ref[k])
        if transcendental:
            assert err <= STRICT_TOL * 8, (case, k, err)
        else:
            # only + - * / sqrt: IEEE-identical to the NumPy path
            assert np.array_equal(got[k], ref[k], equal_nan=True), (case, k, err)


def test_fodo_c1_against_oracle_100_turns():
    """BASELINE config C1 (FODO cell, 10k particles x 100 turns) -- full size on the oracle."""
    from xline_b200 import configs

    line, cols, p0c, m0 = configs.config_fodo(10_000)
    p = make_particles(cols, p0c, m0)
    line.track(p, num_turns=100)
    got = p.to_numpy()
    ref = H.run_oracle(line.to_specs(), cols, p0c, m0, num_turns=100)
    assert np.array_equal(got["state"], ref["state"])
    assert np.array_equal(got["at_turn"], ref["at_turn"])
    worst = max(H.scaled_err(got[k], ref[k]) for k in H.COORDS)
    # documented error growth: ~1e-16 * sqrt(ops); 100 turns of an 11-element cell
    assert worst <= 1e-11, worst
    # strict kernel on the same job
    p2 = make_particles(cols, p0c, m0)
    line.track(p2, num_turns=100, strict=True)
    got2 = p2.to_numpy()
    worst2 = max(H.scaled_err(got2[k], ref[k]) for k in H.COORDS)
    assert worst2 <= 1e-11, worst2  # sin() of the cavity: CUDA vs glibc last-ulp differences, 100 turns


def _edge_margin_lhc(line, snap_x, snap_y):
    return None


def test_lhc_one_turn_against_oracle():
    """C2 lattice (LHC + apertures), 2000-particle subsample x 1 turn against the oracle."""
    from xline_b200 import configs

    line, cols, p0c, m0 = configs.config_lhc(2000)
    p = make_particles(cols, p0c, m0)
    line.track(p, num_turns=1)
    got = p.to_numpy()
    ref = H.run_oracle(line.to_specs(), cols, p0c, m0, num_turns=1)
    differ = np.nonzero((got["state"] != ref["state"]) | (got["at_element"] != ref["at_element"]))[0]
    # loss flags bit-exact except within EDGE_EPS of an aperture edge: with 2000 particles
    # and 7.6k apertures, none is expected that close
    assert len(differ) == 0, differ
    assert (ref["state"] == 0).sum() > 0, "config must exercise losses"
    alive = ref["state"] == 1
    for k in H.COORDS:
        # error relative to the beam's r.m.s. of the coordinate (a coordinate passing through
        # zero has no meaningful elementwise relative error)
        serr = H.scaled_err(got[k][alive], ref[k][alive])
        # FAST kernel over a full LHC turn (~1e6 fp64 operations per particle, FMA-contracted,
        # 1/i! folded into the coefficients): rounding differences with the NumPy path add up
        # to a few 1e-12 of the beam size for the worst of 2000 particles (median ~1e-13; see
        # DESIGN.md "Accuracy" and profiles/accuracy_r1.json).  The STRICT kernel below, which
        # keeps the reference's operation order, meets 1e-12 with two orders of margin.
        assert serr <= FAST_FULL_TURN_TOL, (k, serr)
    lost = ~alive
    for k in H.COORDS:  # frozen at the aperture
        assert H.scaled_err(got[k][lost], ref[k][lost]) <= REL_TOL_ONE_TURN, k
    # strict kernel: IEEE-identical except the 12 cavities (sin)
    p2 = make_particles(cols, p0c, m0)
    line.track(p2, num_turns=1, strict=True)
    got2 = p2.to_numpy()
    assert np.array_equal(got2["state"], ref["state"])
    assert np.array_equal(got2["at_element"], ref["at_element"])
    for k in H.COORDS:
        assert H.scaled_err(got2[k], ref[k]) <= 1e-14, k


def test_fused_records_equal_unfused_bitwise():
    """The pack-time peephole (multipole -> aperture -> drift in one record) must not change
    a single bit: same maps, same order."""
    from xline_b200 import configs

    line, cols, p0c, m0 = configs.config_lhc(20_000)
    line.merge_multipoles = False  # merging sums coefficients: exact in real arithmetic only
    outs = []
    for fuse in (True, False):
        line.fuse_records = fuse
        line.invalidate()
        for strict in (False, True):
            p = make_particles(cols, p0c, m0)
            line.track(p, num_turns=2, strict=strict)
            outs.append(p.to_numpy())
    assert (outs[0]["state"] == 0).sum() > 0
    for k in outs[0]:
        assert np.array_equal(outs[0][k], outs[2][k], equal_nan=True), ("fast", k)
        assert np.array_equal(outs[1][k], outs[3][k], equal_nan=True), ("strict", k)


def test_merged_multipoles_match_separate_kicks():
    """Pack-time merging of co-located thin multipoles ([K1][A1][K2][A2][drift] -> one summed
    kick): same losses at the same places and turns, coordinates equal to rounding noise, and
    particles lost at A1 frozen with the momentum they had after K1 only."""
    from xline_b200 import configs

    n = 40_000
    line, cols, p0c, m0 = configs.config_lhc(n)
    cols["x"][:4000] *= 6.0  # plenty of losses, at A1 apertures too
    res = []
    for merge in (True, False):
        line.merge_multipoles = merge
        line.invalidate()
        p = make_particles(cols, p0c, m0)
        line.track(p, num_turns=1)
        res.append((p.to_numpy(), line.loss_tally.cpu().numpy().copy(), line.pack().record_counts))
    (a, ta, ca), (b, tb, cb) = res
    assert sum(ca.values()) < sum(cb.values()) and any(k & 0x20 and k & 0x80 for k in ca)
    assert np.array_equal(a["state"], b["state"]) and np.array_equal(a["at_element"], b["at_element"])
    assert np.array_equal(a["at_turn"], b["at_turn"]) and np.array_equal(ta, tb)
    lost = a["state"] == 0
    assert lost.sum() > 1000
    a1_elements = {i for i, el in enumerate(line.elements) if type(el).__name__ == "LimitEllipse"}
    assert sum(int(e) in a1_elements for e in a["at_element"][lost]) > 10
    for k in H.COORDS:
        assert H.scaled_err(a[k][~lost], b[k][~lost]) <= FAST_FULL_TURN_TOL, k
        assert H.scaled_err(a[k][lost], b[k][lost]) <= FAST_FULL_TURN_TOL, ("lost", k)
    # first-turn losses: momentum frozen after K1 only -> equal to rounding of the single kick
    first = lost & (a["at_turn"] == 0)
    assert np.allclose(a["px"][first], b["px"][first], rtol=1e-11, atol=1e-16)


def test_loss_tally_and_compaction_paths_agree():
    from xline_b200 import configs

    line, cols, p0c, m0 = configs.config_lhc(6000)
    p1 = make_particles(cols, p0c, m0)
    line.track(p1, num_turns=6)
    tally1 = line.loss_tally.clone()
    a = p1.to_numpy()
    n_lost = int((a["state"] == 0).sum())
    assert n_lost > 0
    assert int(tally1.sum()) == n_lost
    hist = np.bincount(a["at_element"][a["state"] == 0], minlength=len(line))
    assert np.array_equal(hist, tally1.cpu().numpy())
    # same job, survivors re-compacted between 1-turn launches: bit-identical result
    line.invalidate()
    p2 = make_particles(cols, p0c, m0)
    line.track(p2, num_turns=6, turns_per_launch=1)
    assert line.last_stats["kernel_launches"] == 6
    b = p2.to_numpy()
    for k in a:
        if k == "s":  # fast kernel: s = s + (sum of drift lengths of the launch); the grouping
            assert np.allclose(a[k], b[k], rtol=1e-11, atol=0)  # of the sum follows the launches
        else:
            assert np.array_equal(a[k], b[k], equal_nan=True), k
    assert np.array_equal(line.loss_tally.cpu().numpy(), tally1.cpu().numpy())


def test_work_queue_equals_one_item_per_cta_bitwise():
    """Persistent CTAs pulling (particle block, turn segment) items must reproduce the plain
    launch bit for bit (same maps; only the schedule differs), losses included."""
    from xline_b200 import configs

    n = 200_000  # more particle blocks than the device holds at once -> the queue is used
    line, cols, p0c, m0 = configs.config_lhc(n)
    outs = []
    for tpi in (-1, 5, 2):
        line.invalidate()
        p = make_particles(cols, p0c, m0)
        line.track(p, num_turns=11, turns_per_item=tpi)
        outs.append(p.to_numpy())
        tally = line.loss_tally.cpu().numpy().copy()
        if tpi == -1:
            tally0 = tally
        else:
            assert np.array_equal(tally, tally0)
    assert 0 < (outs[0]["state"] == 0).sum() < n
    for k in outs[0]:
        for o in outs[1:]:
            if k == "s":
                assert np.allclose(outs[0][k], o[k], rtol=1e-11, atol=0)
            else:
                assert np.array_equal(outs[0][k], o[k], equal_nan=True), k


def test_compaction_kernel_matches_numpy():
    from xline_b200 import _cabi

    rng = np.random.default_rng(5)
    for n in (1, 31, 4097, 100_003):
        state = torch.from_numpy((rng.random(n) < 0.37).astype(np.int64)).cuda()
        idx = torch.empty(n, dtype=torch.int32, device="cuda")
        cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
        _cabi.check(_cabi.lib().xlb_compact_alive_device(
            state.data_ptr(), n, idx.data_ptr(), cnt.data_ptr(),
            C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        torch.cuda.synchronize()
        want = np.nonzero(state.cpu().numpy() == 1)[0]
        assert int(cnt.item()) == len(want)
        assert np.array_equal(idx[: len(want)].cpu().numpy(), want)


HOST_ENTRY_CASES = [
    pytest.param(False, 3000, None, id="False-3000"), pytest.param(True, 3000, None, id="True-3000"),
    pytest.param(True, 40_000, None, id="True-40000")] + [
    pytest.param(pinned, 3000, case, id="%s-3000-%s" % (pinned, case))
    for case in ("tally", "monitor", "species", "launches") for pinned in (False, True)]


@pytest.mark.parametrize("pinned,n,case", HOST_ENTRY_CASES)
def test_host_entry_point_matches_device_entry_point(pinned, n, case):
    """xlb_track_host == Line.track on device tensors: pageable host buffers (copies inside),
    small pinned buffers (tracked in place through their device aliases, no copies) and pinned
    buffers above the in-place limit (copies again); apertures so that lost particles are written
    back through the same path.  The extra cases add a loss tally, BeamMonitor storage, chi and
    charge_ratio columns of two species, and launches of 3 turns (survivors re-compacted between
    them)."""
    import xline_b200 as xl
    from xline_b200 import _cabi, configs

    line, cols, p0c, m0 = configs.config_fodo(n)
    elements = list(line.elements) + [xl.LimitEllipse(a=3.5e-3, b=3.5e-3)]
    if case == "monitor":
        elements.append(xl.BeamMonitor(num_stores=3, start=1, skip=2, min_particle_id=100, max_particle_id=2099))
    line = xl.Line(elements)
    if case == "species":
        other = np.random.default_rng(3).random(n) < 0.5
        cols = dict(cols, charge_ratio=np.where(other, 2.0, 1.0), chi=np.where(other, 0.5, 1.0))
    turns_per_launch = 3 if case == "launches" else 0
    p = make_particles(cols, p0c, m0)
    line.track(p, num_turns=7, turns_per_launch=turns_per_launch)
    want = p.to_numpy()
    assert 0 < (want["state"] == 0).sum() < n
    hp = xl.Particles(p0c=p0c, mass0=m0, device="cpu", pinned=pinned, **cols)
    packed = line.pack()
    lat = _cabi.Lattice(packed.words.ctypes.data, packed.words.size, packed.chunk_words,
                        packed.n_chunks, packed.n_elements, packed.flags)
    cp = _cabi.Particles()
    cp.n = len(hp)
    for k, t in hp._columns():
        setattr(cp, k, t.data_ptr())
    cp.q0, cp.mass0, cp.p0c = hp.q0, hp.mass0, hp.p0c
    cp.beta0, cp.gamma0, cp.energy0 = hp.beta0, hp.gamma0, hp.energy0
    opts = _cabi.TrackOptions()
    opts.num_turns = 7
    opts.turns_per_launch = turns_per_launch
    if case == "tally":
        tally = torch.zeros(packed.n_elements, dtype=torch.int64, pin_memory=pinned)
        opts.loss_tally = tally.data_ptr()
    if case == "monitor":
        mon = torch.full((packed.monitor_words,), float("nan"), dtype=torch.float64, pin_memory=pinned)
        opts.monitor_data, opts.monitor_words = mon.data_ptr(), packed.monitor_words
    _cabi.check(_cabi.lib().xlb_track_host(C.byref(lat), C.byref(cp), C.byref(opts)))
    got = hp.to_numpy()
    for k in want:
        assert np.array_equal(want[k], got[k], equal_nan=True), k
    if case == "tally":
        assert int(tally.sum()) == (want["state"] == 0).sum()
        assert np.array_equal(tally.numpy(), line.loss_tally[: packed.n_elements].cpu().numpy())
    if case == "monitor":
        assert np.isfinite(mon.numpy()).any()
        assert np.array_equal(mon.numpy(), line._monitor_buf.cpu().numpy(), equal_nan=True)


def test_monitor_records_like_oracle():
    import xline_b200 as xl

    n, turns = 500, 9
    rng = np.random.default_rng(11)
    cols = dict(x=rng.normal(0, 1e-3, n), px=rng.normal(0, 1e-4, n), y=rng.normal(0, 1e-3, n),
                py=rng.normal(0, 1e-4, n), zeta=rng.normal(0, 0.05, n), delta=rng.normal(0, 3e-4, n))
    mon = xl.BeamMonitor(num_stores=3, start=2, skip=2, min_particle_id=10, max_particle_id=409)
    line = xl.Line([
        xl.Drift(length=1.0), xl.Multipole(knl=[0, 0.3]), xl.LimitEllipse(a=3e-3, b=3e-3), mon,
        xl.Drift(length=2.0), xl.Multipole(knl=[0, -0.3]), xl.Cavity(voltage=1e6, frequency=4e8, lag=180),
    ])
    p = make_particles(cols, 450e9, 938.27208816e6)
    line.track(p, num_turns=turns)
    monitors = {}
    ref = H.run_oracle(line.to_specs(), cols, 450e9, 938.27208816e6, num_turns=turns, monitors=monitors)
    store = monitors[3]
    assert (ref["state"] == 0).sum() > 0
    for k in ("x", "px", "y", "py", "zeta", "delta"):
        got = mon.data[k].cpu().numpy()
        want = store[k]
        written = store["at_turn"] >= 0
        assert np.array_equal(np.isnan(got), ~written), k
        assert H.scaled_err(got[written], want[written]) <= 1e-12, k
    gt = mon.data["at_turn"].cpu().numpy()
    assert np.array_equal(gt[store["at_turn"] >= 0], store["at_turn"][store["at_turn"] >= 0].astype(float))


def test_sharding_invariance_full_size():
    """Size-independent property at C2 scale: tracking [A|B] together equals tracking A
    and B separately, bit for bit (particles are independent; order of lanes irrelevant)."""
    from xline_b200 import configs

    n = 300_000
    line, cols, p0c, m0 = configs.config_lhc(n)
    p = make_particles(cols, p0c, m0)
    line.track(p, num_turns=2)
    whole = p.to_numpy()
    cut = 123_457
    parts = []
    for sl in (slice(0, cut), slice(cut, n)):
        q = make_particles({k: v[sl] for k, v in cols.items()}, p0c, m0)
        line.track(q, num_turns=2, particles_per_thread=1)
        parts.append(q.to_numpy())
    for k in whole:
        joined = np.concatenate([parts[0][k], parts[1][k]])
        assert np.array_equal(whole[k], joined, equal_nan=True), k
    lost = whole["state"] == 0
    assert 0 < lost.sum() < n


@pytest.mark.parametrize("config", ["lhc", "petra4"])
def test_kernel_variants_agree_bitwise(config):
    """Every compiled (particles per thread, threads per block) variant of the fast kernel gives
    the same bits: the fast maps spell their FMAs out, so no instantiation is free to fuse a
    different product of a sum of products (csrc/track_impl.cuh, el_drift)."""
    from xline_b200 import configs

    n = 60_000
    line, cols, p0c, m0 = (configs.config_lhc if config == "lhc" else configs.config_petra4)(n)
    ref = None
    for ppt, thr in ((3, 128), (1, 128), (1, 256), (1, 512), (2, 128), (2, 256), (4, 128)):
        p = make_particles(cols, p0c, m0)
        line.track(p, num_turns=2, particles_per_thread=ppt, threads_per_block=thr)
        cur = p.to_numpy()
        if ref is None:
            ref = cur
            continue
        for k in ref:
            assert np.array_equal(ref[k], cur[k], equal_nan=True), (k, ppt, thr)


@pytest.mark.parametrize("config", ["lhc", "petra4", "lhc_beambeam"])
def test_kernel_families_agree_bitwise(config):
    """The specialised kernel families (chi == 1 throughout: no chi register, 4 particles per
    thread; multipole order <= 3: straight-line Horner) give the bits of the general kernels:
    fma(-1, a, b) == b - a, and the Horner steps are the same operations in the same order."""
    from xline_b200 import configs

    n = 50_000
    fn = {"lhc": configs.config_lhc, "petra4": configs.config_petra4, "lhc_beambeam": configs.config_lhc_beambeam}[config]
    line, cols, p0c, m0 = fn(n)
    packed = line.pack(False)
    assert bool(packed.flags & 8) == (config != "lhc")  # XLB_F_LOW_ORDER
    ref = make_particles(cols, p0c, m0)
    line.track(ref, num_turns=2, particles_per_thread=3, threads_per_block=128, _general_kernels=True)
    ref = ref.to_numpy()
    names = set()
    for ppt in (1, 2, 3, 4, 0):
        p = make_particles(cols, p0c, m0)
        line.track(p, num_turns=2, particles_per_thread=ppt)
        cur = p.to_numpy()
        for k in ref:
            assert np.array_equal(ref[k], cur[k], equal_nan=True), (k, ppt)
    # a chi column that is not all ones goes through the general family and scales the kicks
    p = make_particles(cols, p0c, m0)
    p.chi[::2] = 1.0 + 1e-3
    line.track(p, num_turns=1)
    q = make_particles(cols, p0c, m0)
    line.track(q, num_turns=1)
    assert not torch.equal(p.px[::2], q.px[::2]) and torch.equal(p.px[1::2], q.px[1::2])


def test_track_refuses_cpu_particles():
    import xline_b200 as xl

    p = xl.Particles(p0c=1e9, x=[0.0, 1.0], device="cpu")
    with pytest.raises(RuntimeError):
        xl.Line([xl.Drift(length=1.0)]).track(p)


def test_reference_api_semantics_on_device():
    """Reference tests/test_track.py:48-73 and tests/test_losses.py, through the GPU path."""
    import xline_b200 as xl

    el = xl.LimitRect(min_x=-0.1, max_x=0.3, min_y=-0.5, max_y=0.1)
    arr = np.arange(0, 1, 0.001)
    p2 = xl.Particles(x=arr, y=arr)
    el.track(p2)
    survive = (arr >= -0.1) & (arr <= 0.3) & (arr >= -0.5) & (arr <= 0.1)
    assert int((p2.state == 1).sum()) == int(survive.sum())
    p2.remove_lost_particles()
    assert len(p2) == int(survive.sum())
    assert len(p2.lost_particles[0]) == len(arr) - int(survive.sum())
    p2.x += 0.3 + 1e-6
    el.track(p2)
    p2.remove_lost_particles()
    assert len(p2.x) == 0
    # RFMultipole(f=0) == Multipole (tests/test_track.py:33-45)
    p1 = xl.Particles(p0c=1e9, x=1.0, y=1.0)
    q1 = p1.copy()
    xl.RFMultipole(knl=[0.5, 2, 0.2], ksl=[0.5, 3, 0.1]).track(p1)
    xl.Multipole(knl=[0.5, 2, 0.2], ksl=[0.5, 3, 0.1]).track(q1)
    assert p1.compare(q1, abs_tol=1e-15)


# ------------------------------------------------------------------ beam-field elements
BF_CASES = sorted(k for k, m in H.manifest().items() if m["type"] in BEAMFIELD_TYPES)
BF_TOL = 1e-12  # relative to the beam r.m.s. of each coordinate (per particle: test_gpu_beamfield_accuracy)


@pytest.mark.parametrize("strict", [False, True])
@pytest.mark.parametrize("ppt", [1, 2])
@pytest.mark.parametrize("case", BF_CASES)
def test_beamfield_elements_match_reference_outputs(case, ppt, strict):
    m, specs, cols, ref = H.load_case(case)
    got, line = run_gpu(specs, cols, m["p0c"], m["mass0"], particles_per_thread=ppt, strict=strict)
    assert line.pack(strict).flags & 6  # XLB_F_BEAMFIELDS or (segmented fast lattice) XLB_F_BB6D
    assert np.array_equal(got["state"], ref["state"])
    for k in H.COORDS + ("rpp", "rvv"):
        err = H.scaled_err(got[k], ref[k])
        assert err <= BF_TOL, (case, k, err)
    # the kick itself (what the lens adds), relative to the r.m.s. kick
    for k in ("px", "py"):
        kick_ref = ref[k] - cols[k]
        kick_got = got[k] - cols[k]
        scale = np.sqrt(np.mean(kick_ref ** 2))
        if scale > 0:
            assert np.max(np.abs(kick_got - kick_ref)) <= 2e-10 * scale + 1e-16 * np.max(np.abs(cols[k])), (case, k)


def test_bbsimple_lattice_against_oracle():
    """examples/bbsimple: FODO cell with one 6D and one 4D lens, 3 turns."""
    from xline_b200 import configs

    line, meta = configs.load_lattice("bbsimple")
    p0c, m0 = configs.p0c_of(meta)
    rng = np.random.default_rng(7)
    n = 600
    cols = dict(x=rng.normal(0, 2e-3, n), px=rng.normal(0, 2e-4, n), y=rng.normal(0, 2e-3, n),
                py=rng.normal(0, 2e-4, n), zeta=rng.normal(0, 0.3, n), delta=rng.normal(0, 3e-4, n))
    p = make_particles(cols, p0c, m0)
    line.track(p, num_turns=3)
    got = p.to_numpy()
    ref = H.run_oracle(line.to_specs(), cols, p0c, m0, num_turns=3)
    for k in H.COORDS:
        assert H.scaled_err(got[k], ref[k]) <= 5e-12, (k, H.scaled_err(got[k], ref[k]))


def test_segmented_6d_lens_launches_match_fused_kernel_and_oracle():
    """Fast path of lattices with BeamBeam6D lenses: the tracking kernel stops in front of every
    6D lens, a stand-alone lens kernel runs, tracking resumes (xlb_lattice_t::segments).  Must
    agree with the single fused kernel (split_lenses = False) and with the oracle, including turn
    counting, loss bookkeeping, BeamMonitor contents, launch segmentation and the host entry point."""
    import xline_b200 as xl
    from xline_b200 import _cabi
    from tests.test_host_logic import _bb6d

    def lens(**kw):
        return _bb6d(sigma_11=4e-7, sigma_22=1e-9, sigma_33=6e-7, sigma_44=2e-9, sigma_12=1e-9, sigma_34=-2e-9,
                     charge_slices=[3e10, 5e10, 3e10], **kw)

    turns, n = 7, 1500
    ap = 2.2e-3
    els = [lens(), xl.Drift(length=3.0), xl.Multipole(knl=[0, 0.25, 2.0]),
           xl.LimitRect(min_x=-ap, max_x=ap, min_y=-1.2 * ap, max_y=1.2 * ap), xl.Drift(length=2.0),
           lens(phi=2e-4, alpha=1.0), lens(phi=-1e-4),
           xl.BeamBeam4D(charge=2e10, sigma_x=8e-4, sigma_y=5e-4, beta_r=1.0),
           xl.Multipole(knl=[0, -0.25]), xl.LimitEllipse(a=1.2 * ap, b=1.2 * ap), xl.Drift(length=3.0),
           xl.Cavity(voltage=1e6, frequency=4e8, lag=180.0),
           xl.BeamMonitor(num_stores=turns, start=0, skip=1, min_particle_id=0, max_particle_id=n - 1), lens(phi=5e-5)]
    line = xl.Line(els)
    assert [s[2] for s in line.pack().segments.tolist()] == [1, 0, 1, 1, 0, 1, 0]
    rng = np.random.default_rng(11)
    cols = dict(x=rng.normal(0, 9e-4, n), px=rng.normal(0, 3e-5, n), y=rng.normal(0, 9e-4, n),
                py=rng.normal(0, 3e-5, n), zeta=rng.normal(0, 0.05, n), delta=rng.normal(0, 3e-4, n))
    p0c, m0 = 7e12, 938.27208816e6
    ref_mon = {}
    ref = H.run_oracle(line.to_specs(), cols, p0c, m0, num_turns=turns, monitors=ref_mon)
    assert 20 < (ref["state"] == 0).sum() < n // 2
    mon = els[-2]

    def check(got, tol):
        assert np.array_equal(got["state"], ref["state"])
        assert np.array_equal(got["at_element"], ref["at_element"])
        assert np.array_equal(got["at_turn"], ref["at_turn"])
        for k in H.COORDS:
            assert H.scaled_err(got[k], ref[k]) <= tol, (k, H.scaled_err(got[k], ref[k]))
        store = list(ref_mon.values())[0]
        written = store["at_turn"] >= 0
        for k in ("x", "px", "y", "py", "zeta", "delta"):
            g = mon.data[k].cpu().numpy()
            assert np.array_equal(np.isnan(g), ~written)
            assert H.scaled_err(g[written], store[k][written]) <= tol, k

    results = {}
    for name, kw in (("split", {}), ("split_segmented", dict(turns_per_launch=3)),
                     ("split_ppt1", dict(particles_per_thread=1, threads_per_block=256))):
        line.reset_monitors()
        p = make_particles(cols, p0c, m0)
        line.track(p, num_turns=turns, **kw)
        assert line.last_stats["kernel_launches"] == turns * 7
        results[name] = p.to_numpy()
        check(results[name], 2e-11)
    line.split_lenses = False
    line.reset_monitors()
    p = make_particles(cols, p0c, m0)
    line.track(p, num_turns=turns)
    assert line.last_stats["kernel_launches"] == 1
    fused = p.to_numpy()
    check(fused, 2e-11)
    line.split_lenses = True
    for k in H.COORDS:  # same arithmetic in both organisations
        assert H.scaled_err(results["split"][k], fused[k]) <= 1e-13, k
        assert np.array_equal(results["split"][k], results["split_segmented"][k], equal_nan=True) or k == "s", k
    # strict kernel: one fused launch, reference operation order
    line.reset_monitors()
    p = make_particles(cols, p0c, m0)
    line.track(p, num_turns=turns, strict=True)
    check(p.to_numpy(), 1e-12)
    # host entry point with a segmented lattice
    line.reset_monitors()
    hp = make_particles(cols, p0c, m0, device="cpu")
    packed = line.pack()
    lat = packed.c_lattice()
    cp = _cabi.Particles()
    cp.n = len(hp)
    for k, t in hp._columns():
        setattr(cp, k, t.data_ptr())
    cp.q0, cp.mass0, cp.p0c = hp.q0, hp.mass0, hp.p0c
    cp.beta0, cp.gamma0, cp.energy0 = hp.beta0, hp.gamma0, hp.energy0
    opts = _cabi.TrackOptions()
    opts.num_turns = turns
    _cabi.check(_cabi.lib().xlb_track_host(C.byref(lat), C.byref(cp), C.byref(opts)))
    got = hp.to_numpy()
    for k in H.COORDS + ("state", "at_element", "at_turn"):
        assert np.array_equal(got[k], results["split"][k], equal_nan=True), k


def test_lhc_beambeam_c3_one_turn_against_oracle():
    """BASELINE config C3 lattice (72 BeamBeam4D + 2 BeamBeam6D x 15 slices), 300-particle
    subsample x 1 turn (the oracle needs ~1 s per particle-lens for the 6D lenses)."""
    from xline_b200 import configs

    line, cols, p0c, m0 = configs.config_lhc_beambeam(300)
    p = make_particles(cols, p0c, m0)
    line.track(p, num_turns=1)
    got = p.to_numpy()
    ref = H.run_oracle(line.to_specs(), cols, p0c, m0, num_turns=1)
    assert np.array_equal(got["state"], ref["state"])
    for k in H.COORDS:
        assert H.scaled_err(got[k], ref[k]) <= FAST_FULL_TURN_TOL, (k, H.scaled_err(got[k], ref[k]))


def test_lhc_beambeam_c3_unstable_particles_go_non_finite_like_the_oracle():
    """The C3 lattice has no apertures: a particle far outside the dynamic aperture is never
    removed, its coordinates overflow and it stays in the beam as NaN -- in the reference's
    NumPy path and here alike.  The 64 highest-amplitude particles of the 1 M-particle C3 beam,
    10 turns: the same particles (one, particle 948 199) end non-finite, nobody is lost."""
    from xline_b200 import configs

    line, cols, p0c, m0 = configs.config_lhc_beambeam(1_000_000)
    amp = np.hypot(cols["x"] / 2e-4, cols["y"] / 2e-4) + np.hypot(cols["px"] / 2e-6, cols["py"] / 2e-6)
    idx = np.argsort(-amp)[:64]
    sub = {k: np.ascontiguousarray(v[idx]) for k, v in cols.items()}
    p = make_particles(sub, p0c, m0)
    line.track(p, num_turns=10)
    got = p.to_numpy()
    with np.errstate(all="ignore"):
        ref = H.run_oracle(line.to_specs(), {k: v for k, v in sub.items() if k != "particle_id"}, p0c, m0,
                           num_turns=10)
    bad_got = ~np.isfinite(got["x"])
    bad_ref = ~np.isfinite(ref["x"])
    assert np.array_equal(bad_got, bad_ref), (idx[bad_got], idx[bad_ref])
    assert 948_199 in idx[bad_ref]
    assert np.array_equal(got["state"], ref["state"]) and (got["state"] == 1).all()
    assert np.array_equal(got["at_turn"], ref["at_turn"])


def test_psb_like_c5_space_charge_and_monitor_against_oracle():
    """C5 stand-in (xline_b200.configs.config_psb_like): 128 SCQGaussProfile kicks per turn,
    DipoleEdge, curved dipoles, the PSB aperture mix, a cavity and a BeamMonitor."""
    from xline_b200 import configs

    n, turns = 400, 4
    line, cols, p0c, m0 = configs.config_psb_like(n, monitor_stores=turns, monitor_ids=n)
    cols["x"][:5] *= 8.0  # make sure some particles hit the apertures
    p = make_particles(cols, p0c, m0)
    line.track(p, num_turns=turns)
    got = p.to_numpy()
    monitors = {}
    ref = H.run_oracle(line.to_specs(), cols, p0c, m0, num_turns=turns, monitors=monitors)
    assert np.array_equal(got["state"], ref["state"]) and (ref["state"] == 0).sum() > 0
    assert np.array_equal(got["at_element"], ref["at_element"])
    assert np.array_equal(got["at_turn"], ref["at_turn"])
    for k in H.COORDS:
        assert H.scaled_err(got[k], ref[k]) <= 1e-12, (k, H.scaled_err(got[k], ref[k]))
    mon = [el for el in line.elements if type(el).__name__ == "BeamMonitor"][0]
    store = list(monitors.values())[0]
    written = store["at_turn"] >= 0
    for k in ("x", "px", "y", "py", "zeta", "delta"):
        g = mon.data[k].cpu().numpy()
        assert np.array_equal(np.isnan(g), ~written)
        assert H.scaled_err(g[written], store[k][written]) <= 1e-12, k


def test_petra_like_c4_against_oracle():
    """C4 stand-in (config_petra_like): 6 GeV electrons, 4-slice thin quads/bends, DriftExact,
    sextupoles, 500 MHz cavities and RFMultipoles, dynamic-aperture grid beam."""
    from xline_b200 import configs

    line, cols, p0c, m0 = configs.config_petra_like(400)
    p = make_particles(cols, p0c, m0)
    line.track(p, num_turns=3)
    got = p.to_numpy()
    ref = H.run_oracle(line.to_specs(), cols, p0c, m0, num_turns=3)
    assert np.array_equal(got["state"], ref["state"]) and (ref["state"] == 0).sum() > 0
    assert np.array_equal(got["at_turn"], ref["at_turn"])
    alive = ref["state"] == 1
    for k in H.COORDS:
        # amplitude scan up to the dynamic aperture: the outermost (chaotic) orbits amplify the
        # rounding differences of the fast kernel to ~1e-10 within 3 turns
        assert H.scaled_err(got[k][alive], ref[k][alive]) <= 5e-10, (k, H.scaled_err(got[k][alive], ref[k][alive]))
    p2 = make_particles(cols, p0c, m0)
    line.track(p2, num_turns=3, strict=True)
    got2 = p2.to_numpy()
    assert np.array_equal(got2["state"], ref["state"])
    for k in H.COORDS:  # reference operation order: sin/cos/sqrt ulp differences only
        assert H.scaled_err(got2[k][alive], ref[k][alive]) <= 1e-12, (k, H.scaled_err(got2[k][alive], ref[k][alive]))


# ------------------------------------------------------------------ edge cases
def test_edge_cases_empty_single_all_lost_nan():
    import xline_b200 as xl

    line = xl.Line([xl.Drift(length=1.0), xl.Multipole(knl=[0, 0.1]),
                    xl.LimitRect(min_x=-1e-2, max_x=1e-2, min_y=-1e-2, max_y=1e-2), xl.Drift(length=2.0)])
    # empty particle set and zero turns: no launch, no error
    p0 = xl.Particles(p0c=1e9, x=np.zeros(0))
    line.track(p0, num_turns=3)
    assert len(p0) == 0
    p1 = xl.Particles(p0c=1e9, x=[1e-3, 2e-3])
    line.track(p1, num_turns=0)
    assert p1.at_turn.tolist() == [0, 0] and p1.x.tolist() == [1e-3, 2e-3]
    # one particle given as scalars (reference tests/test_track.py:57-61): state flips to 0
    ps = xl.Particles(p0c=1e9, x=1.0, y=1.0)
    line.track(ps)
    assert ps.state.tolist() == [0] and ps.at_element.tolist() == [2] and ps.at_turn.tolist() == [0]
    # NaN compares false in every bound -> lost at the first aperture, coordinates kept
    pn = xl.Particles(p0c=1e9, x=[np.nan, 1e-3, 0.5], y=[0.0, 0.0, 0.0])
    line.track(pn, num_turns=2)
    assert pn.state.tolist() == [0, 1, 0] and pn.at_turn.tolist() == [0, 2, 0]
    assert np.isnan(pn.x[0].item()) and pn.at_element.tolist() == [2, 0, 2]
    # everything lost in the first turn; tracking on is a no-op on the frozen particles
    pa = xl.Particles(p0c=1e9, x=np.full(700, 0.5))
    line.loss_tally.zero_()  # the tally accumulates over calls on the same Line
    line.track(pa, num_turns=2, turns_per_launch=1)
    snap = pa.to_numpy()
    line.track(pa, num_turns=5, turns_per_launch=2)
    again = pa.to_numpy()
    assert (snap["state"] == 0).all() and int(line.loss_tally[2]) == 700
    for k in snap:
        assert np.array_equal(snap[k], again[k], equal_nan=True), k
    # empty line: only the turn counter advances
    pe = xl.Particles(p0c=1e9, x=[1e-3])
    xl.Line([]).track(pe, num_turns=4)
    assert pe.at_turn.tolist() == [4] and pe.x.tolist() == [1e-3]
    # non-contiguous columns are made contiguous, values preserved
    pc = xl.Particles(p0c=1e9, x=np.linspace(0, 1e-3, 10))
    pc.x = torch.linspace(0, 1e-3, 20, dtype=torch.float64, device="cuda")[::2]
    before = pc.x.clone()
    xl.Line([xl.XYShift(dx=1e-4)]).track(pc)
    assert torch.equal(pc.x, before - 1e-4)


def test_monitor_rolling_and_skip():
    import xline_b200 as xl

    n, turns = 64, 11
    mon = xl.BeamMonitor(num_stores=2, start=1, skip=3, min_particle_id=0, max_particle_id=n - 1,
                         is_rolling=True)
    line = xl.Line([xl.Drift(length=1.0), mon])
    rng = np.random.default_rng(2)
    cols = dict(x=rng.normal(0, 1e-3, n), px=rng.normal(0, 1e-4, n))
    p = make_particles(cols, 1e9, 938.27208816e6)
    line.track(p, num_turns=turns)
    monitors = {}
    H.run_oracle(line.to_specs(), cols, 1e9, 938.27208816e6, num_turns=turns, monitors=monitors)
    store = monitors[1]
    # stores happen at turns 1, 4, 7, 10 -> slots 0, 1, 0, 1: the last two survive
    assert sorted(set(store["at_turn"].ravel().tolist())) == [7, 10]
    assert np.array_equal(mon.data["at_turn"].cpu().numpy(), store["at_turn"].astype(float))
    assert np.array_equal(mon.data["x"].cpu().numpy(), store["x"])


def test_petra4_c4_real_lattice_against_oracle():
    """BASELINE config C4 lattice: examples/petra4/h7ba_n8.seq read without MAD-X
    (xline_b200.madx_input), 4-slice TEAPOT thin lenses, 31 025 elements; dynamic-aperture
    grid, 2 turns."""
    from xline_b200 import configs

    line, cols, p0c, m0 = configs.config_petra4(300, x_max=6e-3, y_max=3e-3)
    line.append_element(__import__("xline_b200").LimitEllipse(a=8e-3, b=4e-3), "scraper")
    p = make_particles(cols, p0c, m0)
    line.track(p, num_turns=2)
    got = p.to_numpy()
    ref = H.run_oracle(line.to_specs(), cols, p0c, m0, num_turns=2)
    assert np.array_equal(got["state"], ref["state"]) and np.array_equal(got["at_turn"], ref["at_turn"])
    alive = ref["state"] == 1
    assert 0 < alive.sum()
    for k in H.COORDS:
        scale_ok = H.scaled_err(got[k][alive], ref[k][alive])
        if k == "zeta":
            # zeta of an exact drift is L*(rvv - (1+delta)/pz): a difference of two numbers of
            # the size of the path length, so its rounding noise is absolute, ~1e-16 x the
            # distance travelled (2 x 2301.6 m here), not relative to the (tiny) zeta spread
            assert np.max(np.abs(got[k][alive] - ref[k][alive])) <= 5e-12, k
            continue
        if k == "delta":
            # the grid beam starts at delta = 0: delta is only what the cavities add (~1e-6),
            # and their phase sees the zeta noise above (k * 4e-13 m -> 1e-5 eV of 6 GeV)
            assert np.max(np.abs(got[k][alive] - ref[k][alive])) <= 1e-13, k
            continue
        assert scale_ok <= 1e-10 or np.max(np.abs(got[k][alive] - ref[k][alive])) <= 1e-18, (k, scale_ok)
    p2 = make_particles(cols, p0c, m0)
    line.track(p2, num_turns=2, strict=True)
    got2 = p2.to_numpy()
    assert np.array_equal(got2["state"], ref["state"])
    # strict kernel: one turn of this lattice is bit-identical to the oracle (checked on the
    # B200); over two turns the last-ulp difference between CUDA's and glibc's sin() in the
    # cavities reaches rvv and, through L*rvv, zeta at the 1e-15 m level
    for k in H.COORDS:
        e2 = H.scaled_err(got2[k][alive], ref[k][alive])
        if k == "zeta":
            assert np.max(np.abs(got2[k][alive] - ref[k][alive])) <= 5e-14, k
            continue
        assert e2 <= 1e-13 or np.max(np.abs(got2[k][alive] - ref[k][alive])) <= 1e-16, (k, e2)


def test_trace_elem_by_elem_matches_oracle_element_by_element():
    """Device element-by-element trace (xline/line.py:97-108) against the oracle stepping the
    same line one element at a time -- the replay examples/lhc/benchmark.py:28-48 does against
    SixTrack dumps."""
    from oracle import xline_oracle as xo

    m, specs, cols, _ = H.load_case("line_mixed_3turns")
    line = build_line(specs)
    n = len(cols["x"])
    for strict in (True, False):
        p = make_particles(cols, m["p0c"], m["mass0"])
        trace = line.trace_elem_by_elem(p, strict=strict).cpu().numpy()
        assert trace.shape == (len(line) + 1, 6, n)
        o = xo.OracleParticles(n, p0c=m["p0c"], mass0=m["mass0"], **cols)
        for f, k in enumerate(H.COORDS):
            assert np.array_equal(trace[0, f], cols[k])
        for i, (name, fld) in enumerate(specs):
            rec = xo.TRACKERS[name](o, fld)
            alive_ids = o.particle_id
            row = trace[i + 1]
            gone = np.ones(n, dtype=bool)
            gone[alive_ids] = False
            assert np.isnan(row[:, gone]).all(), (i, name)          # lost: no more rows written
            for f, k in enumerate(H.COORDS):
                got, want = row[f, alive_ids], getattr(o, k)
                if strict and name not in ("Cavity", "RFMultipole"):
                    err = np.max(np.abs(got - want)) if len(want) else 0.0
                    assert err <= 4e-16 * max(np.max(np.abs(want)), 1e-300) * 8 or np.array_equal(got, want), (i, name, k)
                else:
                    assert H.rel_err(got, want) <= 1e-12 or np.max(np.abs(got - want)) <= 1e-18, (i, name, k)
        # the particles themselves ended where a normal one-turn track puts them
        q = make_particles(cols, m["p0c"], m["mass0"])
        line.track(q, num_turns=1, strict=strict)
        a, b = p.to_numpy(), q.to_numpy()
        for k in ("state", "at_element", "at_turn"):
            assert np.array_equal(a[k], b[k])


def test_trace_on_lhc_first_particles():
    from xline_b200 import configs

    line, cols, p0c, m0 = configs.config_lhc(2000)
    p = make_particles(cols, p0c, m0)
    trace = line.trace_elem_by_elem(p, max_particles=8)
    assert trace.shape == (len(line) + 1, 6, 8)
    last = trace[-1].cpu().numpy()
    q = make_particles(cols, p0c, m0)
    line.merge_multipoles = False
    line.track(q, num_turns=1)
    ref = q.to_numpy()
    alive = ref["state"][:8] == 1
    for f, k in enumerate(H.COORDS):
        assert np.array_equal(last[f][alive], ref[k][:8][alive]), k   # same maps, element by element


def test_full_size_c2_schedule_invariance():
    """BASELINE C2 at its full particle count (1 M): the production schedule (persistent CTAs,
    work queue, automatic segmentation with survivor compaction) gives bit-identical particles
    to one plain launch -- the result cannot depend on how the work was cut."""
    from xline_b200 import configs

    n, turns = 1_000_000, 12
    line, cols, p0c, m0 = configs.config_lhc(n)
    p1 = make_particles(cols, p0c, m0)
    line.track(p1, num_turns=turns, turns_per_launch=4)            # queue + 3 launches + compaction
    t1 = line.loss_tally.clone()
    line.loss_tally.zero_()
    p2 = make_particles(cols, p0c, m0)
    line.track(p2, num_turns=turns, turns_per_launch=-1, turns_per_item=-1)   # one plain launch
    assert torch.equal(t1, line.loss_tally)
    lost = int((p1.state == 0).sum())
    assert 0 < lost < n and int(t1.sum()) == lost
    for k, a in p1._columns():
        b = dict(p2._columns())[k]
        if k == "s":
            assert torch.allclose(a, b, rtol=1e-11, atol=0)
        else:
            assert torch.equal(a, b) or torch.equal(torch.nan_to_num(a), torch.nan_to_num(b)), k
    assert int(p1.at_turn.sum()) == int(p2.at_turn.sum())


def test_inverse_elements_return_to_start():
    """Domain property at size: every thin map followed by its inverse restores the beam
    (drifts exactly in x, y up to rounding; kicks to 1 ulp of the kick)."""
    import xline_b200 as xl

    n = 500_000
    rng = np.random.default_rng(9)
    cols = dict(x=rng.normal(0, 1e-3, n), px=rng.normal(0, 1e-4, n), y=rng.normal(0, 1e-3, n),
                py=rng.normal(0, 1e-4, n), zeta=rng.normal(0, 0.05, n), delta=rng.normal(0, 3e-4, n))
    knl, ksl = [1e-4, 0.02, 1.5, 30.0], [0.0, 0.01, -0.7]
    line = xl.Line([
        xl.Drift(length=3.7), xl.Drift(length=-3.7),
        xl.Multipole(knl=knl, ksl=ksl), xl.Multipole(knl=[-k for k in knl], ksl=[-k for k in ksl]),
        xl.XYShift(dx=1e-4, dy=-2e-4), xl.XYShift(dx=-1e-4, dy=2e-4),
        xl.SRotation(angle=23.0), xl.SRotation(angle=-23.0),
        xl.DipoleEdge(h=0.01, e1=0.1), xl.DipoleEdge(h=-0.01, e1=0.1),
    ])
    line.merge_multipoles = False
    p = make_particles(cols, 7e12, 938.27208816e6)
    line.track(p, num_turns=3)
    got = p.to_numpy()
    for k in H.COORDS:  # a few ulp of the beam size after 3 x 10 maps
        assert np.max(np.abs(got[k] - cols[k])) <= 1e-14 * np.max(np.abs(cols[k])), k
    assert np.array_equal(got["delta"], cols["delta"])


def test_work_queue_with_strict_kernel_and_monitor():
    """The queue schedule with the strict kernel and a BeamMonitor in the line: monitor slots,
    turn bookkeeping and particles identical to the plain launch."""
    import xline_b200 as xl
    from xline_b200 import configs

    n, turns = 160_000, 7
    base, cols, p0c, m0 = configs.config_fodo(n)
    mon = xl.BeamMonitor(num_stores=turns, start=0, skip=1, min_particle_id=100, max_particle_id=1123)
    els = list(base.elements) + [xl.LimitEllipse(a=3.5e-3, b=3.5e-3), mon]
    outs = []
    for tpi in (-1, 2):
        line = xl.Line(els)
        p = make_particles(cols, p0c, m0)
        line.track(p, num_turns=turns, strict=True, turns_per_item=tpi, particles_per_thread=1,
                   threads_per_block=128)
        outs.append((p.to_numpy(), {k: v.clone() for k, v in mon.data.items()}))
    (a, ma), (b, mb) = outs
    assert 0 < (a["state"] == 0).sum() < n
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=True), k
    for k in ma:
        assert torch.equal(torch.nan_to_num(ma[k], nan=-7.0), torch.nan_to_num(mb[k], nan=-7.0)), k
    assert int((~torch.isnan(ma["x"])).sum()) > 1000


@pytest.mark.parametrize("seed", range(40))
def test_random_lines_on_the_gpu(seed):
    """The packer fuzz of tests/test_packed_format.py through the kernels: random thin-lens lines
    (every block shape, merged records, small chunks, losses), three turns, strict and fast
    kernels against the oracle."""
    from tests.test_packed_format import _random_line

    rng = np.random.default_rng(1000 + seed)
    line = _random_line(rng)
    line.chunk_words = int(rng.choice([32, 64, 256]))
    n = 150
    cols = dict(x=rng.normal(0, 8e-4, n), px=rng.normal(0, 1e-4, n), y=rng.normal(0, 8e-4, n),
                py=rng.normal(0, 1e-4, n), zeta=rng.normal(0, 0.05, n), delta=rng.normal(0, 3e-4, n))
    p0c, m0 = 26e9, 938.27208816e6
    with np.errstate(all="ignore"):
        ref = H.run_oracle(line.to_specs(), cols, p0c, m0, num_turns=3)
    for strict in (True, False):
        p = make_particles(cols, p0c, m0)
        line.track(p, num_turns=3, strict=strict)
        got = p.to_numpy()
        for k in ("state", "at_element", "at_turn"):
            assert np.array_equal(got[k], ref[k]), (k, strict)
        for k in H.COORDS:
            assert H.scaled_err(got[k], ref[k]) <= (1e-13 if strict else 1e-10), (k, strict)


def test_edited_line_gets_fresh_buffers_and_repacks():
    """ADVICE r1: (a) a line that grew since the last call must not keep its old, smaller loss
    tally; (b) torch.device("cuda") vs "cuda:0" must not reset the tallies on every call; (c) a
    field edited in place (the reference reads fields on every track call) must be tracked through."""
    import xline_b200 as xl
    from xline_b200 import configs

    n = 2000
    base, cols, p0c, m0 = configs.config_fodo(n)
    line = xl.Line(list(base.elements) + [xl.LimitRect(min_x=-2e-3, max_x=2e-3, min_y=-2e-3, max_y=2e-3)])
    p = xl.Particles(p0c=p0c, mass0=m0, device="cuda", **cols)  # un-indexed device on purpose
    line.track(p, num_turns=2)
    t1 = line.loss_tally.clone()
    lost1 = int((p.state == 0).sum())
    assert int(t1.sum()) == lost1 > 0
    line.track(p, num_turns=2)
    assert int(line.loss_tally.sum()) == int((p.state == 0).sum()) >= lost1  # accumulated, not re-created
    # (a) grow the line the way reference code does
    tight = xl.LimitEllipse(a=1e-3, b=1e-3)
    line.elements.append(tight)
    line.element_names.append("tight")
    line.track(p, num_turns=1)
    assert line.loss_tally.numel() == len(line.elements)
    assert int(line.loss_tally[-1]) > 0 and int(line.loss_tally[-1]) == int((p.at_element == len(line) - 1).sum())
    # (c) open the aperture in place: nobody is lost there any more
    before = int((p.state == 0).sum())
    tight.a = 1.0
    tight.b = 1.0
    line.elements[-2].max_x = 1.0
    line.elements[-2].min_x = -1.0
    line.elements[-2].max_y = 1.0
    line.elements[-2].min_y = -1.0
    line.track(p, num_turns=3)
    assert int((p.state == 0).sum()) == before
    # list-valued field edited item by item
    quad = [e for e in line.elements if isinstance(e, xl.Multipole) and len(e.knl) > 1][0]
    ref = xl.Particles(p0c=p0c, mass0=m0, **cols)
    got = xl.Particles(p0c=p0c, mass0=m0, **cols)
    open_line = xl.Line([e for e in line.elements if not isinstance(e, (xl.LimitRect, xl.LimitEllipse))])
    open_line.track(ref, num_turns=1)
    quad.knl[1] = quad.knl[1] * 1.5
    open_line.track(got, num_turns=1)
    assert not torch.equal(ref.px, got.px)
    fresh = xl.Particles(p0c=p0c, mass0=m0, **cols)
    xl.Line([e.copy() for e in open_line.elements]).track(fresh, num_turns=1)
    assert torch.equal(fresh.px, got.px) and torch.equal(fresh.x, got.x)


def test_element_track_loop_is_one_pass_of_the_line():
    """`for el in line.elements: el.track(p)` (the reference's loop, xline/line.py:89-95) equals
    Line.track(p) without touching the turn counter; track_elem_by_elem records the index of the
    element in the line for a particle lost on the way."""
    import xline_b200 as xl
    from xline_b200 import configs

    n = 600
    base, cols, p0c, m0 = configs.config_fodo(n)
    els = list(base.elements) + [xl.LimitRect(min_x=-1.5e-3, max_x=1.5e-3, min_y=-1.5e-3, max_y=1.5e-3)]
    line = xl.Line(els)
    a = make_particles(cols, p0c, m0)
    line.track(a, num_turns=1, strict=True)
    b = make_particles(cols, p0c, m0)
    for el in line.elements:
        el.track(b)
    assert int(b.at_turn.max()) == 0
    c = make_particles(cols, p0c, m0)
    line.track_elem_by_elem(c)
    ga, gb, gc = a.to_numpy(), b.to_numpy(), c.to_numpy()
    assert (ga["state"] == 0).sum() > 0
    for k in ("state",) + tuple(H.COORDS):
        assert np.array_equal(ga[k], gc[k], equal_nan=True) or H.scaled_err(gc[k], ga[k]) < 1e-12, k
        assert np.array_equal(gb["state"], ga["state"])
    assert np.array_equal(gc["at_element"], ga["at_element"])
    assert int(gc["at_turn"].max()) == 0


@pytest.mark.parametrize("config", ["lhc", "petra4"])
@pytest.mark.parametrize("with_chi", [False, True])
def test_horizontal_bend_flag_changes_no_bit(config, with_chi):
    """XLB_HDR_HX_ONLY (curved block records with hyl == 0: the hyl terms of elements.py:139-154
    are left out) against the same lattice packed without the flag (general formula): every
    column bit for bit, with and without a chi column (one-species and general kernel family)."""
    from xline_b200 import configs

    n = 30_000
    line, cols, p0c, m0 = (configs.config_lhc if config == "lhc" else configs.config_petra4)(n)
    cols = dict(cols)
    if with_chi:
        cols["chi"] = 1.0 + 0.01 * np.random.default_rng(3).standard_normal(n)
    flagged = sum(1 for w in line.pack().words if (int(w) >> 31) & 1 and (int(w) & 0xC4) == 0x84)
    outs = []
    for flag in (True, False):
        line.flag_horizontal_bends = flag
        p = make_particles(cols, p0c, m0)
        line.track(p, num_turns=2)
        outs.append(p.to_numpy())
    line.flag_horizontal_bends = True
    assert flagged > 100  # (header words only look like this by construction: tag 0x84.., bit 31)
    for k in outs[0]:
        assert np.array_equal(outs[0][k], outs[1][k], equal_nan=True), k


def test_one_chunk_lattice_resident_in_shared_memory_equals_the_ring():
    """A lattice that fits one chunk is copied to shared memory once per work item and stays
    there; packed into many small chunks the same lattice goes through the TMA ring turn by
    turn.  Same bits, losses included, with and without the work queue."""
    import xline_b200 as xl
    from xline_b200 import configs

    line, cols, p0c, m0 = configs.config_fodo(150_000)
    line = xl.Line(list(line.elements) + [xl.LimitRect(min_x=-3e-3, max_x=3e-3, min_y=-3e-3, max_y=3e-3),
                                          xl.LimitEllipse(a=3.5e-3, b=3.2e-3)])
    outs = []
    for chunk_words, tpi in ((None, -1), (None, 5), (32, -1), (32, 5)):
        line.chunk_words = chunk_words
        p = make_particles(cols, p0c, m0)
        line.track(p, num_turns=23, turns_per_item=tpi)
        assert (line.pack().n_chunks == 1) == (chunk_words is None)
        outs.append(p.to_numpy())
    assert 0 < (outs[0]["state"] == 0).sum() < len(outs[0]["x"])
    for o in outs[1:]:
        for k in o:
            if k == "s":
                assert np.allclose(outs[0][k], o[k], rtol=1e-12, atol=0)
            else:
                assert np.array_equal(outs[0][k], o[k], equal_nan=True), k


@pytest.mark.parametrize("strict", [False, True])
def test_idle_lanes_are_parked_and_never_counted(strict):
    """Lanes whose particle is gone keep running with their warp, parked at the origin.  Here a
    fifth of the beam is lost over 30 different turns at four kinds of aperture, dipole kicks move
    whatever sits at the origin, and one aperture does not contain the origin of its (shifted)
    frame at all, so lanes parked there wander through the ring and trip apertures again: loss flags, at_element, at_turn and the tallies
    must still be the oracle's -- every lost particle counted once, nothing else counted."""
    import xline_b200 as xl

    n, turns = 3000, 60
    rng = np.random.default_rng(11)
    els = [
        xl.Multipole(knl=[3e-5, 0.4], ksl=[-1e-5]), xl.LimitRect(min_x=-4e-3, max_x=4e-3, min_y=-4e-3, max_y=4e-3),
        xl.Drift(length=1.5),
        xl.Multipole(knl=[-1e-5, -0.4, 12.0]), xl.LimitEllipse(a=5e-3, b=4.5e-3), xl.Drift(length=1.5),
        xl.LimitRect(min_x=-3.0e-3, max_x=9e-3, min_y=-9e-3, max_y=9e-3),   # asymmetric box
        xl.Multipole(knl=[1e-3], hxl=1e-3, length=1.0), xl.LimitRectEllipse(max_x=6e-3, max_y=6e-3, a=7e-3, b=6.5e-3),
        xl.Drift(length=0.7),
        # in the shifted frame the box does not contain the origin: a lane parked here is flagged
        # again and again
        xl.XYShift(dx=3e-3, dy=0.0), xl.LimitRect(min_x=-6e-3, max_x=-1e-4, min_y=-9e-3, max_y=9e-3),
        xl.XYShift(dx=-3e-3, dy=0.0),
    ]
    line = xl.Line(els)
    cols = dict(x=rng.normal(0, 1.0e-3, n), px=rng.normal(0, 2e-4, n), y=rng.normal(0, 1.0e-3, n),
                py=rng.normal(0, 2e-4, n), zeta=rng.normal(0, 0.05, n), delta=rng.normal(0, 3e-4, n))
    p0c, m0 = 6.5e12, 938.272e6
    for ppt in (1, 4):
        line.invalidate()
        p = make_particles(cols, p0c, m0)
        line.track(p, num_turns=turns, strict=strict, particles_per_thread=ppt)
        got = p.to_numpy()
        ref = H.run_oracle(line.to_specs(), cols, p0c, m0, num_turns=turns)
        lost = ref["state"] == 0
        assert 0.15 * n < lost.sum() < n  # a fifth of the beam goes, over many turns
        assert len(np.unique(ref["at_turn"][lost])) > 15
        for k in ("state", "at_element", "at_turn"):
            assert np.array_equal(got[k], ref[k]), k
        tally = line.loss_tally.cpu().numpy()
        assert tally.sum() == lost.sum()
        assert np.array_equal(tally, np.bincount(ref["at_element"][lost], minlength=len(line)))
        for k in H.COORDS + ("s",):
            if strict:
                assert np.array_equal(got[k], ref[k]), k
            else:
                assert H.scaled_err(got[k], ref[k]) < 1e-9, k
