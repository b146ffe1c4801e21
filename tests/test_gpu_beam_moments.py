"""Beam moments on the GPU (csrc/moments.cu, xlb_track_device_moments): the accuracy bound
against exact rational sums, bitwise reproducibility under every schedule knob, equality with
the same job cut into calls with a snapshot between them, and tracking left untouched."""
import numpy as np
import pytest
import torch

from tests import moments_oracle as MO

pytestmark = pytest.mark.gpu


def _make(cols, p0c, m0):
    import xline_b200 as xl

    return xl.Particles(p0c=p0c, mass0=m0, device="cuda", **cols)


def _bits(t):
    return t.contiguous().view(torch.int64)


def _same(a, b):
    return torch.equal(_bits(a), _bits(b))


def _check_bound(words, cols, state):
    exact = MO.exact_store(cols, state)
    errs = MO.store_errors(words, exact)
    assert max(errs) <= MO.bound(len(state)), float(max(errs))
    return exact


def test_snapshot_meets_the_bound_with_lost_and_non_finite_particles():
    import xline_b200 as xl

    n = 100_000
    rng = np.random.default_rng(5)
    cols = {k: rng.normal(0.3, s, n) for k, s in zip(MO.COORDS, (1e-3, 1e-5, 2e-3, 3e-5, 0.1, 1e-3))}
    cols["x"][::97] *= 1e6          # wide dynamic range of the terms
    state = np.ones(n, dtype=np.int64)
    state[::5] = 0                   # lost
    cols["px"][1::13] = np.nan       # alive with NaN, or lost with NaN
    cols["zeta"][2::17] = np.inf
    cols["delta"][3::19] = -np.inf
    cols["y"][::10] = np.nan         # every other one of these is lost (state[::5] == 0)
    p = xl.Particles(p0c=1e9, device="cuda", state=state, **cols)
    m = xl.beam_moments(p)
    torch.cuda.synchronize()
    words = m.data[0].cpu().tolist()
    exact = _check_bound(words, cols, state)
    assert 0 < exact["n_nonfinite"] and 0 < exact["n"] < n
    assert int(m.count[0]) == exact["n"] and int(m.n_nonfinite[0]) == exact["n_nonfinite"]
    # the reduction over slots does not depend on anything but the columns
    assert _same(xl.beam_moments(p).data, m.data)


def test_small_and_empty_beams():
    import xline_b200 as xl

    for n in (0, 1, 2047, 2048, 2049, 3 * 2048 + 1):
        rng = np.random.default_rng(n)
        cols = {k: rng.normal(0, 1e-3, n) for k in MO.COORDS}
        p = xl.Particles(p0c=1e9, device="cuda", n=n, **cols) if n else xl.Particles(
            p0c=1e9, device="cuda", **{k: np.zeros(0) for k in MO.COORDS})
        m = xl.beam_moments(p)
        _check_bound(m.data[0].cpu().tolist(), cols, np.ones(n, dtype=np.int64))


def test_multi_level_fold_is_exact_on_exact_sums():
    """More than 2048 tiles, so the tile sums are folded twice: on coordinates k / 1024 with small
    integers k every sum is an integer multiple of 2^-20 below 2^53, which double-double holds
    exactly -- the store must equal the integer sums, so every slot entered exactly once."""
    import xline_b200 as xl

    n = 2048 * 2048 + 12_345
    rng = np.random.default_rng(8)
    ks = {k: rng.integers(-1000, 1001, n) for k in MO.COORDS}
    state = np.where(rng.random(n) < 0.1, 0, 1)
    p = xl.Particles(p0c=1e9, device="cuda", state=state, **{k: v / 1024.0 for k, v in ks.items()})
    words = xl.beam_moments(p).data[0].cpu().numpy()
    ok = state == 1
    assert words[0] == ok.sum() and words[1] == 0
    for q, (u, v) in enumerate(MO.PAIRS):
        a = ks[MO.COORDS[u]][ok]
        want = a.sum() / 1024.0 if v is None else int((a * ks[MO.COORDS[v]][ok]).sum()) / 2.0 ** 20
        assert words[2 + 2 * q] == want and words[3 + 2 * q] == 0.0, q


def _track(line, cols, p0c, m0, turns, moments=None, **kw):
    p = _make(cols, p0c, m0)
    line.track(p, num_turns=turns, moments=moments, **kw)
    torch.cuda.synchronize()
    return p


def test_moments_bitwise_across_kernels_and_schedules():
    import xline_b200 as xl
    from xline_b200 import configs

    n, turns = 60_000, 12
    line, cols, p0c, m0 = configs.config_lhc(n)
    ref = None
    cases = [dict(particles_per_thread=k) for k in (1, 2, 3, 4)]
    cases += [dict(turns_per_launch=t) for t in (-1, 1, 7, 0)]
    cases += [dict(turns_per_item=t) for t in (-1, 1, 3)]
    cases += [dict(threads_per_block=256, particles_per_thread=2)]
    for kw in cases:
        m = xl.BeamMoments(turns + 1)
        _track(line, cols, p0c, m0, turns, moments=m, **kw)
        if ref is None:
            ref = m.data.clone()
            assert not torch.isnan(ref).any()
        assert _same(m.data, ref), kw


def test_heavy_loss_beam_with_compaction_bitwise():
    import xline_b200 as xl
    from xline_b200 import configs

    n, turns = 40_000, 12      # the ramp is on from 32 768 particles
    line, _, p0c, m0 = configs.config_lhc(1000)
    cols = configs.gaussian_beam(n, 2, 0, sx=3e-4, spx=3e-6, amp_max=12.0)
    out = []
    for kw in (dict(turns_per_launch=4, compact_threshold=1e-4), dict(turns_per_launch=-1, turns_per_item=-1),
               dict()):
        m = xl.BeamMoments(turns + 1, skip=1)
        p = _track(line, cols, p0c, m0, turns, moments=m, **kw)
        out.append(m.data.clone())
        assert line.last_stats["compactions"] >= (1 if kw.get("turns_per_launch") == 4 else 0)
    lost = int((p.state == 0).sum())
    assert 0.5 * n < lost < n
    assert int(out[0][-1, 0]) == n - lost - int(((p.state == 1) & ~torch.isfinite(p.x)).sum())
    assert _same(out[0], out[1]) and _same(out[0], out[2])


def _configs():
    from xline_b200 import configs

    def c5():
        return configs.config_psb(4_000)

    return {
        "fodo": lambda: configs.config_fodo(5_000),
        "c2": lambda: configs.config_lhc(20_000),
        "c3": lambda: configs.config_lhc_beambeam(3_000),
        "c5": c5,
    }


@pytest.mark.parametrize("config,turns,start,skip", [("fodo", 20, 0, 3), ("c2", 9, 1, 2), ("c3", 4, 0, 1),
                                                     ("c5", 12, 2, 5)])
def test_track_with_moments_equals_calls_cut_at_the_store_turns(config, turns, start, skip):
    """One call with stores == the same job cut into calls of `skip` turns with a snapshot between
    them, and the particles bitwise those of tracking without stores."""
    import xline_b200 as xl

    line, cols, p0c, m0 = _configs()[config]()
    if config == "c3":
        assert line.pack(False).segments is not None  # 6D lenses as kernels of their own
    num_stores = (turns - start) // skip + 2          # the last one lies past num_turns
    m = xl.BeamMoments(num_stores, start=start, skip=skip)
    p = _track(line, cols, p0c, m0, turns, moments=m)
    plain = _track(line, cols, p0c, m0, turns)
    for k, a in p._columns():
        b = dict(plain._columns())[k]
        if k == "s":
            assert torch.allclose(a, b, rtol=1e-11, atol=0)
        else:
            assert _same(a, b), k

    q = _make(cols, p0c, m0)
    done, want = 0, []
    for t in m.turn.tolist():
        if t > turns:
            break
        if t > done:
            line.track(q, num_turns=t - done)
            done = t
        want.append(xl.beam_moments(q).data[0])
    want = torch.stack(want)
    assert _same(m.data[: len(want)], want)
    assert torch.isnan(m.data[len(want):]).all()
    assert int(m.count[0]) > 0


def test_strict_kernel_lhc_beam_meets_the_bound():
    import xline_b200 as xl
    from xline_b200 import configs

    n = 3_000
    line, cols, p0c, m0 = configs.config_lhc(n)
    m = xl.BeamMoments(2, start=0, skip=1)
    p = _track(line, cols, p0c, m0, 1, moments=m, strict=True)
    words = m.data.cpu().tolist()
    _check_bound(words[0], cols, np.ones(n, dtype=np.int64))
    got = p.to_numpy()
    _check_bound(words[1], {k: got[k] for k in MO.COORDS}, got["state"])
    # the strict kernel is the parity instrument: its coordinates against the oracle's
    from oracle import xline_oracle as xo

    o = xo.OracleParticles(n, p0c=p0c, mass0=m0, **cols)
    xo.line_track(line.to_specs(), o, 1)
    ref = xo.gather_full(o, n)
    assert np.array_equal(ref["state"], got["state"])
    exact = MO.exact_store({k: ref[k] for k in MO.COORDS}, ref["state"])
    assert exact["n"] == int(m.count[1])


def test_beam_lost_mid_call_still_writes_its_stores():
    import xline_b200 as xl

    n = 3_000
    rng = np.random.default_rng(2)
    cols = dict(x=rng.normal(0, 1e-5, n), y=rng.normal(0, 1e-5, n))
    # a dipole kick and a drift: x grows until the aperture takes every particle in turn 2
    line = xl.Line([xl.Multipole(knl=[-1e-4]), xl.Drift(length=5.0),
                    xl.LimitRect(min_x=-1e-3, max_x=1e-3, min_y=-1e-3, max_y=1e-3)])
    m = xl.BeamMoments(8, start=0, skip=1)
    p = _track(line, cols, 1e9, 938.27208816e6, 5, moments=m)
    assert int((p.state == 1).sum()) == 0 and (p.at_turn == 1).all()
    assert m.count.tolist()[:6] == [n, n, 0, 0, 0, 0]
    assert (m.data[2:6] == 0).all()
    assert torch.isnan(m.data[6:]).all()
    # num_turns == 0: only the store at turn 0
    m0 = xl.BeamMoments(3, start=0, skip=1)
    q = _track(line, cols, 1e9, 938.27208816e6, 0, moments=m0)
    assert int(m0.count[0]) == n and torch.isnan(m0.data[1:]).all() and (q.at_turn == 0).all()


def test_moments_refuse_a_trace_and_timed():
    import xline_b200 as xl

    line = xl.Line([xl.Drift(length=1.0)])
    p = xl.Particles(p0c=1e9, x=np.zeros(8), device="cuda")
    with pytest.raises(ValueError):
        line.track(p, moments=xl.BeamMoments(1), timed=True)
    trace = torch.zeros((1, 6, 8), dtype=torch.float64, device="cuda")
    with pytest.raises(ValueError):
        line.track(p, moments=xl.BeamMoments(1), _trace=trace)
    with pytest.raises(ValueError):
        line.track(p, moments=xl.BeamMoments(1, device="cpu"))
