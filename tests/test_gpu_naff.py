"""NAFF tunes on the GPU (xl.naff, xl.monitor_tunes): against the NumPy definition
(tests/naff_oracle.py), invalid signals, bitwise reproducibility across batches, argument checks,
and tunes of particles tracked on the GPU (linear PS Booster, octupole detuning, space-charge and
beam-beam footprints, a frequency map with losses)."""
import numpy as np
import pytest
import torch

from tests import naff_oracle as NO
from tests.test_naff import DETUNING_AMPLITUDES, detuning_columns, detuning_errors, mirror_signals, octupole_fodo

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _signals(T, n, seed):
    """Tones with a second harmonic (10 %), a coupling line (5 %), a closed-orbit offset and noise."""
    rng = np.random.default_rng(seed)
    nu1 = rng.uniform(0.02, 0.48, n)
    nu2 = rng.uniform(0.02, 0.48, n)
    ph = rng.uniform(0, 2 * np.pi, (3, n))
    amp = 10.0 ** rng.uniform(-6, -2, n)
    t = np.arange(T)[:, None]
    def line(nu, a, p):
        return a * np.cos(2 * np.pi * nu * t + p), -a * np.sin(2 * np.pi * nu * t + p)
    u1, p1 = line(nu1, 1.0, ph[0])
    u2, p2 = line(2 * nu1, 0.10, ph[1])
    u3, p3 = line(nu2, 0.05, ph[2])
    u = amp * (u1 + u2 + u3 + 0.3 + 1e-6 * rng.standard_normal((T, n)))
    pu = amp * (p1 + p2 + p3 - 0.1 + 1e-6 * rng.standard_normal((T, n)))
    return u, pu


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def assert_matches_oracle(q, a, ref, what=""):
    """The 1e-12 rule: tunes within 1e-12 and amplitudes within 1e-12 relative of the oracle, NaN
    where the oracle has NaN; signals whose two largest coarse bins are within 1e-9 (relative) are
    exempt and returned as a count."""
    rq, ra, near = ref
    q = q.cpu().numpy() if isinstance(q, torch.Tensor) else q
    a = a.cpu().numpy() if isinstance(a, torch.Tensor) else a
    assert np.array_equal(np.isnan(q), np.isnan(rq)), what
    assert np.array_equal(np.isnan(a), np.isnan(ra)), what
    ok = ~near & np.isfinite(rq)
    dq = np.abs(q[ok] - rq[ok])
    da = np.abs(a[ok] - ra[ok]) / np.maximum(np.abs(ra[ok]), 1e-300)
    assert dq.size == 0 or dq.max() <= 1e-12, (what, dq.max(), int(np.argmax(dq)))
    assert da.size == 0 or da.max() <= 1e-12, (what, da.max())
    return int((near & np.isfinite(rq)).sum())


@pytest.mark.parametrize("T", [64, 1000, 1024, 4096, 8192])
def test_naff_matches_the_oracle(T):
    n = 4096
    u, pu = _signals(T, n, seed=T)
    beta, alpha = 12.5, -0.7
    du, dpu = _dev(u), _dev(pu)
    q, a = _naff(du, dpu, beta, alpha)
    exempt = assert_matches_oracle(q, a, NO.naff(u, pu, beta, alpha), ("complex", T))
    qr, ar = _naff(du)
    exempt_r = assert_matches_oracle(qr, ar, NO.naff(u), ("real", T))
    print("T=%d: %d complex and %d real signals of %d exempt (near-tied coarse bins)" % (T, exempt, exempt_r, n))
    assert exempt + exempt_r <= n // 100


def _naff(u, pu=None, beta=1.0, alpha=0.0):
    import xline_b200 as xl

    q, a = xl.naff(u, pu, beta=beta, alpha=alpha)
    torch.cuda.synchronize()
    return q, a


def test_invalid_signals():
    T = 300
    u, pu = _signals(T, 6, seed=11)
    u[17, 0] = np.nan
    pu[250, 1] = np.inf
    u[:, 2] = 0.0
    pu[:, 2] = 0.0
    u[-1, 3] = -np.inf
    q, a = _naff(_dev(u), _dev(pu), 3.0, 0.5)
    q, a = q.cpu().numpy(), a.cpu().numpy()
    assert np.isnan(q[[0, 1, 2, 3]]).all()
    assert np.isnan(a[[0, 1, 3]]).all() and a[2] == 0.0
    assert np.isfinite(q[4:]).all() and np.isfinite(a[4:]).all()
    assert_matches_oracle(q, a, NO.naff(u, pu, 3.0, 0.5))
    qr, ar = _naff(_dev(u))
    assert_matches_oracle(qr, ar, NO.naff(u))
    q0, a0 = _naff(torch.zeros(T, 0, dtype=torch.float64, device=DEV))
    assert q0.shape == (0,) and a0.shape == (0,) and q0.device.type == "cuda"
    q1, a1 = _naff(_dev(u[:, 5:6]), _dev(pu[:, 5:6]), 3.0, 0.5)
    assert q1.item() == q[5] and a1.item() == a[5]


def test_tunes_stay_in_range():
    """Real signals whose root lies past 1/2 are folded like the oracle's; tones at the edges of
    the ranges stay inside [0, 1/2] (real) and [0, 1) (complex)."""
    x = mirror_signals()
    q, a = _naff(_dev(x))
    assert_matches_oracle(q, a, NO.naff(x))
    assert (q <= 0.5).all()
    rng = np.random.default_rng(7)
    T = 512
    nu = np.concatenate([rng.uniform(-3, 3, 200) / T, 0.5 + rng.uniform(-3, 3, 200) / T])
    t = np.arange(T)[:, None]
    qc, _ = _naff(_dev(np.cos(2 * np.pi * nu * t)), _dev(-np.sin(2 * np.pi * nu * t)))
    qr, _ = _naff(_dev(np.cos(2 * np.pi * nu * t + 1.0)))
    assert ((qc >= 0) & (qc < 1)).all()
    assert ((qr >= 0) & (qr <= 0.5)).all()


def test_bitwise_reproducible_across_batches():
    """A fixed set of signals gives the same bits alone, in batches of 37 and 200 003 at other
    positions, as a column slice of a wider tensor (row stride != n, offset pointer), and twice."""
    T, k = 1000, 16
    u, pu = _signals(T, k, seed=5)
    su, spu = _dev(u), _dev(pu)
    for args in ((), (4.0, 1.5)):
        real = not args
        def run(a, b):
            return _naff(a) if real else _naff(a, b, *args)
        ref = [torch.cat(t).cpu() for t in zip(*[run(su[:, i:i + 1], spu[:, i:i + 1]) for i in range(k)])]
        def same(q, a, cols):
            assert torch.equal(q[cols].cpu(), ref[0]) and torch.equal(a[cols].cpu(), ref[1])
        same(*run(su, spu), slice(None))
        same(*run(su, spu), slice(None))  # twice
        for n, first in ((37, 21), (37, 0), (200_003, 123_457), (200_003, 200_003 - k)):
            g = torch.Generator(device=DEV).manual_seed(n + first)
            bu = torch.randn(T, n, dtype=torch.float64, device=DEV, generator=g)
            bp = torch.randn(T, n, dtype=torch.float64, device=DEV, generator=g)
            bu[:, first:first + k] = su
            bp[:, first:first + k] = spu
            same(*run(bu, bp), slice(first, first + k))
            del bu, bp
        wide_u = torch.zeros(T, 3 * k + 5, dtype=torch.float64, device=DEV)
        wide_p = torch.zeros_like(wide_u)
        wide_u[:, 7:7 + k] = su
        wide_p[:, 7:7 + k] = spu
        vu, vp = wide_u[:, 7:7 + k], wide_p[:, 7:7 + k]
        assert vu.stride(0) != k and vu.data_ptr() != wide_u.data_ptr()
        same(*run(vu, vp), slice(None))


def test_argument_errors():
    import xline_b200 as xl

    u = torch.zeros(128, 8, dtype=torch.float64, device=DEV)
    for bad in (u[:63], torch.zeros(8193, 2, dtype=torch.float64, device=DEV), u.float(), u[:, ::2],
                u.t().contiguous().t()):
        with pytest.raises(ValueError):
            xl.naff(bad)
    with pytest.raises(ValueError):
        xl.naff(u, u[:, :4])
    with pytest.raises(ValueError):
        xl.naff(u, torch.zeros(128, 16, dtype=torch.float64, device=DEV)[:, :8])
    for beta in (0.0, -2.0):
        with pytest.raises(ValueError):
            xl.naff(u, u, beta=beta)
    with pytest.raises(RuntimeError):
        xl.naff(u.cpu())
    # the C entry point's own checks
    import ctypes as C

    from xline_b200 import _cabi

    L = _cabi.lib()
    p = C.c_void_p(u.data_ptr())
    for n, T, stride, pu, beta in ((-1, 128, 8, None, 1.0), (8, 63, 8, None, 1.0), (8, 8193, 8, None, 1.0),
                                   (8, 128, 7, None, 1.0), (8, 128, 8, p, 0.0), (8, 128, 8, p, float("nan"))):
        assert L.xlb_naff_device(p, pu, n, T, stride, beta, 0.0, p, p, None) == -1
    assert L.xlb_naff_device(None, None, 4, 128, 8, 1.0, 0.0, p, p, None) == -1
    assert L.xlb_naff_device(None, None, 0, 128, 0, 1.0, 0.0, None, None, None) == 0


def _twiss_at(line, i):
    from xline_b200 import optics

    tw = optics.twiss(line)
    return tw, (tw["betx"][i], tw["alfx"][i], tw["bety"][i], tw["alfy"][i])


def test_tracked_linear_tunes_match_twiss():
    """Small-amplitude PS Booster particle tracked on the GPU: the complex-signal tunes of
    monitor_tunes are optics.twiss's to 1e-10 (a CPU run of the same case: 1.4e-13 / 5e-15)."""
    import xline_b200 as xl
    from xline_b200 import configs

    line, meta = configs.load_lattice("psb")
    p0c, m0 = configs.p0c_of(meta)
    turns = 1024
    mon = xl.BeamMonitor(num_stores=turns, start=0, skip=1, min_particle_id=0, max_particle_id=1)
    line.insert_element(0, mon, "monitor")
    tw, opt = _twiss_at(line, 0)
    p = xl.Particles(p0c=p0c, mass0=m0, x=[1e-5, 2e-5], px=[0.0, 0.0], y=[1e-5, 0.0], py=[0.0, 1e-7])
    line.track(p, num_turns=turns)
    r = xl.monitor_tunes(mon, optics=opt)
    assert r["qx"].shape == (1, 2)
    qx, qy = r["qx"][0].cpu().numpy(), r["qy"][0].cpu().numpy()
    assert np.abs(qx - tw["qx"] % 1).max() <= 1e-10, qx - tw["qx"] % 1
    assert np.abs(qy - tw["qy"] % 1).max() <= 1e-10, qy - tw["qy"] % 1
    rr = xl.monitor_tunes(mon)
    assert abs(rr["qx"][0, 0].item() - tw["qx"] % 1) <= 1e-10


def test_octupole_detuning_on_the_gpu_tracker():
    import xline_b200 as xl

    k3l = 100.0
    line = octupole_fodo(k3l, ids=len(DETUNING_AMPLITUDES))
    tw, opt = _twiss_at(line, 0)
    p = xl.Particles(p0c=1e9, mass0=938.272e6, **detuning_columns(tw))
    line.track(p, num_turns=2048)
    r = xl.monitor_tunes(line.elements[0], optics=opt)
    q, a = r["qx"][0].cpu().numpy(), r["ax"][0].cpu().numpy()
    assert (q - tw["qx"] % 1).max() <= 1e-3
    assert np.abs(detuning_errors(q, a, tw, k3l)).max() <= 0.01


def _footprint(line, cols, p0c, m0, turns, mon):
    import xline_b200 as xl

    tw, opt = _twiss_at(line, 0)
    p = xl.Particles(p0c=p0c, mass0=m0, **cols)
    line.track(p, num_turns=turns)
    r = xl.monitor_tunes(mon, optics=opt)
    st = p.to_numpy()
    lost = st["state"] != 1
    for plane, q, a in (("x", "qx", "ax"), ("y", "qy", "ay")):
        u, pu = (mon.data[k].cpu().numpy() for k in (plane, "p" + plane))
        b, al = (opt[0], opt[1]) if plane == "x" else (opt[2], opt[3])
        ref = NO.naff(u, pu, b, al)
        exempt = assert_matches_oracle(r[q][0], r[a][0], ref, plane)
        assert exempt <= 2
        # NaN exactly where the window holds a non-finite sample, which includes every particle
        # lost inside it
        bad = ~(np.isfinite(u).all(axis=0) & np.isfinite(pu).all(axis=0))
        assert np.array_equal(np.isnan(r[q][0].cpu().numpy()), bad)
        assert bad[lost & (st["at_turn"] < turns - 1)].all()
    return r, lost


def test_space_charge_footprint_c5():
    from xline_b200 import configs

    n, turns = 500, 1024
    line, cols, p0c, m0 = configs.config_psb(n, monitor_stores=turns, monitor_ids=n)
    r, lost = _footprint(line, cols, p0c, m0, turns, line.elements[0])
    assert r["qx"].shape == (1, n) and np.isfinite(r["qx"][0].cpu().numpy()[~lost]).all()


def test_beam_beam_footprint_c3():
    import xline_b200 as xl
    from xline_b200 import configs

    n, turns = 200, 512
    line, cols, p0c, m0 = configs.config_lhc_beambeam(n)
    mon = xl.BeamMonitor(num_stores=turns, start=0, skip=1, min_particle_id=0, max_particle_id=n - 1)
    line.insert_element(0, mon, "monitor")
    r, lost = _footprint(line, cols, p0c, m0, turns, mon)
    assert r["qx"].shape == (1, n)


def test_frequency_map_with_losses():
    """Two windows of 512 turns on an octupole FODO amplitude grid, some particles lost in either
    window: each window's tunes follow the oracle, diffusion follows its formula and is NaN exactly
    for the particles lost before the end of the second window."""
    import xline_b200 as xl

    T = 512
    ax = np.linspace(0.004, 0.02, 16)
    ay = np.linspace(0.0005, 0.016, 8)
    X, Y = (v.ravel() for v in np.meshgrid(ax, ay))
    n = X.size
    line = octupole_fodo(3000.0, num_stores=2 * T, ids=n)
    line.append_element(xl.LimitEllipse(a=0.1, b=0.1), "aperture")
    tw, opt = _twiss_at(line, 0)
    z = np.zeros(n)
    p = xl.Particles(p0c=1e9, mass0=938.272e6, x=X * np.sqrt(tw["betx"][0]), px=z, y=Y * np.sqrt(tw["bety"][0]),
                     py=z, zeta=z, delta=z)
    line.track(p, num_turns=2 * T)
    st = p.to_numpy()
    lost = st["state"] != 1
    in_second = lost & (st["at_turn"] >= T) & (st["at_turn"] < 2 * T - 1)
    assert in_second.any() and (~lost).sum() >= n // 4
    mon = line.elements[0]
    r = xl.monitor_tunes(mon, num_turns=T, optics=opt, windows=2)
    for w in range(2):
        rows = slice(w * T, (w + 1) * T)
        for plane, q, a in (("x", "qx", "ax"), ("y", "qy", "ay")):
            u, pu = (mon.data[k][rows].cpu().numpy() for k in (plane, "p" + plane))
            b, al = (opt[0], opt[1]) if plane == "x" else (opt[2], opt[3])
            assert_matches_oracle(r[q][w], r[a][w], NO.naff(u, pu, b, al), (w, plane))
    qx, qy = r["qx"], r["qy"]
    expect = torch.log10(torch.sqrt((qx[1] - qx[0]) ** 2 + (qy[1] - qy[0]) ** 2))
    d = r["diffusion"]
    assert r["diffusion"].shape == (n,)
    assert torch.equal(torch.isnan(d), torch.isnan(expect)) and torch.equal(d[~torch.isnan(d)], expect[~torch.isnan(d)])
    d = d.cpu().numpy()
    assert np.array_equal(np.isnan(d), lost & (st["at_turn"] < 2 * T - 1))
