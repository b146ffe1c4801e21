"""Per-particle tunes from turn-by-turn data (NAFF, Laskar), computed on the GPU
(``csrc/naff.cu``; the definition is in ``include/xline_b200.h`` and DESIGN.md §4.7).

A signal is one particle in one plane over T turns.  ``naff`` takes a turn-major ``[T, n]`` slab
-- exactly the layout of a ``BeamMonitor``'s ``data`` fields -- and returns the frequency of the
largest spectral line of every column and its amplitude.  ``monitor_tunes`` does that for both
transverse planes of a monitor, for one turn window (a tune footprint) or two consecutive ones
(a frequency map and its diffusion index).

    mon = xl.BeamMonitor(num_stores=2048, start=0, skip=1, min_particle_id=0, max_particle_id=n - 1)
    line.insert_element(0, mon, "monitor"); line.track(p, num_turns=2048)
    tw = optics.twiss(line)
    fm = xl.monitor_tunes(mon, windows=2, optics=(tw["betx"][0], tw["alfx"][0], tw["bety"][0], tw["alfy"][0]))
    fm["qx"][0], fm["qy"][0], fm["diffusion"]
"""
import ctypes as C
import math

import torch

from . import _cabi

MIN_TURNS = _cabi.NAFF_MIN_TURNS
MAX_TURNS = _cabi.NAFF_MAX_TURNS


def _check_signal(name, a):
    if not isinstance(a, torch.Tensor):
        raise ValueError("naff: %s must be a torch tensor" % name)
    if a.dtype != torch.float64:
        raise ValueError("naff: %s must be float64 (got %s)" % (name, a.dtype))
    if a.dim() != 2:
        raise ValueError("naff: %s must be a [T, n] tensor (got %d dimensions)" % (name, a.dim()))
    T, n = a.shape
    if not MIN_TURNS <= T <= MAX_TURNS:
        raise ValueError("naff: T = %d turns outside [%d, %d]" % (T, MIN_TURNS, MAX_TURNS))
    if n > 1 and a.stride(1) != 1:
        raise ValueError("naff: %s needs unit column stride (got %d)" % (name, a.stride(1)))
    if a.stride(0) < n:
        raise ValueError("naff: %s row stride %d < n = %d" % (name, a.stride(0), n))


def naff(u, pu=None, beta=1.0, alpha=0.0):
    """Tune and amplitude of every column of ``u`` (``[T, n]`` float64 on a CUDA device, unit
    column stride, any row stride >= n): ``(tune [n], amplitude [n])`` on the same device.

    With ``pu`` (same shape and strides as ``u``) each column is the complex signal
    ``(u - i·(alpha·u + beta·pu)) / sqrt(beta)`` -- normalised coordinates for the Twiss ``beta``,
    ``alpha`` at the point the samples were taken -- and the tune lies in [0, 1).  Without it the
    real signal ``u``, tune in [0, 1/2].  The amplitude is sqrt(2J) of a linear particle in the
    complex case.  NaN tune and amplitude for a column with a non-finite sample (a lost particle);
    NaN tune and zero amplitude for a constant one.  Results are bitwise independent of the batch
    (n, column, row stride)."""
    _check_signal("u", u)
    if pu is not None:
        _check_signal("pu", pu)
        if pu.shape != u.shape or pu.stride() != u.stride():
            raise ValueError("naff: pu must have the shape and strides of u (%s %s vs %s %s)"
                             % (tuple(pu.shape), pu.stride(), tuple(u.shape), u.stride()))
        if pu.device != u.device:
            raise ValueError("naff: u on %s, pu on %s" % (u.device, pu.device))
        beta, alpha = float(beta), float(alpha)
        if not (math.isfinite(beta) and beta > 0.0 and math.isfinite(alpha)):
            raise ValueError("naff: beta must be finite and > 0, alpha finite (got %r, %r)" % (beta, alpha))
    if u.device.type != "cuda":
        raise RuntimeError("xline_b200.naff needs tensors on a CUDA device (got %s): there is no CPU path"
                           % u.device)
    T, n = u.shape
    tune = torch.empty(n, dtype=torch.float64, device=u.device)
    amp = torch.empty(n, dtype=torch.float64, device=u.device)
    if n == 0:
        return tune, amp
    with torch.cuda.device(u.device):
        stream = torch.cuda.current_stream(u.device).cuda_stream
        _cabi.check(_cabi.lib().xlb_naff_device(
            C.c_void_p(u.data_ptr()), C.c_void_p(pu.data_ptr() if pu is not None else None), n, T, u.stride(0),
            float(beta), float(alpha), C.c_void_p(tune.data_ptr()), C.c_void_p(amp.data_ptr()), C.c_void_p(stream)))
    return tune, amp


def monitor_tunes(monitor, num_turns=None, start=0, optics=None, windows=1):
    """NAFF tunes of both transverse planes of a tracked ``BeamMonitor``.

    Window ``w < windows`` is the stores ``start + w·T .. start + (w + 1)·T`` (T = ``num_turns``,
    by default as many as fit).  ``optics = (betx, alfx, bety, alfy)`` at the monitor (e.g. from
    ``optics.twiss(line)`` at its element index) analyses the complex normalised signals x/px and
    y/py; ``None`` the real signals x and y.  Returns ``qx, qy, ax, ay`` (``[windows, nn]``, one
    column per monitored particle id) and, with ``windows == 2``, the frequency-map diffusion index
    ``diffusion = log10(sqrt(Δqx² + Δqy²))`` (``[nn]``, NaN where either window is invalid)."""
    if monitor.is_rolling:
        raise ValueError("monitor_tunes: a rolling monitor does not hold consecutive turns in store order")
    if int(monitor.skip) != 1:
        raise ValueError("monitor_tunes: skip = %d; the stores must be consecutive turns (skip = 1)" % monitor.skip)
    if not isinstance(monitor.data, dict) or "x" not in monitor.data:
        raise ValueError("monitor_tunes: the monitor holds no data (track a line that contains it first)")
    windows, start = int(windows), int(start)
    if windows < 1 or start < 0:
        raise ValueError("monitor_tunes: needs windows >= 1 and start >= 0")
    num_stores = int(monitor.data["x"].shape[0])
    T = (num_stores - start) // windows if num_turns is None else int(num_turns)
    if T < 1 or start + windows * T > num_stores:
        raise ValueError("monitor_tunes: %d window(s) of %d turns from store %d run past num_stores = %d"
                         % (windows, T, start, num_stores))
    if optics is not None:
        betx, alfx, bety, alfy = (float(v) for v in optics)
    out = {k: [] for k in ("qx", "qy", "ax", "ay")}
    for w in range(windows):
        rows = slice(start + w * T, start + (w + 1) * T)
        for plane, (q, a) in (("x", ("qx", "ax")), ("y", ("qy", "ay"))):
            u = monitor.data[plane][rows]
            if optics is None:
                tune, amp = naff(u)
            else:
                b, al = (betx, alfx) if plane == "x" else (bety, alfy)
                tune, amp = naff(u, monitor.data["p" + plane][rows], beta=b, alpha=al)
            out[q].append(tune)
            out[a].append(amp)
    res = {k: torch.stack(v) for k, v in out.items()}
    if windows == 2:
        qx, qy = res["qx"], res["qy"]
        res["diffusion"] = torch.log10(torch.sqrt((qx[1] - qx[0]) ** 2 + (qy[1] - qy[0]) ** 2))
    return res
