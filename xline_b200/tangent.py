"""Tangent map of the tracked one-turn map (include/xline_b200.h, "Tangent map"; DESIGN.md §4.8).

``Line.track_tangent(p, t, num_turns)`` tracks ``p`` exactly as ``Line.track`` would and carries,
per particle, the Jacobian ``J = dz/dz0`` over ``z = (x, px, y, py, zeta, delta)``, differentiated
element by element in the kernel (forward mode, no finite differences).  From it:

* ``TangentMap.fli`` -- the fast Lyapunov indicator ``max over turns of log10 ||J||_F``, and
  ``lyapunov(turns)`` -- ``log ||J||_F / turns``: chaos indicators that separate regular from
  chaotic orbits in 1e3 turns;
* ``closed_orbit(line, particles_like)`` -- the fixed point of the one-turn map by Newton's
  method with the exact Jacobian, and the one-turn matrix on it.
"""
import collections
import ctypes as C
import math

import numpy as np
import torch

from . import _cabi
from . import elements as E

_LOG10_SQRT6 = 0.5 * math.log10(6.0)
COORDS = ("x", "px", "y", "py", "zeta", "delta")


class TangentMap:
    """Per-particle Jacobians of ``n`` particles on ``device``: ``jacobian [n, 6, 6]`` (row-major,
    rows and columns in the order x px y py zeta delta) with the true Jacobian equal to
    ``jacobian * 2**log2_scale`` (the kernel rescales by exact powers of two to stay clear of
    overflow), and ``fli [n]``.  A fresh map is the identity: ``log2_scale`` 0, ``fli`` log10 sqrt(6)."""

    def __init__(self, n, device=None):
        device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.jacobian = torch.eye(6, dtype=torch.float64, device=device).repeat(int(n), 1, 1).contiguous()
        self.log2_scale = torch.zeros(int(n), dtype=torch.int64, device=device)
        self.fli = torch.full((int(n),), _LOG10_SQRT6, dtype=torch.float64, device=device)

    def __len__(self):
        return int(self.jacobian.shape[0])

    @property
    def device(self):
        return self.jacobian.device

    def log_norm(self):
        """Natural log of ``||J||_F`` per particle."""
        fro = torch.linalg.matrix_norm(self.jacobian)
        return torch.log(fro) + self.log2_scale.to(torch.float64) * math.log(2.0)

    def lyapunov(self, turns):
        """Finite-time Lyapunov estimate ``log ||J||_F / turns`` per particle."""
        return self.log_norm() / float(turns)

    def matrix(self):
        """``J * 2**log2_scale`` (inf where that overflows)."""
        return torch.ldexp(self.jacobian, self.log2_scale.to(torch.float64)[:, None, None])

    def _check_target(self, p):
        if len(self) != len(p):
            raise ValueError("TangentMap holds %d particles, the beam %d" % (len(self), len(p)))
        if self.jacobian.device != p.x.device:
            raise ValueError("TangentMap is on %s, the particles on %s" % (self.jacobian.device, p.x.device))
        for name in ("jacobian", "log2_scale", "fli"):
            t = getattr(self, name)
            if not t.is_contiguous():
                setattr(self, name, t.contiguous())


def track_tangent(line, p, tangent, num_turns=1, threads_per_block=0):
    """``Line.track_tangent``: see there."""
    from .line import _c_particles

    if p.device.type != "cuda":
        raise RuntimeError("track_tangent needs particles resident on a CUDA device (got %s)" % p.device)
    tangent._check_target(p)
    _refuse_radiation(line, "track_tangent")
    lib = _cabi.lib()
    dev = p.x.device
    with torch.cuda.device(dev):
        packed, words = line._tangent_lattice(dev)
        if len(p) == 0 or num_turns == 0:
            return None
        lat = packed.c_lattice(words.data_ptr())
        cp, cols = _c_particles(p)
        chi = cols.get("chi")
        if chi is not None and bool((chi == 1.0).all()):
            cp.chi = None
        if line.loss_tally is None or line.loss_tally.device != dev or line.loss_tally.numel() < max(packed.n_elements, 1):
            line.loss_tally = torch.zeros(max(packed.n_elements, 1), dtype=torch.int64, device=dev)
        opts = _cabi.TrackOptions()
        opts.num_turns = int(num_turns)
        opts.threads_per_block = int(threads_per_block)
        opts.loss_tally = line.loss_tally.data_ptr()
        stream = torch.cuda.current_stream(dev).cuda_stream
        _cabi.check(lib.xlb_track_tangent_device(C.byref(lat), C.byref(cp), C.byref(opts),
                                                 C.c_void_p(tangent.jacobian.data_ptr()),
                                                 C.c_void_p(tangent.log2_scale.data_ptr()),
                                                 C.c_void_p(tangent.fli.data_ptr()), C.c_void_p(stream)))
        line.last_stats = _cabi.stats()
    return None


ClosedOrbit = collections.namedtuple("ClosedOrbit", "z matrix iterations residual")
ClosedOrbit.__doc__ = """``z``: the orbit (x, px, y, py, zeta, delta) at the start of the line; ``matrix``: the 6x6
one-turn matrix of the tracked map at ``z``; ``iterations``: Newton steps taken; ``residual``: the
largest |M(z) - z| over the solved coordinates at ``z``."""


def _refuse_radiation(line, what):
    if getattr(line, "radiation", None) is not None:
        raise ValueError("%s: radiation is not part of the tangent map yet (set Line.radiation = None)" % what)


def has_rf(line):
    """True when the line holds an RF element with a voltage (a longitudinal restoring force)."""
    return any(isinstance(el, (E.Cavity, E.SawtoothCavity, E.RFMultipole)) and float(el.voltage) != 0.0
               for el in line.elements)


def closed_orbit(line, particles_like, guess=None, mode="auto", tol=1e-14, max_iter=30):
    """The closed orbit of ``line``: ``z`` with ``M(z) = z`` for the tracked one-turn map ``M``,
    by Newton's method on ``M(z) - z`` with the exact Jacobian of one-turn ``track_tangent`` calls
    on a single particle of ``particles_like``'s species and reference momentum.

    ``mode``: ``"4d"`` solves for (x, px, y, py) with delta held at the guess's value (zeta is
    carried along, not solved for); ``"6d"`` solves for all six coordinates and needs an RF
    system; ``"auto"`` is ``"6d"`` when the line holds an RF element with a voltage, else ``"4d"``.
    ``guess``: six coordinates (default zeros).  Stops when the residual -- the largest
    |M(z) - z| over the solved coordinates -- is at most ``tol`` (or no longer decreases after it
    came within 1e3 ``tol``).  Returns a ``ClosedOrbit``.  Raises ``ValueError`` when the
    particle is lost, when ``M - I`` is singular (no isolated fixed point) or when the iteration
    does not converge within ``max_iter`` steps."""
    _refuse_radiation(line, "closed_orbit")
    if mode == "auto":
        mode = "6d" if has_rf(line) else "4d"
    if mode not in ("4d", "6d"):
        raise ValueError("mode must be 'auto', '4d' or '6d'")
    if mode == "6d" and not has_rf(line):
        raise ValueError("a 6d closed orbit needs an RF element with a voltage")
    idx = [0, 1, 2, 3] if mode == "4d" else [0, 1, 2, 3, 4, 5]
    z = np.zeros(6) if guess is None else np.array(guess, dtype=np.float64).reshape(6)
    dev = particles_like.x.device
    from .particles import Particles

    best = math.inf
    for it in range(max_iter + 1):
        p = Particles(p0c=particles_like.p0c, mass0=particles_like.mass0, q0=particles_like.q0, device=dev,
                      **{k: [float(v)] for k, v in zip(COORDS, z)})
        t = TangentMap(1, dev)
        track_tangent(line, p, t, num_turns=1)
        if int(p.state[0]) != 1:
            raise ValueError("closed_orbit: the particle was lost at element %d (iteration %d, z = %s)"
                             % (int(p.at_element[0]), it, z.tolist()))
        mz = np.array([float(getattr(p, k)[0]) for k in COORDS])
        jac = t.matrix()[0].cpu().numpy()
        f = (mz - z)[idx]
        res = float(np.max(np.abs(f)))
        if not math.isfinite(res):
            raise ValueError("closed_orbit: the map is not finite at z = %s" % z.tolist())
        if res <= tol or (res >= best and best <= 1e3 * tol):
            return ClosedOrbit(z, jac, it, res)
        best = min(best, res)
        if it == max_iter:
            break
        a = jac[np.ix_(idx, idx)] - np.eye(len(idx))
        if np.linalg.cond(a) > 1e14:
            raise ValueError("closed_orbit: M - I is singular (cond %.3g): no isolated fixed point" % np.linalg.cond(a))
        z = z.copy()
        z[idx] -= np.linalg.solve(a, f)
    raise ValueError("closed_orbit: no convergence in %d iterations (residual %.3g)" % (max_iter, res))
