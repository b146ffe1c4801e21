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
        _check_target(self, p, ("jacobian", "log2_scale", "fli"))


def _check_target(holder, p, names):
    """Refuse a TangentMap or Envelope of another size or device than ``p``; make its tensors
    ``names`` contiguous."""
    what = type(holder).__name__
    if len(holder) != len(p):
        raise ValueError("%s holds %d particles, the beam %d" % (what, len(holder), len(p)))
    if holder.device != p.x.device:
        raise ValueError("%s is on %s, the particles on %s" % (what, holder.device, p.x.device))
    for name in names:
        t = getattr(holder, name)
        if not t.is_contiguous():
            setattr(holder, name, t.contiguous())


def _launch(line, p, num_turns, threads_per_block, radiation, call):
    """One call of a tangent-map entry point on ``p``: ``call(lib, lat, cp, opts, stream)``."""
    from .line import _c_particles

    lib = _cabi.lib()
    dev = p.x.device
    with torch.cuda.device(dev):
        packed, words = line._tangent_lattice(dev, radiation=radiation)
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
        _cabi.check(call(lib, lat, cp, opts, C.c_void_p(stream)))
        line.last_stats = _cabi.stats()
    return None


def track_tangent(line, p, tangent, num_turns=1, threads_per_block=0, radiation=False):
    """``Line.track_tangent``: see there."""
    _refuse_exciter(line, "track_tangent")
    if p.device.type != "cuda":
        raise RuntimeError("track_tangent needs particles resident on a CUDA device (got %s)" % p.device)
    tangent._check_target(p)
    rad = bool(radiation) and getattr(line, "radiation", None) is not None
    if rad:
        if line.radiation != "mean":
            raise ValueError("track_tangent: radiation=True needs Line.radiation = 'mean' (got %r): the "
                             "quantum map is random and has no tangent" % (line.radiation,))
    else:
        _refuse_radiation(line, "track_tangent")
    _tangent_call(line, p, tangent, num_turns, threads_per_block, rad)
    return None


def _tangent_call(line, p, tangent, num_turns, threads_per_block, rad):
    fn = "xlb_track_tangent_radiation_device" if rad else "xlb_track_tangent_device"
    _launch(line, p, num_turns, threads_per_block, rad,
            lambda lib, lat, cp, opts, stream: getattr(lib, fn)(
                C.byref(lat), C.byref(cp), C.byref(opts), C.c_void_p(tangent.jacobian.data_ptr()),
                C.c_void_p(tangent.log2_scale.data_ptr()), C.c_void_p(tangent.fli.data_ptr()), stream))


class Envelope:
    """Per-particle beam envelopes of ``n`` particles on ``device`` for ``Line.track_envelope``:
    ``cov [n, 6, 6]`` -- the second moment Sigma of a beam around each particle over (x, px, y, py,
    zeta, delta), row-major, symmetric -- and ``energy_loss [n]``, the energy radiated (eV).  Both
    start at zero."""

    def __init__(self, n, device=None):
        device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.cov = torch.zeros((int(n), 6, 6), dtype=torch.float64, device=device)
        self.energy_loss = torch.zeros(int(n), dtype=torch.float64, device=device)

    def __len__(self):
        return int(self.cov.shape[0])

    @property
    def device(self):
        return self.cov.device

    def _check_target(self, p):
        _check_target(self, p, ("cov", "energy_loss"))


def track_envelope(line, p, envelope, num_turns=1, threads_per_block=0):
    """``Line.track_envelope``: see there."""
    _refuse_exciter(line, "track_envelope")
    if p.device.type != "cuda":
        raise RuntimeError("track_envelope needs particles resident on a CUDA device (got %s)" % p.device)
    envelope._check_target(p)
    rad = getattr(line, "radiation", None) is not None
    _launch(line, p, num_turns, threads_per_block, rad,
            lambda lib, lat, cp, opts, stream: lib.xlb_track_envelope_device(
                C.byref(lat), C.byref(cp), C.byref(opts), C.c_void_p(envelope.cov.data_ptr()),
                C.c_void_p(envelope.energy_loss.data_ptr()), stream))
    return None


ClosedOrbit = collections.namedtuple("ClosedOrbit", "z matrix iterations residual")
ClosedOrbit.__doc__ = """``z``: the orbit (x, px, y, py, zeta, delta) at the start of the line; ``matrix``: the 6x6
one-turn matrix of the tracked map at ``z``; ``iterations``: Newton steps taken; ``residual``: the
largest |M(z) - z| over the solved coordinates at ``z``."""


def _refuse_radiation(line, what):
    if getattr(line, "radiation", None) is not None:
        raise ValueError("%s: radiation is left out of the tangent map unless asked for (pass radiation=True, "
                         "or set Line.radiation = None)" % what)


def _refuse_exciter(line, what):
    for i, el in enumerate(line.elements):
        if isinstance(el, E.Exciter):
            raise ValueError("%s: element %d is an Exciter, a turn-dependent map without a tangent map or "
                             "closed orbit (remove it, e.g. track a copy of the line without it)" % (what, i))


def has_rf(line):
    """True when the line holds an RF element with a voltage (a longitudinal restoring force)."""
    return any(isinstance(el, (E.Cavity, E.SawtoothCavity, E.RFMultipole)) and float(el.voltage) != 0.0
               for el in line.elements)


def closed_orbit(line, particles_like, guess=None, mode="auto", tol=1e-14, max_iter=30, radiation=False):
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
    does not converge within ``max_iter`` steps.

    A radiating line is refused unless ``radiation=True``: then the map is the mean-mode map with
    its radiation (for a ``"quantum"`` line as well: the damped orbit is that of the mean loss), and
    only the 6d orbit exists -- delta is not conserved, so ``"4d"`` is refused.  On a line without
    radiation ``radiation=True`` changes nothing."""
    _refuse_exciter(line, "closed_orbit")
    rad = bool(radiation) and getattr(line, "radiation", None) is not None
    if not rad:
        _refuse_radiation(line, "closed_orbit")
    elif mode == "4d":
        raise ValueError("closed_orbit: a radiating line has no 4d closed orbit (delta is not conserved); "
                         "use mode='6d'")
    elif mode == "auto":
        mode = "6d"  # the only orbit of a radiating line: without RF it is refused below
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
        _tangent_call(line, p, t, 1, 0, rad)
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


RadiationEquilibrium = collections.namedtuple(
    "RadiationEquilibrium", "orbit matrix diffusion cov energy_loss damping_times tunes partition emittances "
                            "sigma_delta sigma_zeta iterations")
RadiationEquilibrium.__doc__ = """``orbit``: the damped closed orbit (x, px, y, py, zeta, delta) at the start of
the line; ``matrix``: the one-turn matrix M there, radiation included; ``diffusion``: D, the second
moment one turn of quantum emission adds (Sigma = 0 transported over one turn); ``cov``: the
equilibrium Sigma = M Sigma M^T + D; ``energy_loss``: the energy radiated per turn on the orbit (eV);
per mode, ordered x-, y-, z-like (the plane holding most of the eigenvector): ``damping_times``
(turns, -1/ln|lambda|), ``tunes`` (|arg lambda|/2pi), ``partition`` (2 E0/(tau U)) and ``emittances``;
``sigma_delta``, ``sigma_zeta``: sqrt of the diagonal of ``cov``; ``iterations``: Newton steps."""


def _symplectic_modes(m):
    """Eigenvalues lam_k and eigenvectors v_k (k = 0, 1, 2) of the 6x6 ``m``, one of each complex pair,
    scaled so that v^H S v = i (S the symplectic form); the columns of the returned V are
    (v_0, conj v_0, v_1, conj v_1, v_2, conj v_2).  Raises when an eigenvalue is real (no oscillation)."""
    lam, vec = np.linalg.eig(m)
    S = np.zeros((6, 6))
    for k in range(3):
        S[2 * k, 2 * k + 1], S[2 * k + 1, 2 * k] = 1.0, -1.0
    used, lams, vs = set(), [], []
    for i in np.argsort(-np.abs(lam.imag)):
        if i in used:
            continue
        if abs(lam[i].imag) < 1e-12:
            raise ValueError("radiation_equilibrium: the one-turn matrix has a real eigenvalue %.6g: no stable "
                             "oscillation in every plane" % lam[i].real)
        j = min((jj for jj in range(6) if jj not in used and jj != i), key=lambda jj: abs(lam[jj] - np.conj(lam[i])))
        used |= {i, j}
        v = vec[:, i]
        q = np.conj(v) @ S @ v  # purely imaginary up to the damping
        if q.imag < 0:
            v, l_ = np.conj(v), np.conj(lam[i])
        else:
            l_ = lam[i]
        vs.append(v / math.sqrt(abs(q.imag)))
        lams.append(l_)
    V = np.zeros((6, 6), dtype=complex)
    for k, v in enumerate(vs):
        V[:, 2 * k], V[:, 2 * k + 1] = v, np.conj(v)
    return np.array(lams), V


def radiation_equilibrium(line, particles_like, guess=None, tol=1e-14, max_iter=30):
    """The equilibrium of a radiating ring (``line.radiation`` ``"mean"`` or ``"quantum"``, with an RF
    voltage) from its tangent map and envelope on the GPU:

    1. the damped closed orbit and its one-turn matrix M (``closed_orbit(..., "6d", radiation=True)``);
    2. one ``Line.track_envelope`` turn from Sigma = 0 on the orbit: the diffusion D and the energy
       radiated per turn U;
    3. Sigma = M Sigma M^T + D (``scipy.linalg.solve_discrete_lyapunov``).

    Modes: the eigenvectors v_k of M, one of each complex-conjugate pair, normalised symplectically
    (v^H S v = i, S the block-diagonal symplectic form; for an uncoupled plane with Twiss beta, alpha this
    is v = (sqrt(beta), (i - alpha)/sqrt(beta))/sqrt(2), so that v v^H + conj(v v^H) = [[beta, -alpha],
    [-alpha, gamma]]).  With V = (v_0, conj v_0, ...) and B = V^-1 D V^-H, the emittance of mode k is
    eps_k = B_kk / (1 - |lambda_k|^2): the mean |a_k|^2 of the mode amplitudes a = V^-1 z.  Damping
    times -1/ln|lambda_k| in turns, partition numbers J_k = 2 E0 / (tau_k U) with E0 the reference
    particle's total energy.  Returns a ``RadiationEquilibrium``; raises ``ValueError`` for a line
    without radiation or RF, and as ``closed_orbit`` does."""
    import itertools

    from scipy.linalg import solve_discrete_lyapunov

    from .particles import Particles

    _refuse_exciter(line, "radiation_equilibrium")
    if getattr(line, "radiation", None) is None:
        raise ValueError("radiation_equilibrium: the line does not radiate (set Line.radiation = 'mean' or 'quantum')")
    if not has_rf(line):
        raise ValueError("radiation_equilibrium: the line needs an RF element with a voltage")
    co = closed_orbit(line, particles_like, guess=guess, mode="6d", tol=tol, max_iter=max_iter, radiation=True)
    dev = particles_like.x.device
    p = Particles(p0c=particles_like.p0c, mass0=particles_like.mass0, q0=particles_like.q0, device=dev,
                  **{k: [float(v)] for k, v in zip(COORDS, co.z)})
    env = Envelope(1, dev)
    track_envelope(line, p, env, num_turns=1)
    if int(p.state[0]) != 1:
        raise ValueError("radiation_equilibrium: the particle on the closed orbit was lost")
    D = env.cov[0].cpu().numpy()
    U = float(env.energy_loss[0])
    M = co.matrix
    cov = solve_discrete_lyapunov(M, D)
    cov = 0.5 * (cov + cov.T)
    lam, V = _symplectic_modes(M)
    B = np.linalg.solve(V, np.linalg.solve(V, D.astype(complex)).conj().T).conj().T  # V^-1 D V^-H
    w = np.array([[abs(V[2 * pl, 2 * k]) ** 2 + abs(V[2 * pl + 1, 2 * k]) ** 2 for pl in range(3)] for k in range(3)])
    w = w / w.sum(axis=1, keepdims=True)
    order = max(itertools.permutations(range(3)), key=lambda perm: sum(w[perm[pl], pl] for pl in range(3)))
    energy0 = float(particles_like.energy0)
    tau, tunes, part, eps = [], [], [], []
    for k in order:
        mod = abs(lam[k])
        t_ = -1.0 / math.log(mod)
        tau.append(t_)
        tunes.append(abs(np.angle(lam[k])) / (2 * math.pi))
        part.append(2.0 * energy0 / (t_ * U) if U > 0 else math.nan)
        eps.append(float(B[2 * k, 2 * k].real) / (1.0 - mod * mod))
    return RadiationEquilibrium(co.z, M, D, cov, U, np.array(tau), np.array(tunes), np.array(part), np.array(eps),
                                math.sqrt(cov[5, 5]), math.sqrt(cov[4, 4]), co.iterations)
