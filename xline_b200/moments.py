"""Beam moments: the number of particles and the first and second moments of
(x, px, y, py, zeta, delta) over the surviving beam, reduced on the GPU (``csrc/moments.cu``).

A store holds ``_cabi.MOMENT_WORDS`` float64 words (``include/xline_b200.h``): ``n``,
``n_nonfinite``, then 27 double-double sums (hi, lo): Σu for the six coordinates and Σu·v for
the 21 pairs u <= v, upper triangle in row-major order.  Those sums are what ranks add up
(``sharding.merge_moments``); the centred quantities are derived from them on demand.

    m = xl.BeamMoments(num_stores=1001, start=0, skip=10)
    line.track(p, num_turns=10_000, moments=m)
    m.emittance()["neps_x"]      # normalised horizontal rms emittance, turn 0, 10, ... 10 000
"""
import ctypes as C

import torch

from . import _cabi

COORDS = ("x", "px", "y", "py", "zeta", "delta")
# (u, v) of every pair of a store: the six first moments (v = None), then the products
PAIRS = tuple((u, None) for u in range(6)) + tuple((u, v) for u in range(6) for v in range(u, 6))


def pair_index(u, v=None):
    """Index (0..26) of the pair that holds Σu (``v is None``) or Σu·v."""
    if v is None:
        return u
    u, v = min(u, v), max(u, v)
    return PAIRS.index((u, v))


# ---------------------------------------------------------------------- double-double on tensors
def _two_sum(a, b):
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def _fast_two_sum(a, b):
    s = a + b
    return s, b - (s - a)


def _split(a):
    t = 134217729.0 * a  # 2^27 + 1 (Veltkamp)
    hi = t - (t - a)
    return hi, a - hi


def _two_prod(a, b):
    """Exact product without FMA (Dekker); exact unless an intermediate overflows."""
    p = a * b
    ah, al = _split(a)
    bh, bl = _split(b)
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


def dd_add(ah, al, bh, bl):
    """AccurateDWPlusDW (Joldes, Muller, Popescu 2017): relative error <= 3·2^-106; the same
    operations as the device reduction."""
    sh, sl = _two_sum(ah, bh)
    th, tl = _two_sum(al, bl)
    vh, vl = _fast_two_sum(sh, sl + th)
    return _fast_two_sum(vh, tl + vl)


def _dd_mul(ah, al, bh, bl):
    p, e = _two_prod(ah, bh)
    return _fast_two_sum(p, e + (ah * bl + al * bh))


def _dd_div(ah, al, d):
    """(ah + al) / d for a float64 tensor d, to double-double."""
    q1 = ah / d
    p, e = _two_prod(q1, d)
    r = ((ah - p) - e) + al
    return _fast_two_sum(q1, r / d)


# ---------------------------------------------------------------------- the container
class BeamMoments:
    """Stores ``k < num_stores`` of the beam moments, store k after ``start + k * skip`` turns of
    one ``Line.track(p, num_turns, moments=...)`` call (turn 0 = before the first turn).  Stores
    past ``num_turns`` are not written and keep NaN.

    ``data``: the raw device tensor ``[num_stores, 56]``.  ``count`` / ``n_nonfinite``: the
    particles that count (``state == 1`` and six finite coordinates) and the alive particles with
    a non-finite coordinate.  ``mean [S, 6]``, ``cov [S, 6, 6]`` and ``emittance()`` are derived
    from the sums in double-double and rounded once.
    """

    def __init__(self, num_stores, start=0, skip=1, device=None):
        num_stores, start, skip = int(num_stores), int(start), int(skip)
        if num_stores < 0 or start < 0 or skip < 1:
            raise ValueError("BeamMoments needs num_stores >= 0, start >= 0 and skip >= 1")
        self.num_stores, self.start, self.skip = num_stores, start, skip
        if device is None:
            from .particles import _default_device

            device = _default_device()
        self.data = torch.full((num_stores, _cabi.MOMENT_WORDS), float("nan"), dtype=torch.float64,
                               device=device)
        self.beta0gamma0 = None  # of the particles last tracked into the stores

    def _spec(self):
        spec = _cabi.MomentsSpec()
        spec.num_stores, spec.start, spec.skip = self.num_stores, self.start, self.skip
        return spec

    def _check_target(self, p):
        if self.data.device != p.x.device:
            raise ValueError("BeamMoments on %s, particles on %s" % (self.data.device, p.x.device))
        if not self.data.is_contiguous() or self.data.shape != (self.num_stores, _cabi.MOMENT_WORDS):
            raise ValueError("BeamMoments.data must be a contiguous [num_stores, %d] tensor" % _cabi.MOMENT_WORDS)

    @property
    def turn(self):
        """Turn of every store within the call, ``int64 [S]``."""
        return self.start + self.skip * torch.arange(self.num_stores, dtype=torch.int64)

    @property
    def count(self):
        return self.data[:, 0].to(torch.int64)

    @property
    def n_nonfinite(self):
        return self.data[:, 1].to(torch.int64)

    def sums(self):
        """``(hi, lo)``, each ``[S, 27]``: the pairs of every store."""
        w = self.data[:, _cabi.MOMENT_FIRST:]
        return w[:, 0::2], w[:, 1::2]

    def _mean_dd(self):
        hi, lo = self.sums()
        n = self.data[:, 0:1]
        return _dd_div(hi[:, :6], lo[:, :6], n)

    @property
    def mean(self):
        """``[S, 6]``: Σu / n, rounded once."""
        mh, ml = self._mean_dd()
        return mh + ml

    @property
    def cov(self):
        """``[S, 6, 6]``: ``(Σu·v - Σu·Σv / n) / n`` in double-double, rounded once."""
        hi, lo = self.sums()
        n = self.data[:, 0:1]
        u = torch.tensor([a for a, b in PAIRS[6:]])
        v = torch.tensor([b for a, b in PAIRS[6:]])
        ph, pl = _dd_mul(hi[:, u], lo[:, u], hi[:, v], lo[:, v])
        ph, pl = _dd_div(ph, pl, n)
        dh, dl = dd_add(hi[:, 6:], lo[:, 6:], -ph, -pl)
        ch, cl = _dd_div(dh, dl, n)
        c = ch + cl
        out = torch.empty((self.num_stores, 6, 6), dtype=torch.float64, device=self.data.device)
        out[:, u, v] = c
        out[:, v, u] = c
        return out

    def emittance(self, beta0gamma0=None):
        """Geometric rms emittances ``sqrt(det)`` of the (x, px), (y, py) and (zeta, delta) blocks
        of ``cov`` (``eps_x``, ``eps_y``, ``eps_zeta``; the determinant in double-double, rounded
        once), and the transverse normalised ones ``neps_x``, ``neps_y`` (× β0γ0 of the tracked
        particles, or of ``beta0gamma0``), each ``[S]``."""
        c = self.cov
        bg = self.beta0gamma0 if beta0gamma0 is None else beta0gamma0
        out = {}
        for name, k in (("x", 0), ("y", 2), ("zeta", 4)):
            a, b, d = c[:, k, k], c[:, k, k + 1], c[:, k + 1, k + 1]
            p1h, p1l = _two_prod(a, d)
            p2h, p2l = _two_prod(b, b)
            dh, dl = dd_add(p1h, p1l, -p2h, -p2l)
            out["eps_" + name] = torch.sqrt(dh + dl)
        if bg is not None:
            out["neps_x"] = out["eps_x"] * bg
            out["neps_y"] = out["eps_y"] * bg
        return out

    def __repr__(self):
        return "BeamMoments(num_stores=%d, start=%d, skip=%d, device=%s)" % (
            self.num_stores, self.start, self.skip, self.data.device)


def beam_moments(p):
    """One snapshot of the particles ``p`` (on a CUDA device): a ``BeamMoments`` with one store."""
    from .line import _c_particles

    if p.x.device.type != "cuda":
        raise RuntimeError("xline_b200.beam_moments needs particles on a CUDA device (got %s)" % p.x.device)
    m = BeamMoments(1, device=p.x.device)
    with torch.cuda.device(p.x.device):
        cp, _ = _c_particles(p)
        stream = torch.cuda.current_stream(p.x.device).cuda_stream
        _cabi.check(_cabi.lib().xlb_beam_moments_device(C.byref(cp), C.c_void_p(m.data.data_ptr()),
                                                        C.c_void_p(stream)))
    m.beta0gamma0 = p.beta0 * p.gamma0
    return m
