"""NumPy NAFF: the definition of include/xline_b200.h (xlb_naff_device) step by step, vectorised
over signals.  Test infrastructure only; the library has no CPU path."""
import numpy as np

MIN_TURNS, MAX_TURNS = 64, 8192
MAX_ITER = 40
TOL = 1e-15
NEAR_TIE = 1e-9  # relative gap of the two largest coarse bins below which the coarse k is fragile


def coarse_bin(mag, real):
    """Step 4: argmax over k = 1 .. M-1 (complex) or 1 .. M/2 (real) of ``mag [M, n]``, the lowest
    k on ties; and whether the two largest bins in that range are within NEAR_TIE (relative)."""
    M = mag.shape[0]
    kmax = M // 2 if real else M - 1
    part = mag[1:kmax + 1]
    k = 1 + np.argmax(part, axis=0)  # first occurrence
    top2 = np.sort(part, axis=0)[-2:]
    near = (top2[1] - top2[0]) <= NEAR_TIE * top2[1]
    return k, near


def _phase(x):
    """e^{-2πi x} from the reduced argument x - rint(x)."""
    return np.exp(-2j * np.pi * (x - np.rint(x)))


def naff(u, pu=None, beta=1.0, alpha=0.0, chunk=256, with_passes=False):
    """``u``, ``pu``: ``[T, n]`` arrays (turn-major, like a BeamMonitor field).  Returns
    ``(tune [n], amplitude [n], near_tie [n])``, and with ``with_passes`` the number of refinement
    passes over the samples of every signal (0 for invalid ones)."""
    u = np.asarray(u, dtype=np.float64)
    if u.ndim == 1:
        u = u[:, None]
        pu = None if pu is None else np.asarray(pu, dtype=np.float64)[:, None]
    T, n = u.shape
    tune = np.full(n, np.nan)
    amp = np.full(n, np.nan)
    near = np.zeros(n, dtype=bool)
    passes = np.zeros(n, dtype=np.int64)
    for c0 in range(0, n, chunk):
        sl = slice(c0, min(n, c0 + chunk))
        a = u[:, sl]
        if pu is None:
            z = a.astype(np.complex128)
            finite = np.isfinite(a).all(axis=0)
        else:
            b = np.asarray(pu, dtype=np.float64)[:, sl]
            with np.errstate(invalid="ignore"):  # inf samples: NaN z, flagged by `finite`
                z = a / np.sqrt(beta) - 1j * (alpha * a + beta * b) / np.sqrt(beta)
            finite = np.isfinite(a).all(axis=0) & np.isfinite(b).all(axis=0)
        tune[sl], amp[sl], near[sl], passes[sl] = _naff_block(z, pu is None, finite)
    return (tune, amp, near, passes) if with_passes else (tune, amp, near)


def _naff_block(z, real, finite):
    T, n = z.shape
    tune = np.full(n, np.nan)
    amp = np.full(n, np.nan)
    near = np.zeros(n, dtype=bool)
    passes = np.zeros(n, dtype=np.int64)
    z = np.where(finite[None, :], z, 0.0)
    z = z - z.mean(axis=0, keepdims=True)                          # 1
    zero = finite & np.all(z == 0, axis=0)
    amp[zero] = 0.0
    ok = np.nonzero(finite & ~zero)[0]
    if ok.size == 0:
        return tune, amp, near, passes
    t = np.arange(T)
    w = 2.0 * np.sin(np.pi * t / T) ** 2                            # 2: 1 - cos(2πt/T)
    zw = (z[:, ok] * w[:, None]).T                                   # [m, T]
    M = 1 << int(np.ceil(np.log2(T)))
    k, near_ok = coarse_bin(np.abs(np.fft.fft(zw, M, axis=1)).T, real)  # 4
    near[ok] = near_ok
    tc = t - 0.5 * T
    lo, hi, nu = (k - 1) / M, (k + 1) / M, k / M                     # 5
    s0 = np.zeros(ok.size, dtype=np.complex128)
    active = np.ones(ok.size, dtype=bool)
    for _ in range(MAX_ITER):
        i = np.nonzero(active)[0]
        if i.size == 0:
            break
        a = zw[i] * _phase(nu[i, None] * tc[None, :])                # 3: w·z·e^{-2πiν t_c}
        S0, S1, S2 = a.sum(axis=1), (a * tc).sum(axis=1), (a * tc * tc).sum(axis=1)
        s0[i] = S0
        passes[ok[i]] += 1
        # D = Re(conj(Z)·Z') = 2π·Im(conj(S0)·S1),  D' = 4π²·(|S1|² - Re(conj(S0)·S2))
        d = (np.conj(S0) * S1).imag
        dd = np.abs(S1) ** 2 - (np.conj(S0) * S2).real
        hit = (d == 0) & (dd < 0)  # a stationary point that is a maximum
        up = d > 0
        lo[i] = np.where(~hit & up, nu[i], lo[i])
        hi[i] = np.where(~hit & ~up, nu[i], hi[i])
        with np.errstate(divide="ignore", invalid="ignore"):
            nxt = nu[i] - d / (2 * np.pi * dd)
        bad = ~(dd < 0) | ~((nxt >= lo[i]) & (nxt <= hi[i]))  # inclusive: a converged step is 0
        nxt = np.where(bad, 0.5 * (lo[i] + hi[i]), nxt)
        nxt = np.where(hit, nu[i], nxt)
        step = np.abs(nxt - nu[i])
        nu[i] = nxt
        active[i] = ~(hit | (step < TOL))
    nu = np.where(nu > 0.5, 1.0 - nu, nu) if real else np.where(nu >= 1.0, nu - 1.0, nu)  # 6: fold
    tune[ok] = nu
    amp[ok] = np.abs(s0) / T
    return tune, amp, near, passes
