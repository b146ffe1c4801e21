"""TEST INFRASTRUCTURE -- a NumPy interpreter of packed lattices that hold EXCITER records.

Walks the words of ``xline_b200.lattice.pack_line`` as ``include/xline_b200.h`` documents them --
chunks, record headers, the path-length words, and the data region after the chunks that holds the
exciters' samples -- and applies the element maps with the helpers of ``tests/packed_interpreter.py``
(the same arithmetic).  It covers the fast encoding of thin-lens lines: drifts, multipoles (straight,
curved, radiating), thin and edge blocks, the LIMIT_* records, shifts, rotations, dipole edges,
cavities, monitors (which store nothing here) and EXCITER; anything else raises.  Each particle's
turn is its own ``at_turn`` (the starting column plus the turns done), as the kernel takes it.
Nothing in the product imports this file.
"""
import numpy as np

from tests import packed_interpreter as PI

T_EXCITER = 0x40


def exciter_index(f64, i64, w, at_turn, zeta, beta0):
    """EXCITER at word ``w``, [hdr,A][B,start_turn][n_samples,data_offset]: the sample index of every
    particle, -1 for none -- u = t*A - (zeta*B)/beta0, v = floor(u + 0.5), each operation rounded once."""
    a, b, start, n = f64[w + 1], f64[w + 2], i64[w + 3], int(i64[w + 4])
    t = (np.asarray(at_turn, dtype=np.int64) - start).astype(np.float64)
    with np.errstate(invalid="ignore"):
        v = np.floor((t * a - (zeta * b) / beta0) + 0.5)
        ok = (v >= 0) & (v < n)
    return np.where(ok, v, -1.0).astype(np.int64)


def _exciter(p, beam, f64, i64, w, aux):
    """EXCITER at word ``w``: the MULTIPOLE pairs from pair 3, the samples in the data region."""
    idx = exciter_index(f64, i64, w, beam.at_turn[p.idx], p.zeta, beam.beta0)
    off, n = int(i64[w + 5]), int(i64[w + 4])
    assert n == 0 or off + n <= len(f64)
    s = np.where(idx >= 0, f64[off + np.maximum(idx, 0)], 0.0) if n else np.zeros(len(idx))
    dpx, dpy = PI._horner(p, f64[w + 6: w + 6 + 2 * (aux + 1)].reshape(aux + 1, 2), aux, False)
    p.px = p.px + (-p.chi * (s * dpx))
    p.py = p.py + p.chi * (s * dpy)


def _lose(p, lost, elem):
    """``_Live.lose`` keeping every particle's own turn in ``at_turn``."""
    turns = p.beam.at_turn.copy()
    p.lose(lost, elem, 0)
    p.beam.at_turn[:] = turns


def _limit(p, tag, aux, w, f64, elem):
    pair = lambda m: f64[w + 2 * m: w + 2 * m + 2]  # noqa: E731
    x, y = p.x, p.y
    if tag == PI.T_LIMIT_RECT:
        lim = np.array([f64[w + 1], pair(1)[0], pair(1)[1], pair(2)[0]])
        inside, drift = PI._inside(PI.AP_RECT_SYM if aux & 1 else PI.AP_RECT, x, y, lim, False), pair(3)[0]
    elif tag == PI.T_LIMIT_ELLIPSE:
        lim = np.array([f64[w + 1], pair(1)[0], pair(1)[1], pair(2)[0]])
        inside, drift = PI._inside(PI.AP_ELLIPSE, x, y, lim, False), pair(3)[0]
    else:
        mx, my = f64[w + 1], pair(1)[0]
        lim = np.array([pair(1)[1], pair(2)[0], pair(2)[1], pair(3)[0]])
        inside = (x >= -mx) & (x <= mx) & (y >= -my) & (y <= my) & PI._inside(PI.AP_ELLIPSE, x, y, lim, False)
        drift = pair(4)[0]
    _lose(p, ~inside, elem)
    if aux & 0x10:
        (PI._drift_exact if aux & 0x20 else PI._drift)(p, drift)


def track(packed, cols, p0c, mass0, num_turns=1):
    """Interpret ``packed`` (fast encoding, no segments) for ``num_turns`` turns; ``cols`` may hold
    ``at_turn``.  Returns the full-length columns like ``packed_interpreter.track``."""
    assert packed.segments is None and not packed.strict
    words = np.ascontiguousarray(packed.words, dtype=np.uint64)
    f64, i64 = words.view(np.float64), words.view(np.int64)
    beam = PI._Beam(cols, p0c, mass0)
    beam.at_turn = np.array(np.broadcast_to(np.asarray(cols.get("at_turn", 0), dtype=np.int64), (beam.n,)))
    cw = packed.chunk_words
    for _ in range(num_turns):
        p = PI._Live(beam)
        done = False
        s_pass = 0.0
        for ch in range(packed.n_chunks):
            if done:
                break
            w = ch * cw
            while True:
                hdr = int(words[w])
                tag, aux, size, elem = hdr & 0xFF, (hdr >> 8) & 0xFF, (hdr >> 16) & 0x3FFF, hdr >> 32
                assert w % 2 == 0 and w + 2 * size <= (ch + 1) * cw, "record straddles a chunk"
                p0 = f64[w + 1]
                nxt = w + 2 * size
                if tag == PI.T_END_CHUNK:
                    break
                if tag == PI.T_END_TURN:
                    assert p0 == s_pass, "END_TURN must carry the length of the pass"
                    done = True
                    break
                s_at, adv = PI._path_length_words(tag, aux, w, f64, i64)
                if s_at is not None:
                    assert f64[s_at] == s_pass, "s_here of record at word %d" % w
                s_pass = s_pass + adv
                if len(p) == 0:
                    w = nxt
                    continue
                if (tag & 0xE0) == 0x80:  # thin block: kick, aperture, drift
                    pairs = f64[w + 4: w + 4 + 2 * (aux + 1)].reshape(aux + 1, 2)
                    t = 2 + aux + 1
                    dpx, dpy = PI._horner(p, pairs, aux, False)
                    curved = None
                    if tag & 4:
                        curved = tuple(f64[w + 2 * t: w + 2 * t + 4])
                        t += 2
                    p.px, p.py, p.zeta = PI._kick(p, dpx, dpy, curved, False, k0=pairs[aux])
                    if tag & 3:
                        lim = f64[w + 2 * t: w + 2 * t + 4]
                        _lose(p, ~PI._inside(tag & 3, p.x, p.y, lim, False), int(i64[w + 2]))
                    PI._closing_drift(p, tag, p0)
                elif (tag & 0xC0) == 0xC0:  # dipole edge -> [drift]
                    e = f64[w + 2: w + 4]
                    p.px = p.px + e[0] * p.x
                    p.py = p.py + e[1] * p.y
                    PI._closing_drift(p, tag, p0)
                elif tag == T_EXCITER:
                    _exciter(p, beam, f64, i64, w, aux)
                elif tag == PI.T_DRIFT:
                    PI._drift(p, p0)
                elif tag == PI.T_DRIFT_EXACT:
                    PI._drift_exact(p, p0)
                elif tag in (PI.T_MULTIPOLE, PI.T_MULTIPOLE_CURVED):
                    PI._multipole(p, f64, w, tag, aux, False)
                elif tag == PI.T_MULTIPOLE_RAD:
                    PI._multipole_rad(p, beam, words, f64, i64, w, aux, elem, False)
                elif tag in (PI.T_LIMIT_RECT, PI.T_LIMIT_ELLIPSE, PI.T_LIMIT_RECT_ELLIPSE):
                    _limit(p, tag, aux, w, f64, elem)
                elif tag == PI.T_XYSHIFT:
                    p.x = p.x - p0
                    p.y = p.y - f64[w + 2]
                elif tag == PI.T_SROTATION:
                    cz, sz = p0, f64[w + 2]
                    p.x, p.y = cz * p.x + sz * p.y, -sz * p.x + cz * p.y
                    p.px, p.py = cz * p.px + sz * p.py, -sz * p.px + cz * p.py
                elif tag == PI.T_DIPOLE_EDGE:
                    p.px = p.px + p0 * p.x
                    p.py = p.py + f64[w + 2] * p.y
                elif tag == PI.T_CAVITY:
                    k, lag = f64[w + 2], f64[w + 3]
                    wave = np.sin(lag - k * (p.zeta / p.rvv / beam.beta0))
                    PI._add_to_energy(p, beam, p.charge_ratio * beam.q0 * p0 * wave)
                elif tag != PI.T_MONITOR:
                    raise NotImplementedError("tag 0x%02x is outside this interpreter's scope" % tag)
                w = nxt
        assert done, "lattice without END_TURN"
        p.commit()
        beam.at_turn[p.idx] += 1
    return beam.result()
