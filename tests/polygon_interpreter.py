"""TEST INFRASTRUCTURE -- a NumPy interpreter of packed lattices that hold LIMIT_POLYGON records.

Walks the words of ``xline_b200.lattice.pack_line(..., polygons=True)`` as include/xline_b200.h
documents them, with the element maps and bookkeeping of ``tests/packed_interpreter.py`` (whose
helpers it uses), for the record kinds the polygon tests pack: thin blocks, drifts, straight
multipoles, XYShift, SRotation, the LIMIT_* apertures with their fused drifts and LIMIT_POLYGON.
Any other record raises.  Strict encoding: bit for bit the oracle; fast: to rounding.
"""
import numpy as np

from tests import packed_interpreter as PI

T_LIMIT_POLYGON = 19


def polygon_inside(f64, i64, w, x, y):
    """[hdr,n_edges][s_here,drift] then [y_lo,y_hi][x_lo,slope] per edge, at word ``w``."""
    n_edges = int(i64[w + 1])
    odd = np.zeros(len(x), dtype=bool)
    for y_lo, y_hi, x_lo, slope in f64[w + 4: w + 4 + 4 * n_edges].reshape(-1, 4):
        assert y_lo < y_hi
        with np.errstate(invalid="ignore"):  # inf * 0 for an infinite y at a vertical edge
            odd ^= (y >= y_lo) & (y < y_hi) & (x < x_lo + (y - y_lo) * slope)
    return odd


def _path_length_words(tag, aux, w, f64, i64):
    if tag == T_LIMIT_POLYGON:
        return w + 2, (f64[w + 3] if aux & 0x10 else 0.0)
    return PI._path_length_words(tag, aux, w, f64, i64)


def _fused_drift(p, aux, L):
    if aux & 0x10:
        (PI._drift_exact if aux & 0x20 else PI._drift)(p, L)


def track(packed, cols, p0c, mass0, num_turns=1):
    """Interpret ``packed`` (no segments, no monitors) for ``num_turns`` turns."""
    assert packed.segments is None
    words = np.ascontiguousarray(packed.words, dtype=np.uint64)
    f64, i64 = words.view(np.float64), words.view(np.int64)
    strict = packed.strict
    beam = PI._Beam(cols, p0c, mass0)
    cw = packed.chunk_words
    for turn in range(num_turns):
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
                assert w + 2 * size <= (ch + 1) * cw, "record straddles a chunk"
                p0 = f64[w + 1]
                pair = lambda m, _w=w: f64[_w + 2 * m: _w + 2 * m + 2]  # noqa: E731
                nxt = w + 2 * size
                if tag == PI.T_END_CHUNK:
                    break
                if tag == PI.T_END_TURN:
                    assert p0 == s_pass, "END_TURN must carry the length of the pass"
                    done = True
                    break
                s_at, adv = _path_length_words(tag, aux, w, f64, i64)
                if s_at is not None:
                    assert f64[s_at] == s_pass, "s_here of record at word %d" % w
                s_pass = s_pass + adv
                if len(p) == 0:
                    w = nxt
                    continue
                if (tag & 0xE0) == 0x80:  # thin block: kick -> [aperture] -> [drift]
                    order = aux
                    pairs = f64[w + 4: w + 4 + 2 * (order + 1)].reshape(order + 1, 2)
                    t = 2 + order + 1
                    dpx, dpy = PI._horner(p, pairs, order, strict)
                    curved = None
                    if tag & 4:
                        curved = (pair(t)[0], pair(t)[1], pair(t + 1)[0], pair(t + 1)[1])
                        t += 2
                    p.px, p.py, p.zeta = PI._kick(p, dpx, dpy, curved, strict, k0=pairs[order])
                    if tag & 3:
                        lim = np.concatenate([pair(t), pair(t + 1)])
                        p.lose(~PI._inside(tag & 3, p.x, p.y, lim, strict), int(i64[w + 2]), turn)
                    PI._closing_drift(p, tag, p0)
                elif tag == PI.T_DRIFT:
                    PI._drift(p, p0)
                elif tag == PI.T_DRIFT_EXACT:
                    PI._drift_exact(p, p0)
                elif tag == PI.T_MULTIPOLE:
                    pairs = f64[w + 2: w + 2 + 2 * (aux + 1)].reshape(aux + 1, 2)
                    dpx, dpy = PI._horner(p, pairs, aux, strict)
                    p.px, p.py, p.zeta = PI._kick(p, dpx, dpy, None, strict)
                elif tag == PI.T_XYSHIFT:
                    p.x = p.x - p0
                    p.y = p.y - pair(1)[0]
                elif tag == PI.T_SROTATION:
                    cz, sz = p0, pair(1)[0]
                    p.x, p.y = cz * p.x + sz * p.y, -sz * p.x + cz * p.y
                    p.px, p.py = cz * p.px + sz * p.py, -sz * p.px + cz * p.py
                elif tag in (PI.T_LIMIT_RECT, PI.T_LIMIT_ELLIPSE):
                    lim = np.array([p0, pair(1)[0], pair(1)[1], pair(2)[0]])
                    kind = PI.AP_ELLIPSE if tag == PI.T_LIMIT_ELLIPSE else (PI.AP_RECT_SYM if aux & 1 else PI.AP_RECT)
                    p.lose(~PI._inside(kind, p.x, p.y, lim, strict), elem, turn)
                    _fused_drift(p, aux, pair(3)[0])
                elif tag == T_LIMIT_POLYGON:
                    p.lose(~polygon_inside(f64, i64, w, p.x, p.y), elem, turn)
                    _fused_drift(p, aux, f64[w + 3])
                else:
                    raise NotImplementedError("tag 0x%02x is outside this interpreter's scope" % tag)
                w = nxt
        assert done, "lattice without END_TURN"
        p.commit()
        beam.at_turn[p.idx] += 1
    return beam.result()
