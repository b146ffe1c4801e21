"""``Line``: the reference's element container (``xline/line.py:24-490``) whose ``track``
is served by the fused sm_100a kernel instead of the Python loop at
``xline/line.py:89-95``.

``Line.track(p)`` keeps the reference's signature (one pass over the elements, in place,
returns ``None``); ``num_turns`` fuses the caller's turn loop into the same launch.
"""
import ctypes as C
import json

import numpy as np
import torch

from . import _cabi
from . import elements as E
from .lattice import F_LOW_ORDER, MONITOR_FIELDS, algorithmic_ops, check_radiation, element_specs, pack_line

_thick = (E.Drift, E.DriftExact)
deg2rad = np.pi / 180.0


def _is_thick(element):
    """xline/line.py:12-14."""
    return bool(getattr(element, "isthick", False)) or isinstance(element, _thick)


def _c_particles(p):
    """``(xlb_particles_t, {column: tensor})`` over the columns of ``p`` (made contiguous in place)."""
    cols = {}
    for k, t in p._columns():
        if not t.is_contiguous():
            t = t.contiguous()
            p._assign(k, t)
        cols[k] = t
    cp = _cabi.Particles()
    cp.n = len(p)
    for k, t in cols.items():
        setattr(cp, k, t.data_ptr())
    cp.q0, cp.mass0, cp.p0c = p.q0, p.mass0, p.p0c
    cp.beta0, cp.gamma0, cp.energy0 = p.beta0, p.gamma0, p.energy0
    return cp, cols


class Line(E.Element):
    _base = (("elements", tuple), ("element_names", tuple))
    _pack_options = ("fuse_records", "chunk_words", "merge_multipoles", "split_lenses", "flag_horizontal_bends",
                     "polygon_apertures", "radiation", "radiation_seed")

    def __setattr__(self, name, value):
        # edit tracking (elements.py): the element list and the packing options stamp the line,
        # everything else (caches, outputs such as loss_tally / last_stats) is plain state
        if name in ("elements", "element_names"):
            E.Element.__setattr__(self, name, list(value))
        else:
            object.__setattr__(self, name, value)
            if name in self._pack_options:
                E._touch(self)

    def __init__(self, elements=(), element_names=None):
        self.elements = list(elements)
        if element_names is None:
            element_names = ["e%d" % i for i in range(len(self.elements))]
        self.element_names = list(element_names)
        assert len(self.elements) == len(self.element_names)  # xline/line.py:38
        self._cache = {}
        self.fuse_records = True  # pack-time peephole: multipole -> aperture -> drift in one record
        self.chunk_words = None   # 8-byte words per TMA chunk (None = lattice.DEFAULT_CHUNK_WORDS)
        self.merge_multipoles = True  # fast encoding: co-located thin multipoles become one kick
        self.split_lenses = True      # fast encoding: BeamBeam6D lenses run as kernels of their own
        self.flag_horizontal_bends = True  # fast encoding: XLB_HDR_HX_ONLY on curved blocks with hyl == 0
        # track LimitPolygon apertures with the project's even-odd rule (include/xline_b200.h); off,
        # a line that holds one refuses to pack, like the reference's LimitPolygon.track
        self.polygon_apertures = False
        # synchrotron radiation in every Multipole of length > 0: None (off), "mean" or "quantum", and
        # the seed of its counter-based random stream (include/xline_b200.h, DESIGN.md §4.9)
        self.radiation = None
        self.radiation_seed = 0
        self._monitor_buf = None
        self._buffers_key = None
        self.loss_tally = None
        self.last_stats = None

    def __len__(self):
        assert len(self.elements) == len(self.element_names)
        return len(self.elements)

    # ------------------------------------------------------------------ serialisation
    def to_dict(self, keepextra=True):
        out = {"elements": [], "element_names": list(self.element_names)}
        for el in self.elements:
            d = el.to_dict(keepextra)
            d.pop("data", None)
            out["elements"].append(d)
        return out

    @classmethod
    def from_dict(cls, dct, keepextra=True):
        classes = E.element_classes()
        els = []
        for d in dct["elements"]:
            kind = classes[d["__class__"]]
            d = dict(d)
            if kind is E.BeamMonitor:
                d.setdefault("data", [])
            els.append(kind.from_dict(d, keepextra))
        return cls(elements=els, element_names=list(dct["element_names"]))

    def to_json(self, filename, keepextra=True):
        def enc(o):
            if isinstance(o, np.ndarray):
                return o.tolist()
            if isinstance(o, (np.floating, np.integer, np.bool_)):
                return o.item()
            raise TypeError(type(o))

        with open(filename, "w") as fh:
            json.dump(self.to_dict(keepextra), fh, default=enc)

    @classmethod
    def from_json(cls, filename, keepextra=True):
        with open(filename) as fh:
            return cls.from_dict(json.load(fh), keepextra)

    def copy(self, keepextra=True):
        return Line.from_dict(self.to_dict(keepextra), keepextra)

    # ------------------------------------------------------------------ editing (host)
    def invalidate(self):
        """Drop the packed-lattice cache, the loss tallies and the monitor storage.  Edits made
        through the elements or the line (``el.voltage = ...``, ``el.knl[1] = ...``,
        ``line.elements.append(...)``) are noticed by ``pack`` on their own (edit tracking,
        ``elements.py``); this call is for what tracking cannot see -- elements of foreign classes
        (the reference's own, duck-typed) edited in place."""
        self._cache.clear()
        self._monitor_buf = None
        self._buffers_key = None
        self.loss_tally = None

    def insert_element(self, idx, element, name):
        self.elements.insert(idx, element)
        self.element_names.insert(idx, name)
        self.invalidate()
        return self

    def append_element(self, element, name):
        self.elements.append(element)
        self.element_names.append(name)
        self.invalidate()
        return self

    def append_line(self, line):
        self.elements += list(line.elements)
        self.element_names += list(line.element_names)
        self.invalidate()
        return self

    def get_length(self):  # xline/line.py:122-130
        return sum(el.length for el in self.elements if _is_thick(el))

    def get_s_elements(self, mode="upstream"):  # xline/line.py:132-144
        assert mode in ("upstream", "downstream")
        s, out = 0.0, []
        for el in self.elements:
            if mode == "upstream":
                out.append(s)
            if _is_thick(el):
                s += el.length
            if mode == "downstream":
                out.append(s)
        return out

    def get_elements_of_type(self, types):
        if not hasattr(types, "__iter__"):
            types = (types,)
        types = tuple(types)
        pairs = [(el, nm) for el, nm in zip(self.elements, self.element_names) if isinstance(el, types)]
        return [p[0] for p in pairs], [p[1] for p in pairs]

    def _filtered(self, keep):
        els, names = [], []
        for el, nm in zip(self.elements, self.element_names):
            if keep(el):
                els.append(el)
                names.append(nm)
        return Line(els, names)

    def remove_inactive_multipoles(self, inplace=False):  # xline/line.py:146-166
        new = self._filtered(lambda el: not (isinstance(el, E.Multipole) and not np.any(el.knl)
                                             and not np.any(el.ksl) and el.hxl == 0 and el.hyl == 0))
        return self._adopt(new) if inplace else new

    def remove_zero_length_drifts(self, inplace=False):  # xline/line.py:168-184
        new = self._filtered(lambda el: not (isinstance(el, _thick) and el.length == 0.0))
        return self._adopt(new) if inplace else new

    def merge_consecutive_drifts(self, inplace=False):  # xline/line.py:186-211
        els, names = [], []
        for el, nm in zip(self.elements, self.element_names):
            if els and isinstance(el, _thick) and isinstance(els[-1], _thick):
                els[-1] = type(els[-1])(length=els[-1].length + el.length)  # keeps the first one's kind
                names[-1] = names[-1] + "_" + nm
            else:
                els.append(el.copy() if isinstance(el, _thick) else el)
                names.append(nm)
        new = Line(els, names)
        return self._adopt(new) if inplace else new

    def merge_consecutive_multipoles(self, inplace=False):  # xline/line.py:213-251
        els, names = [], []
        for el, nm in zip(self.elements, self.element_names):
            prev = els[-1] if els else None
            if (isinstance(el, E.Multipole) and isinstance(prev, E.Multipole)
                    and prev.hxl == el.hxl and prev.hyl == el.hyl):
                n = max(len(prev.knl), len(prev.ksl), len(el.knl), len(el.ksl))
                knl, ksl = np.zeros(n), np.zeros(n)
                for src in (prev, el):
                    knl[: len(src.knl)] += np.asarray(src.knl, dtype=float)
                    ksl[: len(src.ksl)] += np.asarray(src.ksl, dtype=float)
                els[-1] = E.Multipole(knl=list(knl), ksl=list(ksl), hxl=prev.hxl, hyl=prev.hyl,
                                      length=prev.length)
                names[-1] = names[-1] + "_" + nm
            else:
                els.append(el)
                names.append(nm)
        new = Line(els, names)
        return self._adopt(new) if inplace else new

    def get_element_ids_of_type(self, types, start_idx_offset=0):  # xline/line.py:270-282
        assert start_idx_offset >= 0
        types = tuple(types) if hasattr(types, "__iter__") else (types,)
        return [i + start_idx_offset for i, el in enumerate(self.elements) if isinstance(el, types)]

    # ---- error handling (alignment, multipole errors): xline/line.py:328-415 ------------
    def find_element_ids(self, element_name):
        """Index of the element and the index just after it, any ``<name>_aperture`` element
        that follows included (xline/line.py:330-348)."""
        idx_el = self.element_names.index(element_name)
        try:
            idx_after = self.element_names.index(element_name + "_aperture") + 1
        except ValueError:
            idx_after = idx_el + 1
        return idx_el, idx_after

    def _add_offset_error_to(self, element_name, dx=0, dy=0):  # xline/line.py:350-358
        idx_el, idx_after = self.find_element_ids(element_name)
        self.insert_element(idx_el, E.XYShift(dx=dx, dy=dy), element_name + "_offset_in")
        self.insert_element(idx_after + 1, E.XYShift(dx=-dx, dy=-dy), element_name + "_offset_out")

    def _add_aperture_offset_error_to(self, element_name, arex=0, arey=0):  # xline/line.py:360-373
        idx_el, idx_after = self.find_element_ids(element_name)
        idx_aper = idx_after - 1
        if self.element_names[idx_aper] != element_name + "_aperture":
            print("Info: Element", element_name, ": arex/y provided without aperture -> arex/y ignored")
            return
        self.insert_element(idx_aper, E.XYShift(dx=arex, dy=arey), element_name + "_aperture_offset_in")
        self.insert_element(idx_after + 1, E.XYShift(dx=-arex, dy=-arey),
                            element_name + "_aperture_offset_out")

    def _add_tilt_error_to(self, element_name, angle):  # xline/line.py:375-400 (angle in degrees)
        idx_el, idx_after = self.find_element_ids(element_name)
        element = self.elements[idx_el]
        if isinstance(element, E.Multipole) and (element.hxl or element.hyl):
            dpsi = angle * deg2rad
            hxl0, hyl0 = element.hxl, element.hyl
            element.hxl = hxl0 * np.cos(dpsi) - hyl0 * np.sin(dpsi)
            element.hyl = hxl0 * np.sin(dpsi) + hyl0 * np.cos(dpsi)
        self.insert_element(idx_el, E.SRotation(angle=angle), element_name + "_tilt_in")
        self.insert_element(idx_after + 1, E.SRotation(angle=-angle), element_name + "_tilt_out")

    def _add_multipole_error_to(self, element_name, knl=(), ksl=()):  # xline/line.py:402-415
        assert element_name in self.element_names
        element = self.elements[self.element_names.index(element_name)]
        for attr, extra in (("knl", knl), ("ksl", ksl)):
            extra = np.trim_zeros(np.asarray(extra, dtype=float), trim="b")
            cur = list(getattr(element, attr))
            cur += [0] * (len(extra) - len(cur))
            for i, c in enumerate(extra):
                cur[i] = float(cur[i] + c)
            setattr(element, attr, cur)
        self.invalidate()

    def _adopt(self, other):
        self.elements, self.element_names = other.elements, other.element_names
        self.invalidate()
        return self

    # ------------------------------------------------------------------ packing
    def to_specs(self):
        """``[(type_name, fields), ...]`` -- neutral description (tests feed it to the oracle)."""
        return element_specs(self.elements)

    def algorithmic_ops_per_turn(self):
        return algorithmic_ops(self.elements, self.radiation)

    def _content_stamp(self):
        """(ids of the elements, newest edit stamp among them and the line): changes whenever the
        element list or a tracked field changed.  O(len) -- only evaluated when the global edit
        clock moved since the last look."""
        newest = self.__dict__.get("_rev", 0)
        for el in self.elements:
            r = el.__dict__.get("_rev", 0) if hasattr(el, "__dict__") else 0
            if r > newest:
                newest = r
        return (tuple(map(id, self.elements)), newest)

    def _current_stamp(self):
        clock = E.edit_clock()
        seen = self._cache.get("stamp")
        if seen is not None and seen[0] == clock and seen[2] == len(self.elements):
            return seen[1]
        stamp = self._content_stamp()
        if seen is None or seen[1] != stamp:
            self._cache.clear()  # the line changed: packed lattices and device copies are stale
            self._cache["generation"] = Line._generations = getattr(Line, "_generations", 0) + 1
        self._cache["stamp"] = (clock, stamp, len(self.elements))
        return stamp

    def pack(self, strict=False, chunk_words=None):
        """Host-side packed lattice (``lattice.PackedLattice``), cached until the line or one of
        its elements is edited."""
        if chunk_words is None:
            chunk_words = self.chunk_words
        self._current_stamp()
        key = ("host", bool(strict), chunk_words, self.fuse_records, self.merge_multipoles, self.split_lenses,
               self.flag_horizontal_bends, self.polygon_apertures, self.radiation, self.radiation_seed,
               getattr(self, "_keep_noops", False))
        hit = self._cache.get("host_%d" % strict)
        if hit is not None and hit[0] == key:
            return hit[1]
        kw = {} if chunk_words is None else {"chunk_words": chunk_words}
        packed = pack_line(self.elements, strict=strict, fuse=self.fuse_records,
                           merge=self.merge_multipoles, split_lenses=self.split_lenses,
                           hx_only=self.flag_horizontal_bends, polygons=self.polygon_apertures,
                           radiation=self.radiation, radiation_seed=self.radiation_seed,
                           drop_noops=not getattr(self, "_keep_noops", False), **kw)
        lat = packed.c_lattice()
        _cabi.check(_cabi.lib().xlb_lattice_validate(C.byref(lat)))
        self._cache["host_%d" % strict] = (key, packed)
        return packed

    def _device_lattice(self, device, strict):
        packed = self.pack(strict)
        key = ("dev", str(device), bool(strict), id(packed))
        hit = self._cache.get(key[:3])
        if hit is not None and hit[0] == key:
            return packed, hit[1]
        words = torch.from_numpy(packed.words.view(np.int64)).to(device)
        self._cache[key[:3]] = (key, words)
        return packed, words

    # ------------------------------------------------------------------ the hot path
    def track(self, p, num_turns=1, strict=False, turns_per_launch=0, particles_per_thread=0,
              threads_per_block=0, timed=False, turns_per_item=0, compact_threshold=0.0, moments=None,
              _trace=None, _count_turns=True,
              _element_offset=0, _general_kernels=False):
        """``for el in self.elements: el.track(p)`` (xline/line.py:89-95), ``num_turns``
        times, in one fused kernel launch on ``p``'s GPU.  Mutates ``p`` in place and
        returns ``None`` like the reference.

        ``strict=True`` selects the reference-operation-order kernel (parity instrument).
        ``turns_per_launch`` > 0 splits the job and re-compacts survivors between launches
        (when more than ``compact_threshold`` of the lanes went idle; 0 = the library's 1/128).
        ``moments``: a ``BeamMoments`` that receives the beam moments on its store turns of this
        call (``xline_b200.moments``); the particles are tracked exactly as without.
        """
        if p.device.type != "cuda":
            raise RuntimeError(
                "xline_b200.Line.track needs particles resident on a CUDA device (got %s); "
                "there is no CPU tracking path in this package" % p.device)
        if self.radiation is not None:
            check_radiation(self.radiation, self.radiation_seed)
            if strict:
                raise ValueError("radiation: strict=True has no radiating kernel (set Line.radiation = None)")
        lib = _cabi.lib()
        dev = p.x.device  # the tensors' own (indexed) device: torch.device("cuda") != torch.device("cuda:0")
        with torch.cuda.device(dev):
            packed, words = self._device_lattice(dev, strict)
            n = len(p)
            if moments is not None:
                moments._check_target(p)
            elif n == 0 or num_turns == 0:
                return None
            lat = packed.c_lattice(words.data_ptr())
            if _general_kernels:  # test hook: the unspecialised kernel family (chi column, any order)
                lat.flags &= ~F_LOW_ORDER
            cp, cols = _c_particles(p)
            # one species (chi == 1 throughout, the reference's default) is the fast case of the C ABI:
            # no chi column is handed over and the kernels without a chi register run (4 particles per
            # thread).  The answer is cached on the tensor's storage and version counter, so an in-place
            # edit of p.chi is seen on the next call.
            chi = cols.get("chi")
            if chi is not None:
                ckey = (chi.data_ptr(), chi._version, n)
                if getattr(p, "_chi_key", None) != ckey:
                    p._chi_key, p._chi_trivial = ckey, bool((chi == 1.0).all())
                if p._chi_trivial and not _general_kernels:
                    cp.chi = None
                elif self.radiation is not None:
                    raise ValueError("radiation: one species only -- every chi must be 1 (set Line.radiation = None)")
            # tallies and monitor storage belong to one state of the line on one device: a line that
            # was edited since (other element count, other monitor layout) gets fresh ones
            bkey = (self._cache.get("generation"), packed.n_elements, packed.monitor_words, dev)
            if self._buffers_key != bkey or self.loss_tally is None:
                self.loss_tally = torch.zeros(max(packed.n_elements, 1), dtype=torch.int64, device=dev)
                self._monitor_buf = None
                self._buffers_key = bkey
            if particles_per_thread == 0 and (packed.flags & 2) and not strict:
                # beam-field lattice: the thin-lens records still dominate when lenses are
                # sparse (LHC + 74 lenses: 3 particles/thread wins); dense space-charge
                # lattices prefer fewer (PS Booster with 120 kicks/turn: 1.57e8 / 1.91e8 / 1.59e8
                # particle-turns/s for 1 / 2 / 3; the kernels that carry the 6D lens spill and
                # are best with 1)
                nbf = sum(v for k, v in packed.record_counts.items() if k in (16, 17, 18))
                sparse = nbf < 0.05 * max(sum(packed.record_counts.values()), 1)
                dense_ppt = 1 if (packed.record_counts.get(18, 0) and packed.segments is None) else 2
                particles_per_thread, threads_per_block = ((3, threads_per_block or 128) if sparse
                                                           else (dense_ppt, threads_per_block or 256))
            opts = _cabi.TrackOptions()
            opts.num_turns = int(num_turns)
            opts.particles_per_thread = int(particles_per_thread)
            opts.threads_per_block = int(threads_per_block)
            opts.turns_per_launch = int(turns_per_launch)
            opts.turns_per_item = int(turns_per_item)
            opts.compact_threshold = float(compact_threshold)
            opts.flags = 0 if _count_turns else _cabi.OPT_NO_TURN_COUNT
            opts.element_index_offset = int(_element_offset)
            if _trace is not None:
                opts.trace = _trace.data_ptr()
                opts.trace_particles = int(_trace.shape[2])
            opts.loss_tally = self.loss_tally.data_ptr()
            if packed.monitor_words > 0:
                if self._monitor_buf is None:
                    self._monitor_buf = torch.full((packed.monitor_words,), float("nan"),
                                                   dtype=torch.float64, device=dev)
                opts.monitor_data = self._monitor_buf.data_ptr()
                opts.monitor_words = packed.monitor_words
            stream = torch.cuda.current_stream(dev).cuda_stream
            if moments is not None:
                if timed:
                    raise ValueError("timed=True does not combine with moments")
                _cabi.check(lib.xlb_track_device_moments(C.byref(lat), C.byref(cp), C.byref(opts),
                                                         C.byref(moments._spec()), C.c_void_p(moments.data.data_ptr()),
                                                         C.c_void_p(stream)))
                moments.beta0gamma0 = p.beta0 * p.gamma0
            else:
                fn = lib.xlb_track_device_timed if timed else lib.xlb_track_device
                _cabi.check(fn(C.byref(lat), C.byref(cp), C.byref(opts), C.c_void_p(stream)))
            self.last_stats = _cabi.stats()
            if packed.monitor_words > 0:
                self._publish_monitors(packed)
        return None

    def _publish_monitors(self, packed):
        for slot in packed.monitor_layout:
            el = self.elements[slot["element_index"]]
            ns, nn = slot["num_stores"], slot["nn"]
            if ns <= 0 or nn <= 0:
                continue
            view = self._monitor_buf[slot["offset"]: slot["offset"] + len(MONITOR_FIELDS) * ns * nn]
            view = view.view(len(MONITOR_FIELDS), ns, nn)
            el.data = {k: view[i] for i, k in enumerate(MONITOR_FIELDS)}

    def reset_monitors(self):
        if self._monitor_buf is not None:
            self._monitor_buf.fill_(float("nan"))

    def trace_elem_by_elem(self, p, max_particles=None, strict=False):
        """Device form of ``track_elem_by_elem`` (xline/line.py:97-108): one pass over the line
        with the debug kernel, returning a tensor ``[len(self) + 1, 6, K]`` -- row 0 the
        starting coordinates, row ``i + 1`` the coordinates (x, px, y, py, zeta, delta) of the
        first ``K = max_particles`` particles after element ``i``; NaN from the element where
        a particle was lost.  ``p`` is tracked in place.  The line is packed element by element
        (no record fusing, no merging, no-ops kept) so every element owns a row."""
        n = len(p)
        k_ = n if max_particles is None else min(int(max_particles), n)
        # temporary packing options with a cache of their own; set without stamping the line, so the
        # regular packed lattice stays valid afterwards
        names = ("fuse_records", "merge_multipoles", "split_lenses", "_cache", "_buffers_key", "loss_tally",
                 "_monitor_buf")
        saved = {k: self.__dict__[k] for k in names}
        for k, v in zip(names, (False, False, False, {}, None, None, None)):
            object.__setattr__(self, k, v)
        self._keep_noops = True
        try:
            trace = torch.full((len(self) + 1, 6, k_), float("nan"), dtype=torch.float64, device=p.device)
            for f, name in enumerate(("x", "px", "y", "py", "zeta", "delta")):
                trace[0, f] = getattr(p, name)[:k_]
            self.track(p, num_turns=1, strict=strict, _trace=trace[1:])
        finally:
            self._keep_noops = False
            for k, v in saved.items():
                object.__setattr__(self, k, v)
        return trace

    def _tangent_lattice(self, device, radiation=False):
        """The element-by-element packing of ``trace_elem_by_elem`` (one record per element: no
        record fusing, no merging, no split lenses, no-ops kept) in the fast encoding, with a cache
        entry of its own, and its copy on ``device``.  ``radiation=True``: the same packing with every
        Multipole of length > 0 a mean-mode radiating record, whatever ``self.radiation`` is (the
        tangent map and the envelope linearise about the mean-mode orbit), under a key of its own."""
        self._current_stamp()
        name = "tangent_rad" if radiation else "tangent"
        key = (name, self.chunk_words, self.flag_horizontal_bends, self.polygon_apertures, str(device))
        hit = self._cache.get(name)
        if hit is not None and hit[0] == key:
            return hit[1], hit[2]
        kw = {} if self.chunk_words is None else {"chunk_words": self.chunk_words}
        if radiation:
            kw["radiation"] = "mean"
        packed = pack_line(self.elements, strict=False, fuse=False, merge=False, split_lenses=False,
                           hx_only=self.flag_horizontal_bends, polygons=self.polygon_apertures,
                           drop_noops=False, **kw)
        _cabi.check(_cabi.lib().xlb_lattice_validate(C.byref(packed.c_lattice())))
        words = torch.from_numpy(packed.words.view(np.int64)).to(device)
        self._cache[name] = (key, packed, words)
        return packed, words

    def track_tangent(self, p, tangent, num_turns=1, threads_per_block=0, radiation=False):
        """Track ``p`` as ``track`` would, ``num_turns`` turns, and carry the Jacobian of every
        particle in ``tangent`` (a ``TangentMap`` of ``len(p)`` particles): both are updated in
        place, and a second call continues where the first stopped.  Returns ``None``.  Losses,
        ``at_element``, ``at_turn`` and ``loss_tally`` behave as in ``track``; a lost particle's
        Jacobian and FLI are frozen where it was lost.  Monitors store nothing here.  BeamBeam6D
        lenses are refused (``ValueError``).  A radiating line is refused unless ``radiation=True``,
        which differentiates the mean-mode radiation too (a ``"quantum"`` line is refused: the random
        map has no tangent); on a line without radiation ``radiation=True`` changes nothing.  See
        ``xline_b200.tangent``."""
        from .tangent import track_tangent

        return track_tangent(self, p, tangent, num_turns=num_turns, threads_per_block=threads_per_block,
                             radiation=radiation)

    def track_envelope(self, p, envelope, num_turns=1, threads_per_block=0):
        """Track ``p`` as ``track_tangent`` would and carry, per particle, the second moment ``Sigma``
        of a beam around it in ``envelope`` (an ``Envelope`` of ``len(p)`` particles): every element
        maps ``Sigma -> J Sigma J^T``; on a radiating line (``"mean"`` or ``"quantum"``) the particle
        follows the mean-mode map and every radiating half adds the variance of the quantum mode's
        energy loss, and ``envelope.energy_loss`` accumulates the energy radiated (eV).  Both are
        updated in place.  See ``xline_b200.tangent``."""
        from .tangent import track_envelope

        return track_envelope(self, p, envelope, num_turns=num_turns, threads_per_block=threads_per_block)

    def track_elem_by_elem(self, p, start=True, end=False):
        """Debug path (xline/line.py:97-108): one single-element launch per element,
        returning the copies of ``p`` the reference returns.  As there, the turn counter is not
        touched; a particle lost on the way records the index of the element in THIS line."""
        out = []
        if start:
            out.append(p.copy())
        for i, el in enumerate(self.elements):
            solo = self._cache.get(("solo", i))
            if solo is None or solo.elements[0] is not el:
                solo = self._cache[("solo", i)] = Line([el], ["e"])
            for opt in ("polygon_apertures", "radiation", "radiation_seed"):
                if getattr(solo, opt) != getattr(self, opt):
                    setattr(solo, opt, getattr(self, opt))
            solo.track(p, _count_turns=False, _element_offset=i)
            out.append(p.copy())
        if end:
            out.append(p.copy())
        return out

    # ------------------------------------------------------------------ loaders
    @classmethod
    def from_madx_sequence(cls, sequence, classes=None, ignored_madtypes=(), exact_drift=False,
                           drift_threshold=1e-6, install_apertures=False, apply_madx_errors=False):
        """xline/line.py:297-324 for a thin ``madx_input.MadSequence`` (or any object with
        ``elements`` / ``element_positions()`` / ``length`` like a cpymad sequence)."""
        from .madx_input import iter_from_madx_sequence

        names, els = [], []
        for nm, el in iter_from_madx_sequence(sequence, classes or E.element_classes(), ignored_madtypes,
                                              exact_drift, drift_threshold, install_apertures):
            names.append(nm)
            els.append(el)
        line = cls(els, names)
        if apply_madx_errors:
            line._apply_madx_errors(sequence)
        return line

    def _apply_madx_errors(self, madx_sequence):
        """xline/line.py:417-489: turn the alignment / field errors attached to the elements of
        the expanded MAD-X sequence into XYShift / SRotation wrappers and multipole
        coefficients.  Returns the names of elements that carry errors but are not in this line."""
        not_found = []
        for element, name in zip(madx_sequence.expanded_elements, madx_sequence.expanded_element_names()):
            if name not in self.element_names:
                if element.align_errors or element.field_errors:
                    not_found.append(name)
                    continue
            if element.align_errors:
                err = element.align_errors
                if err.dx or err.dy:
                    self._add_offset_error_to(name, err.dx, err.dy)
                if err.dpsi:
                    self._add_tilt_error_to(name, angle=err.dpsi / deg2rad)
                if err.arex or err.arey:
                    self._add_aperture_offset_error_to(name, err.arex, err.arey)
            if element.field_errors:
                dkn, dks = np.asarray(element.field_errors.dkn), np.asarray(element.field_errors.dks)
                if dkn.any() or dks.any():
                    last = max(np.flatnonzero(dkn)[-1] if dkn.any() else 0,
                               np.flatnonzero(dks)[-1] if dks.any() else 0) + 1
                    self._add_multipole_error_to(name, dkn[:last], dks[:last])
        return not_found

    @classmethod
    def from_sixinput(cls, sixinput, classes=None):
        """xline/line.py:279-295 with this package's SixTrack reader."""
        from .sixtrack_input import expand_struct

        line_data, rest, iconv = expand_struct(sixinput, classes or E.element_classes())
        line = cls([el for _, _, el in line_data], [nm for nm, _, _ in line_data])
        line.other_info = {"rest": rest, "iconv": iconv}
        return line
