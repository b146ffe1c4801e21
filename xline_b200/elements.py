"""Element classes of the drop-in API (same names, fields, defaults and positional order
as the reference's ``xline/elements.py`` and ``xline/be_beamfields/*.py``).

The classes here carry *parameters only*.  All arithmetic happens in the CUDA kernel
(``csrc/track_impl.cuh``); ``Element.track(p)`` is a one-element ``Line.track``.  Field
tables below restate the reference's ``_description`` / ``_extra`` lists
(``xline/base_classes.py:24-52`` builds dataclasses from them); the generated classes
accept the fields as keyword or positional arguments in table order, list-valued
fields default to fresh lists, and they offer ``get_fields / to_dict / from_dict / copy``
like ``xline/base_classes.py:59-82``.
"""
import copy as _copy

import numpy as _np

__all__ = [
    "Element", "Drift", "DriftExact", "Multipole", "RFMultipole", "Cavity", "SawtoothCavity",
    "XYShift", "SRotation", "LimitRect", "LimitEllipse", "LimitRectEllipse", "BeamMonitor",
    "DipoleEdge", "BeamBeam4D", "BeamBeam6D", "SCCoasting", "SCQGaussProfile",
    "SCInterpolatedProfile", "Elens", "LimitPolygon", "Exciter", "element_classes",
]


# ---- edit tracking ---------------------------------------------------------------------------
# The reference reads element fields on every ``track`` call (xline/elements.py), so code written
# against it edits fields in place -- ``el.voltage = ...``, ``el.knl[1] = ...``,
# ``line.elements.append(...)`` -- and expects the next ``Line.track`` to see it.  Here the fields
# are packed once into the device lattice, so every edit made *through an element* (attribute
# assignment, item assignment / in-place arithmetic on a list- or array-valued field, mutation of
# ``Line.elements``) advances a global edit clock and stamps the owner with it; ``Line.pack``
# compares the clock (O(1) when nothing was edited anywhere) and re-packs when an element of the
# line carries a newer stamp.  List and array values are COPIED into tracked containers on
# assignment: the element owns its data, an edit of the caller's original object afterwards does
# not reach the element (the reference would alias it).
_EDIT_CLOCK = [0]


def edit_clock():
    return _EDIT_CLOCK[0]


def _touch(owner):
    _EDIT_CLOCK[0] += 1
    if owner is not None:
        object.__setattr__(owner, "_rev", _EDIT_CLOCK[0])


def _mutator(name):
    base = getattr(list, name)

    def method(self, *a, **k):
        out = base(self, *a, **k)
        _touch(self._owner)
        return out

    method.__name__ = name
    return method


class _FieldList(list):
    """``list`` that stamps its owner (an element or a line) on every mutation."""

    __slots__ = ("_owner",)

    def __init__(self, values=(), owner=None):
        list.__init__(self, values)
        self._owner = owner

    for _n in ("__setitem__", "__delitem__", "__iadd__", "__imul__", "append", "extend", "insert", "pop",
               "remove", "clear", "sort", "reverse"):
        locals()[_n] = _mutator(_n)
    del _n

    def __deepcopy__(self, memo):
        return [_copy.deepcopy(v, memo) for v in self]

    def __copy__(self):
        return list(self)

    def __reduce_ex__(self, protocol):
        return (list, (list(self),))


class _FieldArray(_np.ndarray):
    """``ndarray`` that stamps its owner on item assignment and in-place arithmetic."""

    _owner = None

    def __array_finalize__(self, obj):
        self._owner = getattr(obj, "_owner", None)

    def __setitem__(self, key, value):
        _np.ndarray.__setitem__(self, key, value)
        _touch(self._owner)

    def __array_ufunc__(self, ufunc, method, *inputs, out=None, **kwargs):
        plain = lambda v: v.view(_np.ndarray) if isinstance(v, _FieldArray) else v  # noqa: E731
        if out is not None:
            for o in out:
                if isinstance(o, _FieldArray):
                    _touch(o._owner)
            kwargs["out"] = tuple(plain(o) for o in out)
        return getattr(ufunc, method)(*[plain(v) for v in inputs], **kwargs)

    def __deepcopy__(self, memo):
        return _np.array(self, copy=True).view(_np.ndarray)

    def __reduce_ex__(self, protocol):
        return _np.array(self).view(_np.ndarray).__reduce_ex__(protocol)


def _tracked(value, owner):
    if isinstance(value, _np.ndarray):
        arr = _np.array(value, copy=True).view(_FieldArray)
        arr._owner = owner
        return arr
    if isinstance(value, list):
        return _FieldList(value, owner)
    return value


class Element:
    """Base of all elements.  ``_base`` / ``_extra`` are ``(name, default)`` tuples; a
    callable default is a factory (the reference writes list defaults as lambdas,
    ``xline/base_classes.py:10-21``)."""

    _base = ()
    _extra = ()
    _untracked = ("data",)  # BeamMonitor.data is an output, re-published after every track call
    iscollective = False  # xline/base_classes.py:57

    def __setattr__(self, name, value):
        if name.startswith("_") or name in self._untracked:
            object.__setattr__(self, name, value)
            return
        object.__setattr__(self, name, _tracked(value, self))
        _touch(self)

    def __init__(self, *args, **kwargs):
        names = [n for n, _ in self._base] + [n for n, _ in self._extra]
        if len(args) > len(names):
            raise TypeError(
                "%s takes at most %d positional arguments" % (type(self).__name__, len(names))
            )
        given = dict(zip(names, args))
        for k, v in kwargs.items():
            if k not in names:
                raise TypeError("%s got an unexpected field %r" % (type(self).__name__, k))
            if k in given:
                raise TypeError("%s got multiple values for %r" % (type(self).__name__, k))
            given[k] = v
        for n, d in tuple(self._base) + tuple(self._extra):
            if n in given:
                setattr(self, n, given[n])
            else:
                setattr(self, n, d() if callable(d) else d)

    # -- reference API (xline/base_classes.py:59-82) ---------------------------------
    @classmethod
    def _names(cls, keepextra):
        names = [n for n, _ in cls._base]
        if keepextra:
            names += [n for n, _ in cls._extra]
        return names

    @property
    def _fields(self):
        return self._names(True)

    @property
    def _base_fields(self):
        return self._names(False)

    @property
    def _extra_fields(self):
        return [n for n, _ in self._extra]

    def get_fields(self, keepextra=False):
        return self._names(keepextra)

    def to_dict(self, keepextra=False):
        out = {}
        for k in self._names(keepextra):
            v = getattr(self, k)
            if isinstance(v, _FieldList):  # plain containers outward (copies: edits go through the element)
                v = list(v)
            elif isinstance(v, _FieldArray):
                v = _np.array(v).view(_np.ndarray)
            out[k] = v
        out["__class__"] = type(self).__name__
        return out

    @classmethod
    def from_dict(cls, dct, keepextra=True):
        self = cls()
        for k in cls._names(False):
            setattr(self, k, dct[k])
        if keepextra:
            for k, _ in cls._extra:
                if k in dct:
                    setattr(self, k, dct[k])
        return self

    def copy(self, keepextra=True):
        return type(self).from_dict(_copy.deepcopy(self.to_dict(keepextra)), keepextra)

    def __repr__(self):
        body = ", ".join("%s=%r" % (k, getattr(self, k)) for k in self._names(True))
        return "%s(%s)" % (type(self).__name__, body)

    def __eq__(self, other):
        if type(other) is not type(self):
            return False
        a, b = self.to_dict(True), other.to_dict(True)
        if a.keys() != b.keys():
            return False
        for k, v in a.items():
            w = b[k]
            if isinstance(v, _np.ndarray) or isinstance(w, _np.ndarray):
                if not _np.array_equal(_np.asarray(v), _np.asarray(w)):
                    return False
            elif v != w:
                return False
        return True

    __hash__ = None

    # -- the operator the reference defines on every element -------------------------
    def track(self, p):
        """``el.track(p)``: push ``p`` through this single element on the GPU (in place).  Like the
        reference's ``el.track`` it does not touch the turn counter (``at_turn`` advances in
        ``Line.track`` only); the one-element lattice is cached on the element until it is edited."""
        from .line import Line

        solo = self.__dict__.get("_solo")
        if solo is None or solo[0] != self.__dict__.get("_rev"):
            solo = (self.__dict__.get("_rev"), Line(elements=[self], element_names=["e0"]))
            object.__setattr__(self, "_solo", solo)
        return solo[1].track(p, _count_turns=False)


def _zero_list():
    return [0]


class Drift(Element):
    """Drift in expanded form (xline/elements.py:43-56)."""

    _base = (("length", 0),)


class DriftExact(Drift):
    """Drift in exact form (xline/elements.py:59-72)."""

    _base = (("length", 0),)


class Multipole(Element):
    """Thin multipole, optional curvature terms (xline/elements.py:84-156)."""

    _base = (("knl", _zero_list), ("ksl", _zero_list), ("hxl", 0), ("hyl", 0), ("length", 0))

    @property
    def order(self):
        return max(len(self.knl), len(self.ksl)) - 1


class RFMultipole(Element):
    """RF multipole (xline/elements.py:159-227); pn/ps and lag in degrees."""

    _base = (
        ("voltage", 0), ("frequency", 0), ("lag", 0),
        ("knl", _zero_list), ("ksl", _zero_list), ("pn", _zero_list), ("ps", _zero_list),
    )

    @property
    def order(self):
        return max(len(self.knl), len(self.ksl)) - 1


class Cavity(Element):
    """RF cavity, lag in degrees (xline/elements.py:230-245)."""

    _base = (("voltage", 0), ("frequency", 0), ("lag", 0))


class SawtoothCavity(Element):
    """Linearised (sawtooth) cavity (xline/elements.py:248-263)."""

    _base = (("voltage", 0), ("frequency", 0), ("lag", 0))


class XYShift(Element):
    """Shift of the reference frame (xline/elements.py:266-276)."""

    _base = (("dx", 0), ("dy", 0))


class SRotation(Element):
    """Rotation about s, angle in degrees (xline/elements.py:374-390)."""

    _base = (("angle", 0),)


class LimitRect(Element):
    """Rectangular aperture, inclusive bounds (xline/elements.py:393-420)."""

    _base = (("min_x", -1.0), ("max_x", 1.0), ("min_y", -1.0), ("max_y", 1.0))


class LimitEllipse(Element):
    """Elliptical aperture (xline/elements.py:423-442)."""

    _base = (("a", 1.0), ("b", 1.0))


class LimitPolygon(Element):
    """Polygonal aperture (xline/elements.py:476-483), the closed polygon through the vertices
    ``(x_vertices[k], y_vertices[k])``.  The reference's ``track`` raises ``NotImplementedError``,
    and by default so does packing a line that contains one.  With ``Line.polygon_apertures = True``
    the line tracks it by this project's definition (include/xline_b200.h, DESIGN.md): even-odd
    rule, half-open on axis-aligned boundaries (left and bottom edges inside, right and top edges
    outside), NaN and inf coordinates lost.  ``LimitPolygon.track(p)`` on its own still raises.
    The MAD-X ``octagon`` aperture (xline/loader_mad.py:229-242) maps to this class."""

    _base = (("x_vertices", tuple), ("y_vertices", tuple))


class Exciter(Element):
    """Thin multipole whose strength follows a sampled waveform: an AC dipole, power-converter ripple
    or a transverse excitation (damper noise, chirps).  The field names follow xtrack's ``Exciter``;
    the map is this project's own (include/xline_b200.h, DESIGN.md §4.11).  A particle at turn ``T``
    (its ``at_turn``) with longitudinal position ``zeta`` reads sample
    ``floor((T - start_turn) * sampling_frequency / frev - zeta * sampling_frequency / (c beta0) + 1/2)``
    -- with ``sampling_frequency == frev`` the sample of its own turn -- and receives the kick of
    ``Multipole(knl, ksl)`` times that sample; before the first sample and after the last it receives
    none.  ``samples`` is copied into the lattice when the line is packed, and edits re-pack the line
    like every other field.  Not a ``Multipole``: no fuser or merger treats it as one."""

    _base = (("knl", _zero_list), ("ksl", _zero_list), ("samples", tuple), ("sampling_frequency", 0),
             ("frev", 0), ("start_turn", 0))

    @property
    def order(self):
        return max(len(self.knl), len(self.ksl)) - 1


class Elens(Element):
    """Hollow electron lens (xline/elements.py:281-370): parameters only.  Its map is outside the
    hot path this package serves (SURVEY.md section 8a: debug prints in the reference's ``track``);
    packing a line that contains one raises ``ValueError``.  The class exists so that
    ``Line.from_dict`` reads the reference's JSON files."""

    _base = (("voltage", 0), ("current", 0), ("inner_radius", 0), ("outer_radius", 0),
             ("ebeam_center_x", 0), ("ebeam_center_y", 0), ("elens_length", 0))


class LimitRectEllipse(Element):
    """Intersection of rectangle and ellipse (xline/elements.py:445-474)."""

    _base = (("max_x", 1.0), ("max_y", 1.0), ("a", 1.0), ("b", 1.0))


class BeamMonitor(Element):
    """Turn-by-turn recorder (xline/elements.py:485-527).  ``data`` is filled by
    ``Line.track`` with a dict of ``[num_stores, n_ids]`` tensors (x, px, y, py, zeta,
    delta, at_turn); slots never written hold NaN.  A store happens on turns with
    ``turn >= start and (turn - start) % skip == 0`` into slot ``(turn - start) // skip``
    (modulo ``num_stores`` when ``is_rolling``)."""

    _base = (
        ("num_stores", 0), ("start", 0), ("skip", 1), ("max_particle_id", 0),
        ("min_particle_id", 0), ("is_rolling", False), ("is_turn_ordered", True),
        ("data", list),
    )


class DipoleEdge(Element):
    """Dipole edge focusing (xline/elements.py:530-548)."""

    _base = (("h", 0), ("e1", 0), ("hgap", 0), ("fint", 0))


class BeamBeam4D(Element):
    """Weak-strong 4D beam-beam lens (xline/be_beamfields/beambeam.py:11-82)."""

    _base = (
        ("charge", 0), ("sigma_x", 1.0), ("sigma_y", 1.0), ("beta_r", 1.0),
        ("x_bb", 0), ("y_bb", 0), ("d_px", 0), ("d_py", 0),
    )
    _extra = (("min_sigma_diff", 1e-28), ("enabled", True))


class BeamBeam6D(Element):
    """Hirata synchro-beam 6D lens (xline/be_beamfields/beambeam.py:85-283)."""

    _base = (
        ("phi", 0), ("alpha", 0), ("x_bb_co", 0), ("y_bb_co", 0),
        ("charge_slices", 0.0), ("zeta_slices", 0.0),
        ("sigma_11", 1.0), ("sigma_12", 0), ("sigma_13", 0), ("sigma_14", 0),
        ("sigma_22", 0), ("sigma_23", 0), ("sigma_24", 0), ("sigma_33", 1.0),
        ("sigma_34", 0), ("sigma_44", 0),
        ("x_co", 0), ("px_co", 0), ("y_co", 0), ("py_co", 0), ("zeta_co", 0), ("delta_co", 0),
        ("d_x", 0), ("d_px", 0), ("d_y", 0), ("d_py", 0), ("d_zeta", 0), ("d_delta", 0),
    )
    _extra = (("min_sigma_diff", 1e-28), ("threshold_singular", 1e-28), ("enabled", True))


class SCCoasting(Element):
    """Space charge, coasting beam (xline/be_beamfields/spacecharge.py:9-52)."""

    _base = (
        ("number_of_particles", 0.0), ("circumference", 1.0), ("sigma_x", 1.0),
        ("sigma_y", 1.0), ("length", 0.0), ("x_co", 0.0), ("y_co", 0.0),
    )
    _extra = (("min_sigma_diff", 1e-8), ("enabled", True))


class SCQGaussProfile(Element):
    """Space charge, q-Gaussian bunch (xline/be_beamfields/spacecharge.py:55-104)."""

    _base = (
        ("number_of_particles", 0.0), ("bunchlength_rms", 1.0), ("sigma_x", 1.0),
        ("sigma_y", 1.0), ("length", 0.0), ("x_co", 0.0), ("y_co", 0.0),
    )
    _extra = (("min_sigma_diff", 1e-8), ("enabled", True), ("q_parameter", 1.0))


def _unit_profile():
    return [1.0, 1.0]


class SCInterpolatedProfile(Element):
    """Space charge, tabulated line density (xline/be_beamfields/spacecharge.py:107-177)."""

    _base = (
        ("number_of_particles", 0.0), ("line_density_profile", _unit_profile), ("dz", 1.0),
        ("z0", -0.5), ("sigma_x", 1.0), ("sigma_y", 1.0), ("length", 0.0),
        ("x_co", 0.0), ("y_co", 0.0),
    )
    _extra = (("method", 0), ("min_sigma_diff", 1e-8), ("enabled", True))


def element_classes():
    """name -> class, the namespace loaders take as ``classes=`` (xline/line.py:280,298)."""
    return {n: globals()[n] for n in __all__ if n not in ("Element", "element_classes")}
