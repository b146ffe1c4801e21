"""MAD-X import without cpymad / MAD-X (SURVEY.md §8f-2).

The reference's ``Line.from_madx_sequence`` (``xline/line.py:297-324`` ->
``xline/loader_mad.py:6-249``) iterates a *cpymad* sequence that MAD-X has already expanded,
made thin and decorated with error tables.  Neither cpymad nor MAD-X exists here, so this
module interprets the subset of the MAD-X language that the shipped lattice files and the
reference's own tests use (``examples/petra4/h7ba_n8.seq``, ``tests/psb/*``,
``tests/test_madx_import.py``):

* :class:`MadxFile` -- statement parser + expression evaluator + command interpreter:
  ``=`` (immediate) and ``:=`` (deferred) variables, element definitions with class
  inheritance, attribute updates (``name, k1 := kqf;`` / ``name->k1 = ...``), ``call, file``,
  ``beam``, nested ``sequence`` blocks with ``refer`` / ``from`` / in-place definitions
  (flattened on use), ``select, flag=makethin`` + ``makethin``, ``select, flag=error`` +
  ``ealign`` / ``efcomp`` (absolute ``dkn`` / ``dks``).  ``match`` blocks, ``twiss``, ``ptc_*``,
  macros and ``if`` / ``while`` are skipped and listed in ``MadxFile.skipped``;
  ``mad.sequence[name]`` quacks like a cpymad sequence (``elements``,
  ``element_positions()``, ``length``, ``expanded_elements``, ``expanded_element_names()``,
  per-element ``align_errors`` / ``field_errors``), ``$start`` / ``$end`` markers included;
* :func:`makethin` -- TEAPOT thin slicing of quadrupoles / bends (``n`` slices: end drifts
  ``L/(2(n+1))``, inner drifts ``L n/(n^2-1)``), centre kicks for sextupoles and octupoles,
  ``dipedge`` elements at bend faces, a centre marker carrying the original name when
  ``n > 1``, apertures copied to the slices -- the element types MAD-X ``makethin`` hands to
  the reference's loader;
* :func:`iter_from_madx_sequence` -- the element mapping of ``xline/loader_mad.py:23-249``
  restated for this package's classes.  The objects produced here quack like cpymad
  elements, so the reference's own loader can be run on them: that is how the mapping is
  pinned (``tests/test_madx_import.py``).

Host-side setup, not on the hot path.  Unpinned: agreement with MAD-X's own ``makethin``
output (no MAD-X binary to compare with); ``rbend`` lengths are taken as arc lengths.
"""
import math
import os
import re
from types import SimpleNamespace

import numpy as np


class _BaseType:
    def __init__(self, name):
        self.name = name


_ALIGN_KEYS = ("dx", "dy", "ds", "dphi", "dtheta", "dpsi", "mrex", "mrey", "mscalx", "mscaly", "arex", "arey")
_TYPE_DEFAULTS = {
    "multipole": dict(lrad=0.0, knl=[0.0], ksl=[0.0]),
    "hkicker": dict(kick=0.0), "vkicker": dict(kick=0.0),
    "kicker": dict(hkick=0.0, vkick=0.0), "tkicker": dict(hkick=0.0, vkick=0.0),
    "rfcavity": dict(volt=0.0, freq=0.0, lag=0.0),
    "dipedge": dict(h=0.0, e1=0.0, hgap=0.0, fint=0.0),
    "rfmultipole": dict(volt=0.0, freq=0.0, lag=0.0, knl=[0.0], ksl=[0.0], pnl=[0.0], psl=[0.0]),
    "crabcavity": dict(volt=0.0, freq=0.0, lag=0.0, tilt=0.0),
    "beambeam": dict(slot_id=0),
}


class MadElement:
    """A (thick or thin) element instance; attribute access like a cpymad element."""

    align_errors = None
    field_errors = None

    def __init__(self, name, base_type, attrs, position=0.0):
        self.name = name
        self.base_type = _BaseType(base_type)
        self.position = position  # entry position [m]
        for k, v in _TYPE_DEFAULTS.get(base_type, {}).items():
            setattr(self, k, list(v) if isinstance(v, list) else v)
        for k, v in attrs.items():
            setattr(self, k, v)
        if not hasattr(self, "l"):
            self.l = 0.0

    def attributes(self):
        return {k: v for k, v in vars(self).items()
                if k not in ("name", "base_type", "position", "align_errors", "field_errors")}

    def __repr__(self):
        return "MadElement(%s: %s @ %.6f)" % (self.name, self.base_type.name, self.position)


class MadSequence:
    def __init__(self, name, length, elements, beam=None):
        self.name = name
        self.length = length
        self.elements = elements
        # the BEAM attached to the sequence (cpymad: ``sequence.beam``); the crab-cavity mapping
        # reads ``beam.pc`` [GeV] (xline/loader_mad.py:108-125)
        self.beam = beam

    def element_positions(self):
        return [e.position for e in self.elements]

    # cpymad names for the expanded (used) sequence, consumed by Line._apply_madx_errors
    @property
    def expanded_elements(self):
        return self.elements

    def expanded_element_names(self):
        return [e.name for e in self.elements]

    def element_names(self):
        return [e.name for e in self.elements]


_FUNCS = {k: getattr(math, k) for k in
          ("sin", "cos", "tan", "asin", "acos", "atan", "sqrt", "exp", "log", "sinh", "cosh", "tanh", "floor",
           "ceil")}
_FUNCS.update({"abs": abs, "pi": math.pi, "twopi": 2 * math.pi, "clight": 299792458.0, "e": math.e,
               "true": 1.0, "false": 0.0, "degrad": 180.0 / math.pi, "raddeg": math.pi / 180.0,
               "pmass": 0.93827208816, "emass": 0.51099895e-3, "qelect": 1.602176634e-19})
_BASE_TYPES = {
    "quadrupole", "sbend", "rbend", "sextupole", "octupole", "marker", "monitor", "hmonitor",
    "vmonitor", "instrument", "drift", "hkicker", "vkicker", "kicker", "tkicker", "rfcavity",
    "multipole", "dipedge", "collimator", "rcollimator", "ecollimator", "elseparator", "solenoid",
    "placeholder", "sequence", "rfmultipole", "crabcavity", "beambeam",
}
_STRING_ATTRS = {"apertype", "particle", "file", "flag", "style", "sequence", "pattern", "class", "range",
                 "refer", "refpos", "from", "format", "table", "column", "period", "type", "name"}
_COMMANDS = {"beam", "use", "call", "select", "makethin", "ealign", "efcomp", "seqedit", "flatten", "endedit",
             "set", "option", "return", "stop", "exit", "quit", "title", "twiss", "survey", "save", "value",
             "show", "print", "system", "assign", "create", "fill", "write", "readtable", "savebeta",
             "eoption", "esave", "cycle", "install", "remove", "move", "reflect", "setvars", "plot",
             "setplot", "resbeam", "ptc_create_universe", "ptc_create_layout", "ptc_end", "ptc_twiss",
             "emit", "sixtrack", "aperture", "exec", "help", "delete", "dumpsequ", "extract", "coguess"}
_SKIPPED_BLOCKS = {"match": "endmatch", "track": "endtrack"}


class _SequenceAccessor:
    """``mad.sequence(name)`` -> the thick sequence as written (kept for scripts that slice
    explicitly with :func:`makethin`); ``mad.sequence[name]`` / ``mad.sequence.name`` -> the
    cpymad view: thin if ``makethin`` ran on it, ``$start`` / ``$end`` markers, error tables."""

    def __init__(self, mad):
        self._mad = mad

    def __call__(self, name, markers=False):
        return self._mad._thick_sequence(name.lower(), markers)

    def __getitem__(self, name):
        return self._mad._used_sequence(name.lower())

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)
        return self[name]

    def __contains__(self, name):
        return name.lower() in self._mad.sequences

    def keys(self):
        return list(self._mad.sequences)


class MadxFile:
    """Interpreter for the MAD-X subset described in the module docstring.

    ``MadxFile(path)`` executes a file (``call`` statements are followed relative to the
    directory of the calling file, like ``mad.call(path, chdir=True)`` in
    ``tests/test_madx_import.py:46``); ``MadxFile(text=...)`` / ``.input(text)`` execute a string
    (cpymad ``madx.input``).  ``defaults`` pre-sets variables that the files leave undefined
    (MAD-X takes undefined variables as 0)."""

    def __init__(self, path=None, text=None, defaults=None):
        self.vars = {}        # name -> float (immediate) or expression string (deferred)
        self.elements = {}    # name -> (parent, {attr: float | list | str | ("expr", text)})
        self.sequences = {}   # name -> dict(l=, refer=, refpos=, items=[(name, at, from)])
        self.beam = {}
        self.skipped = []     # commands / blocks that were ignored
        self.sequence = _SequenceAccessor(self)
        self._cache = {}
        self._cur_seq = None
        self._skip_until = None
        self._returned = False
        self._thin = {}       # sequence name -> makethin request (selections, options); re-run on access,
        self._thin_cache = {}  # so that deferred strengths set after MAKETHIN still reach the slices
        self._thin_sel = []   # select, flag=makethin entries
        self._err_sel = []    # select, flag=error entries
        self._errors = {}     # sequence name -> {element name: {"align": {...}, "dkn": [...], "dks": [...]}}
        self._used = None
        self._dirs = []
        for k, v in (defaults or {}).items():
            self.vars[k.lower()] = float(v)
        if path is not None:
            self.call(path)
        if text is not None:
            self.input(text)

    # ---- parsing -----------------------------------------------------------------------
    @staticmethod
    def _statements(text):
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
        lines = []
        for ln in text.splitlines():
            ln = ln.split("!")[0].split("//")[0]
            lines.append(ln)
        for st in " ".join(lines).split(";"):
            st = st.strip()
            if st:
                yield st

    def call(self, path):
        path = os.path.join(self._dirs[-1], path) if self._dirs and not os.path.isabs(path) else path
        with open(path) as fh:
            text = fh.read()
        self._dirs.append(os.path.dirname(os.path.abspath(path)))
        try:
            self.input(text)
        finally:
            self._dirs.pop()
            self._returned = False

    def input(self, text):
        for raw in self._statements(text):
            if self._returned:
                break
            self._execute(raw)
        return self

    _parse = input  # former name

    def _execute(self, raw):
        st = raw.lower()
        if self._skip_until is not None:
            if st.split(",")[0].strip() == self._skip_until:
                self._skip_until = None
            return
        head = re.split(r"[,\s]", st, 1)[0]
        if st == "endsequence":
            self._cur_seq = None
            return
        if head in _SKIPPED_BLOCKS:
            self.skipped.append(head)
            self._skip_until = _SKIPPED_BLOCKS[head]
            return
        if "{" in st and re.match(r"^(if|while|elseif|else)\b|^[\w.]+\s*(\(.*?\))?\s*:\s*macro\b", st):
            self.skipped.append(head)
            return
        m = re.match(r"^([\w.$]+)\s*:\s*([\w.]+)\s*(?:,(.*))?$", st)
        if m:
            name, parent, rest = m.group(1), m.group(2), m.group(3) or ""
            attrs = self._attrs(rest, raw)
            if parent == "sequence":
                self._cur_seq = name
                self.sequences[name] = dict(l=attrs.get("l", 0.0), refer=attrs.get("refer", "centre"),
                                            refpos=attrs.get("refpos"), items=[])
                self._thin.pop(name, None)
                self._thin_cache.pop(name, None)
                return
            at, frm = attrs.pop("at", None), attrs.pop("from", None)
            self.elements[name] = (parent, attrs)
            self._invalidate()
            if self._cur_seq is not None and at is not None:
                self.sequences[self._cur_seq]["items"].append((name, at, frm))
            return
        if self._cur_seq is not None:
            m = re.match(r"^([\w.$]+)\s*,(.*)$", st)
            if m:
                attrs = self._attrs(m.group(2), raw)
                if "at" in attrs:
                    self.sequences[self._cur_seq]["items"].append((m.group(1), attrs["at"], attrs.get("from")))
                    return
        if head in _COMMANDS:
            self._command(head, self._attrs(st[len(head):].lstrip(" ,"), raw[len(head):].lstrip(" ,")))
            return
        m = re.match(r"^([\w.$]+)\s*->\s*(\w+)\s*(:?=)\s*(.+)$", st)
        if m and m.group(1) in self.elements:
            self._update_element(m.group(1), self._attrs("%s %s %s" % m.group(2, 3, 4)))
            return
        m = re.match(r"^([\w.$]+)\s*,(.*)$", st)
        if m and m.group(1) in self.elements:
            self._update_element(m.group(1), self._attrs(m.group(2), raw))
            return
        m = re.match(r"^(?:const\s+|real\s+|int\s+|shared\s+)*([\w.]+)\s*(:?=)\s*(.+)$", st)
        if m:
            name, op, expr = m.group(1), m.group(2), m.group(3).strip()
            self.vars[name] = expr if op == ":=" else self.value(expr)
            self._invalidate()
            return
        self.skipped.append(st)

    def _invalidate(self):
        self._cache.clear()
        self._thin_cache.clear()

    def _update_element(self, name, attrs):
        attrs.pop("at", None)
        self.elements[name][1].update(attrs)
        self._invalidate()

    def _attrs(self, rest, raw_rest=None):
        """``a = 1, b := expr, c = {..}, flag`` -> dict.  ``=`` values are evaluated now,
        ``:=`` values are kept as ("expr", text); string-valued attributes stay strings."""
        out = {}
        depth, cur, parts = 0, "", []
        for ch in rest:
            if ch in "({":
                depth += 1
            elif ch in ")}":
                depth -= 1
            if ch == "," and depth == 0:
                parts.append(cur)
                cur = ""
            else:
                cur += ch
        if cur.strip():
            parts.append(cur)
        for part in parts:
            m = re.match(r"^\s*([\w.]+)\s*(:?=)\s*(.+?)\s*$", part)
            if not m:
                flag = part.strip()
                if re.fullmatch(r"-?[\w.]+", flag):
                    out[flag.lstrip("-")] = not flag.startswith("-")
                continue
            key, op, val = m.group(1), m.group(2), m.group(3)
            if key in _STRING_ATTRS:
                if key == "file" and raw_rest is not None:  # paths keep their case
                    mm = re.search(r"file\s*:?=\s*[\"']?([^\"',;]+)", raw_rest, flags=re.I)
                    val = mm.group(1).strip() if mm else val
                out[key] = val.strip("\"' ")
            elif op == ":=":
                out[key] = ("expr", val)
            else:
                out[key] = self.value(val)
        return out

    # ---- commands ----------------------------------------------------------------------
    def _command(self, cmd, a):
        if cmd == "call":
            self.call(a["file"])
        elif cmd == "return":
            self._returned = True
        elif cmd == "beam":
            self.beam.update({k: (self.value(v[1]) if isinstance(v, tuple) else v) for k, v in a.items()})
        elif cmd == "use":
            self._used = a.get("sequence", a.get("period"))
            self._errors.pop(self._used, None)  # USE re-expands the sequence: errors are dropped
        elif cmd == "select":
            flag = a.get("flag")
            if flag not in ("makethin", "error"):
                self.skipped.append("select, flag=%s" % flag)
                return
            sel = self._thin_sel if flag == "makethin" else self._err_sel
            if a.get("clear"):
                del sel[:]
                return
            entry = dict(pattern=a.get("pattern"), cls=a.get("class"), full=bool(a.get("full")),
                         slice=int(a.get("slice", 1)), thick=bool(a.get("thick", False)))
            if entry["full"] and flag == "error":
                del sel[:]
            sel.append(entry)
        elif cmd == "makethin":
            name = a["sequence"]
            style = a.get("style", "teapot")
            if style not in ("teapot", "simple"):
                raise NotImplementedError("makethin style %s" % style)
            if name not in self.sequences:
                raise ValueError("makethin: unknown sequence %s" % name)
            self._thin[name] = dict(sels=list(self._thin_sel), makedipedge=bool(a.get("makedipedge", True)),
                                    style=style)
            self._thin_cache.pop(name, None)
            self._errors.pop(name, None)
        elif cmd in ("ealign", "efcomp"):
            if self._used is None:
                raise ValueError("%s before USE" % cmd)
            if cmd == "efcomp" and any(k in a for k in ("dknr", "dksr", "radius", "order")):
                raise NotImplementedError("efcomp: only absolute dkn / dks errors are supported")
            table = self._errors.setdefault(self._used, {})
            vals = {k: (self.value(v[1]) if isinstance(v, tuple) else v) for k, v in a.items()}
            for el in self._plain_used(self._used).elements:
                if not any(_matches(self, el, s) for s in self._err_sel):
                    continue
                rec = table.setdefault(el.name, {})
                if cmd == "ealign":
                    rec["align"] = {k: float(vals.get(k, 0.0)) for k in _ALIGN_KEYS}
                else:
                    for k in ("dkn", "dks"):
                        if k in vals:
                            v = vals[k]
                            rec[k] = [float(t) for t in (v if isinstance(v, list) else [v])]
        elif cmd in ("seqedit", "flatten", "endedit", "set", "option", "title", "stop", "exit", "quit"):
            pass  # sequences are always flattened on use; nothing to do
        else:
            self.skipped.append(cmd)

    # ---- evaluation --------------------------------------------------------------------
    def value(self, expr, _stack=()):
        """Evaluate an expression (deferred variables resolved recursively; undefined
        variables are 0, as in MAD-X)."""
        if isinstance(expr, (int, float)):
            return float(expr)
        if isinstance(expr, list):
            return [self.value(t, _stack) for t in expr]
        if isinstance(expr, tuple):
            return self.value(expr[1], _stack)
        expr = expr.strip()
        try:
            return float(expr)
        except ValueError:
            pass
        if expr in self._cache:
            return self._cache[expr]
        if expr.startswith("{") and expr.endswith("}"):
            res = [self.value(t, _stack) for t in _split_top(expr[1:-1]) if t.strip()]
            self._cache[expr] = res
            return res
        env = dict(_FUNCS)
        pyexpr = expr.replace("^", "**")

        def arrow(m):  # beam->pc, element->attr
            owner, attr = m.group(1), m.group(2)
            if owner == "beam":
                val = self.beam.get(attr, 0.0)
            elif owner in self.elements:
                val = self.element_attrs(owner)[1].get(attr, 0.0)
            else:
                val = 0.0
            return repr(float(val))

        pyexpr = re.sub(r"([a-z_][\w.$]*)\s*->\s*(\w+)", arrow, pyexpr)
        for nm in set(re.findall(r"[a-z_][\w.]*", pyexpr)):
            if nm in _FUNCS:
                continue
            if nm in _stack:
                raise ValueError("circular definition of %s" % nm)
            if re.fullmatch(r"e[+-]?\d*", nm):
                continue
            val = self.value(self.vars[nm], _stack + (nm,)) if nm in self.vars else 0.0
            safe = re.sub(r"\W", "_", nm)
            if safe != nm:
                pyexpr = re.sub(r"(?<![\w.])" + re.escape(nm) + r"(?![\w.])", safe, pyexpr)
            env[safe] = val
        res = float(eval(pyexpr, {"__builtins__": {}}, env))  # noqa: S307 (lattice file arithmetic)
        self._cache[expr] = res
        return res

    def element_attrs(self, name):
        """(base type, merged attribute values) following the class inheritance chain."""
        chain = []
        cur = name
        while cur in self.elements:
            parent, attrs = self.elements[cur]
            chain.append(attrs)
            if parent == cur:  # ``quadrupole: quadrupole, ...`` style redefinition of a base type
                break
            cur = parent
        if cur not in _BASE_TYPES:
            raise ValueError('MAD element "%s" not recognized' % cur)
        merged = {}
        for attrs in reversed(chain):
            merged.update(attrs)
        return cur, {k: (v if isinstance(v, (str, bool)) else self.value(v)) for k, v in merged.items()}

    # ---- sequences ---------------------------------------------------------------------
    def _seq_length(self, name):
        return self.value(self.sequences[name]["l"])

    def _flatten(self, name, offset, out, depth=0):
        if depth > 16:
            raise ValueError("sequence nesting too deep (recursive definition?)")
        sq = self.sequences[name]
        refer = sq["refer"]
        centres = {}
        for ename, at, frm in sq["items"]:
            pos = self.value(at)
            if frm is not None:
                if frm not in centres:
                    raise ValueError("from=%s: not placed before %s in sequence %s" % (frm, ename, name))
                pos += centres[frm]
            centres[ename] = pos
            if ename in self.sequences and ename not in self.elements:
                length = self._seq_length(ename)
                sub = self.sequences[ename]
                if sub.get("refpos"):
                    inner = {n: self.value(a) for n, a, _ in sub["items"]}
                    start = pos - inner[sub["refpos"]]
                else:
                    start = pos - {"entry": 0.0, "centre": 0.5 * length, "exit": length}[refer]
                self._flatten(ename, offset + start, out, depth + 1)
                continue
            base, attrs = self.element_attrs(ename)
            length = float(attrs.get("l", 0.0))
            entry = pos - {"entry": 0.0, "centre": 0.5 * length, "exit": length}[refer]
            out.append(MadElement(ename, base, attrs, offset + entry))

    def _beam_namespace(self):
        """``beam`` command attributes as cpymad exposes them; ``pc`` [GeV] is derived from ``energy``
        and the particle mass when only the energy was given."""
        b = dict(self.beam)
        mass = b.get("mass", {"proton": 0.93827208816, "electron": 0.51099895e-3,
                              "positron": 0.51099895e-3}.get(str(b.get("particle", "proton")).lower()))
        if "pc" not in b and "energy" in b and mass is not None:
            b["pc"] = math.sqrt(max(float(b["energy"]) ** 2 - mass ** 2, 0.0))
        if "energy" not in b and "pc" in b and mass is not None:
            b["energy"] = math.hypot(float(b["pc"]), mass)
        return SimpleNamespace(**b)

    def _thick_sequence(self, name, markers=False):
        """The flattened thick sequence: elements at their ENTRY positions."""
        out = []
        self._flatten(name, 0.0, out)
        length = self._seq_length(name)
        if markers:
            out = ([MadElement(name + "$start", "marker", {}, 0.0)] + out
                   + [MadElement(name + "$end", "marker", {}, length)])
        return MadSequence(name, length, out, self._beam_namespace())

    def _plain_used(self, name):
        if name not in self._thin:
            return self._thick_sequence(name)
        if name not in self._thin_cache:
            req = self._thin[name]
            self._thin_cache[name] = makethin(
                self._thick_sequence(name), slice_fn=(lambda el: _selected_slices(self, el, req["sels"])),
                centre_markers=True, makedipedge=req["makedipedge"], style=req["style"])
        return self._thin_cache[name]

    def _used_sequence(self, name):
        base = self._plain_used(name)
        els = ([MadElement(name + "$start", "marker", {}, 0.0)] + list(base.elements)
               + [MadElement(name + "$end", "marker", {}, base.length)])
        table = self._errors.get(name, {})
        for el in els:
            rec = table.get(el.name)
            if rec is None:
                continue
            if "align" in rec:
                el.align_errors = SimpleNamespace(**rec["align"])
            if "dkn" in rec or "dks" in rec:
                dkn = np.zeros(21)
                dks = np.zeros(21)
                dkn[:len(rec.get("dkn", []))] = rec.get("dkn", [])
                dks[:len(rec.get("dks", []))] = rec.get("dks", [])
                el.field_errors = SimpleNamespace(dkn=dkn, dks=dks)
        return MadSequence(name, base.length, els, base.beam)


def _split_top(text):
    depth, cur, parts = 0, "", []
    for ch in text:
        if ch in "({":
            depth += 1
        elif ch in ")}":
            depth -= 1
        if ch == "," and depth == 0:
            parts.append(cur)
            cur = ""
        else:
            cur += ch
    parts.append(cur)
    return parts


def _matches(mad, el, sel):
    """MAD-X SELECT semantics for the keys used here: ``full``, ``class`` (base type or any
    user class in the inheritance chain), ``pattern`` (regular expression, searched)."""
    if sel["full"]:
        return True
    ok = sel["pattern"] is not None or sel["cls"] is not None
    if sel["pattern"] is not None:
        ok = ok and re.search(sel["pattern"], el.name) is not None
    if sel["cls"] is not None:
        chain, cur = [el.base_type.name], re.sub(r"\.\.\d+$|_de[nx]$", "", el.name)
        while cur in mad.elements:
            chain.append(cur)
            cur = mad.elements[cur][0]
        ok = ok and sel["cls"] in chain
    return ok


def _selected_slices(mad, el, sels):
    n = 1
    for s in sels:
        if s["full"] or (s["pattern"] is None and s["cls"] is None) or _matches(mad, el, s):
            n = s["slice"]
    return n


def _teapot(length, n):
    """Kick positions (from the entry) of an n-slice TEAPOT thin-lens model."""
    if n == 1:
        return [0.5 * length]
    end = length / (2.0 * (1 + n))
    inner = length * n / (n * n - 1.0)
    return [end + i * inner for i in range(n)]


def makethin(seq, slices=None, default_slices=1, slice_fn=None, centre_markers=False, makedipedge=True,
             style="teapot"):
    """Thin version of a thick :class:`MadSequence` (what MAD-X ``makethin`` would hand to the
    loader): ``slices`` maps a base type to its number of TEAPOT slices
    (``examples/petra4/track_p1.py:26-30`` uses 4 for ``sbend`` and ``quadrupole``), or
    ``slice_fn(element)`` gives it per element (``select, flag=makethin`` entries).  With
    ``centre_markers`` an element cut into more than one slice leaves a marker carrying its
    name (and aperture) at its centre, as MAD-X does (``tests/test_madx_import.py:113-135``
    counts it)."""
    slices = dict(slices or {})
    out = []

    def kicks(length, n):
        if style == "simple" and n > 1:
            return [(i + 0.5) * length / n for i in range(n)]
        return _teapot(length, n)

    def aperture_of(el):
        return {k: getattr(el, k) for k in ("apertype", "aperture") if hasattr(el, k)}

    def sliced(el, n, make_attrs):
        L = float(el.l)
        pos = kicks(L, n)
        half = n // 2
        for i, s in enumerate(pos):
            if centre_markers and n > 1 and i == half and n % 2 == 0:
                out.append(MadElement(el.name, "marker", dict(l=0.0, **aperture_of(el)), el.position + 0.5 * L))
            attrs = make_attrs()
            attrs.update(aperture_of(el))
            out.append(MadElement("%s..%d" % (el.name, i + 1) if n > 1 else el.name, "multipole", attrs,
                                  el.position + s))
            if centre_markers and n > 1 and i == half and n % 2 == 1:
                # odd slice count: the middle kick sits at the centre; the marker follows it
                out.append(MadElement(el.name, "marker", dict(l=0.0, **aperture_of(el)), el.position + 0.5 * L))

    for el in seq.elements:
        base, L = el.base_type.name, float(el.l)
        n = int(slice_fn(el)) if slice_fn is not None else int(slices.get(base, default_slices))
        tilt = float(getattr(el, "tilt", 0.0))
        if base in ("quadrupole", "sextupole", "octupole") and L > 0:
            order = {"quadrupole": 1, "sextupole": 2, "octupole": 3}[base]
            strength = float(getattr(el, "k%d" % order, 0.0))
            skew = float(getattr(el, "k%ds" % order, 0.0))
            sliced(el, n, lambda: dict(knl=[0.0] * order + [strength * L / n], ksl=[0.0] * order + [skew * L / n],
                                       lrad=L / n, l=0.0, tilt=tilt))
        elif base in ("sbend", "rbend") and L > 0:
            angle = float(getattr(el, "angle", 0.0))
            k1 = float(getattr(el, "k1", 0.0))
            h = angle / L
            e1, e2 = float(getattr(el, "e1", 0.0)), float(getattr(el, "e2", 0.0))
            if base == "rbend":
                e1, e2 = e1 + angle / 2, e2 + angle / 2
            hgap, fint = float(getattr(el, "hgap", 0.0)), float(getattr(el, "fint", 0.0))
            if makedipedge:
                out.append(MadElement(el.name + "_den", "dipedge", dict(h=h, e1=e1, hgap=hgap, fint=fint, l=0.0),
                                      el.position))
            sliced(el, n, lambda: dict(knl=[angle / n, k1 * L / n], ksl=[0.0, 0.0], lrad=L / n, l=0.0, tilt=tilt))
            if makedipedge:
                out.append(MadElement(el.name + "_dex", "dipedge", dict(h=h, e1=e2, hgap=hgap, fint=fint, l=0.0),
                                      el.position + L))
        elif base in ("hkicker", "vkicker", "kicker", "tkicker"):
            attrs = dict(lrad=L, l=0.0, tilt=tilt, **aperture_of(el))
            for k in ("kick", "hkick", "vkick"):
                if hasattr(el, k):
                    attrs[k] = float(getattr(el, k))
            out.append(MadElement(el.name, base, attrs, el.position + 0.5 * L))
        elif base == "rfcavity":
            attrs = dict(volt=float(getattr(el, "volt", 0.0)), freq=float(getattr(el, "freq", 0.0)),
                         lag=float(getattr(el, "lag", 0.0)), l=0.0, **aperture_of(el))
            if hasattr(el, "harmon"):
                attrs["harmon"] = float(el.harmon)
            out.append(MadElement(el.name, base, attrs, el.position + 0.5 * L))
        else:
            out.append(MadElement(el.name, base, el.attributes(), el.position))
    out.sort(key=lambda e: e.position)
    return MadSequence(seq.name, seq.length, out, getattr(seq, "beam", None))


_DRIFT_LIKE = ("marker", "monitor", "hmonitor", "vmonitor", "collimator", "rcollimator", "elseparator",
               "instrument", "solenoid", "drift")


def iter_from_madx_sequence(sequence, classes, ignored_madtypes=(), exact_drift=False,
                            drift_threshold=1e-6, install_apertures=False):
    """``(name, element)`` pairs for a thin sequence -- restates the mapping of
    ``xline/loader_mad.py:6-249`` (implicit drifts :29-32, element table :40-183, tilt
    wrappers :186-197, apertures :199-246, closing drift :248-249) for the element types this
    package supports."""
    if not isinstance(classes, dict):
        classes = {k: getattr(classes, k) for k in dir(classes) if not k.startswith("_")}
    Drift = classes["DriftExact"] if exact_drift else classes["Drift"]
    Multipole = classes["Multipole"]
    old_pp, i_drift = 0.0, 0
    pairs = sorted(zip(sequence.element_positions(), sequence.elements), key=lambda t: t[0])
    for pp, ee in pairs:
        if pp > old_pp + drift_threshold:
            yield "drift_%d" % i_drift, Drift(length=(pp - old_pp))
            old_pp = pp
            i_drift += 1
        kind = ee.base_type.name
        new = None
        skiptilt = False
        if kind in _DRIFT_LIKE:
            new = Drift(length=ee.l)
            old_pp += ee.l
        elif kind in ignored_madtypes:
            # the reference falls through with whatever `newele` held before (loader_mad.py:55-56:
            # the previous element again, or a NameError for the first one); an ignored type is
            # skipped here
            continue
        elif kind == "multipole":
            knl = list(getattr(ee, "knl", [0]))
            ksl = list(getattr(ee, "ksl", [0]))
            new = Multipole(knl=knl, ksl=ksl, hxl=knl[0], hyl=ksl[0], length=ee.lrad)
        elif kind in ("tkicker", "kicker"):
            new = Multipole(knl=[-ee.hkick] if hasattr(ee, "hkick") else [],
                            ksl=[ee.vkick] if hasattr(ee, "vkick") else [], length=ee.lrad, hxl=0, hyl=0)
        elif kind == "vkicker":
            new = Multipole(knl=[], ksl=[ee.kick], length=ee.lrad, hxl=0, hyl=0)
        elif kind == "hkicker":
            new = Multipole(knl=[-ee.kick], ksl=[], length=ee.lrad, hxl=0, hyl=0)
        elif kind == "dipedge":
            new = classes["DipoleEdge"](h=ee.h, e1=ee.e1, hgap=ee.hgap, fint=ee.fint)
        elif kind == "rfcavity":
            new = classes["Cavity"](voltage=ee.volt * 1e6, frequency=ee.freq * 1e6, lag=ee.lag * 360)
        elif kind == "rfmultipole":  # loader_mad.py:97-106
            new = classes["RFMultipole"](voltage=ee.volt * 1e6, frequency=ee.freq * 1e6, lag=ee.lag * 360,
                                         knl=list(ee.knl), ksl=list(ee.ksl), pn=[v * 360 for v in ee.pnl],
                                         ps=[v * 360 for v in ee.psl])
        elif kind == "crabcavity":  # loader_mad.py:108-125: ee.volt in MV, sequence.beam.pc in GeV
            pc = sequence.beam.pc
            if abs(ee.tilt - math.pi / 2) < 1e-9:
                new = classes["RFMultipole"](frequency=ee.freq * 1e6, ksl=[-ee.volt / pc * 1e-3],
                                             ps=[ee.lag * 360 + 90])
                skiptilt = True
            else:
                new = classes["RFMultipole"](frequency=ee.freq * 1e6, knl=[ee.volt / pc * 1e-3],
                                             pn=[ee.lag * 360 + 90])
        elif kind == "beambeam":  # loader_mad.py:128-170: placeholders, to be configured afterwards
            if int(getattr(ee, "slot_id", 0)) in (6, 60):
                new = classes["BeamBeam6D"](
                    phi=0.0, alpha=0.0, x_bb_co=0.0, y_bb_co=0.0, charge_slices=[0.0], zeta_slices=[0.0],
                    sigma_11=1.0, sigma_12=0.0, sigma_13=0.0, sigma_14=0.0, sigma_22=1.0, sigma_23=0.0,
                    sigma_24=0.0, sigma_33=0.0, sigma_34=0.0, sigma_44=0.0, x_co=0.0, px_co=0.0, y_co=0.0,
                    py_co=0.0, zeta_co=0.0, delta_co=0.0, d_x=0.0, d_px=0.0, d_y=0.0, d_py=0.0, d_zeta=0.0,
                    d_delta=0.0)
            else:
                new = classes["BeamBeam4D"](charge=0.0, sigma_x=1.0, sigma_y=1.0, beta_r=1.0, x_bb=0.0,
                                            y_bb=0.0, d_px=0.0, d_py=0.0)
        elif kind == "placeholder":
            slot = int(getattr(ee, "slot_id", 0))
            if slot in (1, 2, 3):
                new = classes[{1: "SCCoasting", 2: "SCQGaussProfile", 3: "SCInterpolatedProfile"}[slot]]()
            else:
                new = Drift(length=ee.l)
                old_pp += ee.l
        else:
            raise ValueError('MAD element "%s" not recognized' % kind)
        tilt = math.degrees(ee.tilt) if (abs(getattr(ee, "tilt", 0.0)) > 0 and not skiptilt) else 0
        if abs(tilt) > 0:
            yield ee.name + "_pretilt", classes["SRotation"](angle=tilt)
        yield ee.name, new
        if abs(tilt) > 0:
            yield ee.name + "_posttilt", classes["SRotation"](angle=-tilt)
        if install_apertures and hasattr(ee, "aperture") and min(ee.aperture) > 0:
            ap = ee.aperture
            if ee.apertype == "rectangle":
                yield ee.name + "_aperture", classes["LimitRect"](min_x=-ap[0], max_x=ap[0], min_y=-ap[1], max_y=ap[1])
            elif ee.apertype == "ellipse":
                yield ee.name + "_aperture", classes["LimitEllipse"](a=ap[0], b=ap[1])
            elif ee.apertype == "circle":
                yield ee.name + "_aperture", classes["LimitEllipse"](a=ap[0], b=ap[0])
            elif ee.apertype == "rectellipse":
                yield ee.name + "_aperture", classes["LimitRectEllipse"](max_x=ap[0], max_y=ap[1], a=ap[2], b=ap[3])
            elif ee.apertype == "octagon":  # loader_mad.py:229-242; tracked with Line.polygon_apertures = True
                # (8 vertices, 6 stored edges: the top and bottom edges are horizontal)
                v1 = (ap[0], ap[0] * math.tan(ap[2]))
                v2 = (ap[1] / math.tan(ap[3]), ap[1])
                yield ee.name + "_aperture", classes["LimitPolygon"](
                    x_vertices=[v1[0], v2[0], -v2[0], -v1[0], -v1[0], -v2[0], v2[0], v1[0]],
                    y_vertices=[v1[1], v2[1], v2[1], v1[1], -v1[1], -v2[1], -v2[1], -v1[1]])
            else:
                raise ValueError("Aperture type not recognized")
    if sequence.length > old_pp:
        yield "drift_%d" % i_drift, Drift(length=(sequence.length - old_pp))
