"""In-tree build of ``libxline_b200.so`` (hand-written sm_100a CUDA + the C ABI).

Plain ``nvcc`` invocations, no torch involvement: the shared library exposes only the
``extern "C"`` entry points of ``include/xline_b200.h``.  Objects are cached by source
mtime under ``xline_b200/csrc/_build`` so that rebuilding after an edit recompiles only
the translation units that changed.
"""
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "_build")
LIB = os.path.join(HERE, "libxline_b200.so")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]

# (object name, source, extra flags)
UNITS = [
    ("cabi", "cabi.cu", []),
    ("moments", "moments.cu", []),                                            # beam-moment reduction
    ("naff", "naff.cu", []),                                                  # NAFF tunes of monitor data
    ("tangent", "tangent.cu", []),                                            # tangent map (Jacobians, FLI)
    ("track_fast", "track_fast.cu", []),
    ("track_fast_nc", "track_fast.cu", ["-DXLB_NOCHI=1"]),                      # chi == 1 throughout
    ("track_fast_nc_lo", "track_fast.cu", ["-DXLB_NOCHI=1", "-DXLB_MAXORDER=3"]),  # + multipole order <= 3
    ("track_strict", "track_strict.cu", ["-fmad=false"]),
    ("track_fast_bf", "track_fast.cu", ["-DXLB_BEAMFIELDS=1"]),        # + BeamBeam4D, space charge
    ("track_fast_bf_nc_lo", "track_fast.cu", ["-DXLB_BEAMFIELDS=1", "-DXLB_NOCHI=1", "-DXLB_MAXORDER=3"]),
    ("track_fast_bf6", "track_fast.cu", ["-DXLB_BEAMFIELDS=2"]),       # + BeamBeam6D
    ("track_strict_bf", "track_strict.cu", ["-DXLB_BEAMFIELDS=2", "-fmad=false"]),
]
HEADERS = ["track_impl.cuh", "kargs.h", "launch_plan.h", "variants.inc", "beamfields.cuh",
           "faddeeva_coeffs.inc", "synrad_table.inc", os.path.join("..", "..", "include", "xline_b200.h")]


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: cannot build libxline_b200.so")
    return exe


def _newest_header():
    t = 0.0
    for h in HEADERS:
        p = os.path.join(CSRC, h)
        if os.path.exists(p):
            t = max(t, os.path.getmtime(p))
    return t


def _compile(unit, verbose):
    name, src, extra = unit
    srcp = os.path.join(CSRC, src)
    obj = os.path.join(OBJ, name + ".o")
    dep_t = max(os.path.getmtime(srcp), _newest_header(), os.path.getmtime(__file__))
    if os.path.exists(obj) and os.path.getmtime(obj) >= dep_t:
        return obj, ""
    cmd = [_nvcc()] + ARCH + COMMON + extra + ["-Xptxas", "-v", "-c", srcp, "-o", obj]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, res.stdout, res.stderr))
    with open(os.path.join(OBJ, name + ".ptxas.txt"), "w") as fh:
        fh.write(res.stderr)
    return obj, res.stderr


def _units():
    return list(UNITS)


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    if force:
        for f in os.listdir(OBJ):
            os.remove(os.path.join(OBJ, f))
    units = _units()
    with ThreadPoolExecutor(max_workers=min(len(units), os.cpu_count() or 2)) as ex:
        results = list(ex.map(lambda u: _compile(u, verbose), units))
    objs = [r[0] for r in results]
    newest = max(os.path.getmtime(o) for o in objs)
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < newest:
        cmd = [_nvcc()] + ARCH + ["-shared", "-o", LIB] + objs
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (res.stdout, res.stderr))
    if verbose:
        for r in results:
            if r[1]:
                sys.stderr.write(r[1])
    return LIB


def ptxas_report():
    """Registers / spills per kernel from the last compile (for DESIGN.md and tests)."""
    out = {}
    for name, _, _ in UNITS:
        p = os.path.join(OBJ, name + ".ptxas.txt")
        if os.path.exists(p):
            out[name] = open(p).read()
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
