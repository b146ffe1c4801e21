"""ctypes binding of ``libxline_b200.so`` (the C ABI in ``include/xline_b200.h``).

There is deliberately no fallback: if the shared library is missing or does not load,
importing this module raises, and so does every ``Line.track``.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libxline_b200.so")

ABI_VERSION = 4
OPT_NO_TURN_COUNT = 1  # xlb_track_options_t::flags
MOMENT_WORDS = 56  # XLB_MOMENT_WORDS: words of one beam-moment store
MOMENT_PAIRS = 27  # XLB_MOMENT_PAIRS: (hi, lo) sums of a store
MOMENT_FIRST = 2   # XLB_MOMENT_FIRST: word of the first pair, after n and n_nonfinite
NAFF_MIN_TURNS = 64    # XLB_NAFF_MIN_TURNS: shortest signal xlb_naff_device takes
NAFF_MAX_TURNS = 8192  # XLB_NAFF_MAX_TURNS: longest
TANGENT_SCALE_LOG2 = 512     # XLB_TANGENT_SCALE_LOG2: the tangent map's overflow guard, 2^512
TANGENT_MAX_THREADS = 256    # XLB_TANGENT_MAX_THREADS

EXPORTS = (
    "xlb_abi_version", "xlb_last_error", "xlb_lattice_validate", "xlb_track_device",
    "xlb_track_device_timed", "xlb_track_host", "xlb_get_stats", "xlb_compact_alive_device",
    "xlb_measure_fp64_peak", "xlb_measure_dfma_latency", "xlb_kernel_variant_count",
    "xlb_kernel_variant_info", "xlb_selftest_exact_division", "xlb_beam_moments_device",
    "xlb_track_device_moments", "xlb_naff_device", "xlb_track_tangent_device",
    "xlb_track_tangent_radiation_device", "xlb_track_envelope_device",
)


class Lattice(C.Structure):
    _fields_ = [
        ("words", C.c_void_p), ("n_words", C.c_int64), ("chunk_words", C.c_int32),
        ("n_chunks", C.c_int32), ("n_elements", C.c_int32), ("flags", C.c_uint32),
        ("n_segments", C.c_int32), ("segments", C.c_void_p),
    ]


_DCOLS = ("x", "px", "y", "py", "zeta", "delta", "rpp", "rvv", "s", "chi", "charge_ratio")
_ICOLS = ("state", "at_element", "at_turn", "particle_id")


class Particles(C.Structure):
    _fields_ = (
        [("n", C.c_int64)]
        + [(k, C.c_void_p) for k in _DCOLS]
        + [(k, C.c_void_p) for k in _ICOLS]
        + [(k, C.c_double) for k in ("q0", "mass0", "p0c", "beta0", "gamma0", "energy0")]
    )


class TrackOptions(C.Structure):
    _fields_ = [
        ("num_turns", C.c_int32), ("particles_per_thread", C.c_int32),
        ("threads_per_block", C.c_int32), ("turns_per_launch", C.c_int32),
        ("loss_tally", C.c_void_p), ("monitor_data", C.c_void_p), ("monitor_words", C.c_int64),
        ("compact_threshold", C.c_double), ("turns_per_item", C.c_int32), ("flags", C.c_int32),
        ("trace", C.c_void_p), ("trace_particles", C.c_int64), ("element_index_offset", C.c_int64),
    ]


class MomentsSpec(C.Structure):
    _fields_ = [("num_stores", C.c_int64), ("start", C.c_int64), ("skip", C.c_int64)]


class TrackStats(C.Structure):
    _fields_ = [
        ("n_alive_in", C.c_int64), ("n_alive_out", C.c_int64), ("kernel_launches", C.c_int32),
        ("compactions", C.c_int32), ("regs_per_thread", C.c_int32), ("smem_bytes", C.c_int32),
        ("blocks", C.c_int32), ("threads", C.c_int32), ("kernel_ms", C.c_float),
    ]


_lib = None


def lib():
    """The loaded library (raises ``RuntimeError`` when it is absent -- no CPU path)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "xline_b200: %s is missing -- build it with `python -m xline_b200.build` "
            "(there is no CPU fallback for Line.track)" % LIB_PATH
        )
    L = C.CDLL(LIB_PATH)
    L.xlb_abi_version.restype = C.c_int
    L.xlb_last_error.restype = C.c_char_p
    L.xlb_lattice_validate.argtypes = [C.POINTER(Lattice)]
    for fn in (L.xlb_track_device, L.xlb_track_device_timed):
        fn.argtypes = [C.POINTER(Lattice), C.POINTER(Particles), C.POINTER(TrackOptions), C.c_void_p]
        fn.restype = C.c_int
    L.xlb_track_device_moments.argtypes = [C.POINTER(Lattice), C.POINTER(Particles), C.POINTER(TrackOptions),
                                           C.POINTER(MomentsSpec), C.c_void_p, C.c_void_p]
    L.xlb_track_device_moments.restype = C.c_int
    L.xlb_beam_moments_device.argtypes = [C.POINTER(Particles), C.c_void_p, C.c_void_p]
    L.xlb_beam_moments_device.restype = C.c_int
    L.xlb_naff_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_double,
                                  C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
    L.xlb_naff_device.restype = C.c_int
    L.xlb_track_tangent_device.argtypes = [C.POINTER(Lattice), C.POINTER(Particles), C.POINTER(TrackOptions),
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.xlb_track_tangent_device.restype = C.c_int
    L.xlb_track_tangent_radiation_device.argtypes = L.xlb_track_tangent_device.argtypes
    L.xlb_track_tangent_radiation_device.restype = C.c_int
    L.xlb_track_envelope_device.argtypes = [C.POINTER(Lattice), C.POINTER(Particles), C.POINTER(TrackOptions),
                                            C.c_void_p, C.c_void_p, C.c_void_p]
    L.xlb_track_envelope_device.restype = C.c_int
    L.xlb_track_host.argtypes = [C.POINTER(Lattice), C.POINTER(Particles), C.POINTER(TrackOptions)]
    L.xlb_track_host.restype = C.c_int
    L.xlb_get_stats.argtypes = [C.POINTER(TrackStats)]
    L.xlb_compact_alive_device.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    L.xlb_measure_fp64_peak.argtypes = [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.xlb_kernel_variant_count.restype = C.c_int
    L.xlb_kernel_variant_info.argtypes = [C.c_int, C.c_char_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    if L.xlb_abi_version() != ABI_VERSION:
        raise RuntimeError("libxline_b200.so ABI version mismatch")
    _lib = L
    return L


def check(rc):
    if rc != 0:
        msg = lib().xlb_last_error().decode("utf-8", "replace")
        if rc == -1:
            raise ValueError("xline_b200: " + msg)
        raise RuntimeError("xline_b200 (code %d): %s" % (rc, msg))


def stats():
    st = TrackStats()
    check(lib().xlb_get_stats(C.byref(st)))
    return {k: getattr(st, k) for k, _ in TrackStats._fields_}


def kernel_variants():
    L = lib()
    out = []
    for i in range(L.xlb_kernel_variant_count()):
        buf = C.create_string_buffer(64)
        regs, thr = C.c_int(0), C.c_int(0)
        check(L.xlb_kernel_variant_info(i, buf, 64, C.byref(regs), C.byref(thr)))
        out.append(dict(name=buf.value.decode(), regs=regs.value, max_threads=thr.value))
    return out


def measure_dfma_latency():
    """Cycles per DFMA of one warp running 1, 2, 4, 8 independent chains."""
    out = (C.c_double * 4)()
    L = lib()
    L.xlb_measure_dfma_latency.argtypes = [C.POINTER(C.c_double), C.c_int]
    check(L.xlb_measure_dfma_latency(out, 4))
    return dict(zip((1, 2, 4, 8), [float(v) for v in out]))


def selftest_exact_division(divisors, mode, samples_per_thread=64, seed=1, exponent_span=200):
    """(mismatches, samples) of the strict kernels' division sequences against the device's own
    IEEE division (``xlb_selftest_exact_division``)."""
    L = lib()
    L.xlb_selftest_exact_division.argtypes = [C.POINTER(C.c_double), C.c_int, C.c_int, C.c_int, C.c_uint64,
                                              C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    arr = (C.c_double * len(divisors))(*[float(v) for v in divisors])
    bad, n = C.c_uint64(0), C.c_uint64(0)
    check(L.xlb_selftest_exact_division(arr, len(divisors), int(mode), int(samples_per_thread), int(seed),
                                        int(exponent_span), C.byref(bad), C.byref(n)))
    return bad.value, n.value


def measure_fp64_peak(repeats=5):
    fl, ms = C.c_double(0), C.c_double(0)
    check(lib().xlb_measure_fp64_peak(repeats, C.byref(fl), C.byref(ms)))
    return fl.value, ms.value
