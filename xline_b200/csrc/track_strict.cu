// Strict variants: compiled with -fmad=false; evaluates every map in the reference's
// operation order (XLB_STRICT 1) so results are IEEE-identical to the NumPy path wherever
// only + - * / sqrt are involved.  Parity instrument, not the performance path.
#define XLB_STRICT 1
#define XLB_NOCHI 0
#define XLB_MAXORDER 0
#ifndef XLB_BEAMFIELDS
#define XLB_BEAMFIELDS 0
#endif
#if XLB_BEAMFIELDS
#define XLB_NS strict_bf
#else
#define XLB_NS strict_lean
#endif
#include "track_impl.cuh"
#include "variants.inc"

namespace xlb {
using namespace XLB_NS;

#if XLB_BEAMFIELDS
#define XLB_TABLE strict_bf_table
#define XLB_TABLE_FN strict_bf_variants
#define XLB_SUFFIX "/beamfields"
#else
#define XLB_TABLE strict_table
#define XLB_TABLE_FN strict_variants
#define XLB_SUFFIX "/lean"
#endif
static const Variant XLB_TABLE[] = {
    XLB_VARIANT_ENTRY("strict/ppt1" XLB_SUFFIX, 1, 256, 1),
    XLB_VARIANT_ENTRY("strict/ppt2" XLB_SUFFIX, 2, 256, 1),
#if !XLB_BEAMFIELDS
    XLB_VARIANT_ENTRY("strict/ppt2/t128" XLB_SUFFIX, 2, 128, 3),
    XLB_VARIANT_ENTRY("strict/ppt3/t128" XLB_SUFFIX, 3, 128, 3),
#endif
    XLB_TRACE_ENTRY("strict/trace"),
    XLB_POLYGON_VARIANT_ENTRY("strict/ppt1" XLB_SUFFIX "/polygons", 1, 256, 1),
    XLB_POLYGON_VARIANT_ENTRY("strict/ppt2" XLB_SUFFIX "/polygons", 2, 256, 1),
#if !XLB_BEAMFIELDS
    XLB_POLYGON_VARIANT_ENTRY("strict/ppt2/t128" XLB_SUFFIX "/polygons", 2, 128, 3),
    XLB_POLYGON_VARIANT_ENTRY("strict/ppt3/t128" XLB_SUFFIX "/polygons", 3, 128, 3),
#endif
    XLB_POLYGON_TRACE_ENTRY("strict/trace/polygons"),
};
const Variant *XLB_TABLE_FN(int *n) {
  *n = static_cast<int>(sizeof(XLB_TABLE) / sizeof(XLB_TABLE[0]));
  return XLB_TABLE;
}

#if !XLB_BEAMFIELDS
// Self-test of the division sequences of the strict kernels against the IEEE division of the
// same device: every thread draws dividends (random mantissa, exponent spread over 2^+-span,
// every 16th one constructed next to a rounding midpoint of the quotient) and counts the
// quotients that differ in any bit.  divisors[0..n_div) with mode 0 = small integers through
// div_small_int and the constant table, mode 1 = arbitrary divisors through div_known_recip.
__global__ void selftest_division_kernel(const double *divisors, int n_div, int mode, int per_thread,
                                         unsigned long long seed, int span,
                                         unsigned long long *mismatches) {
  unsigned long long s = seed + 0x9E3779B97F4A7C15ULL * (blockIdx.x * blockDim.x + threadIdx.x + 1);
  unsigned long long bad = 0;
  for (int d = 0; d < n_div; ++d) {
    const double b = divisors[d];
    const double y = mode == 0 ? c_recip.v[static_cast<int>(b)].y : 1.0 / b;
    const double bb = mode == 0 ? c_recip.v[static_cast<int>(b)].x : b;
    for (int k = 0; k < per_thread; ++k) {
      s ^= s << 13; s ^= s >> 7; s ^= s << 17;
      const unsigned long long m = s & 0x800fffffffffffffULL;
      s ^= s << 13; s ^= s >> 7; s ^= s << 17;
      const long long e = 1023 + static_cast<long long>(s % (2 * span + 1)) - span;
      double a = __longlong_as_double(static_cast<long long>(m | (static_cast<unsigned long long>(e) << 52)));
      if ((k & 15) == 0) {
        // dividend next to a midpoint: a = RN((q + ulp(q)/2) * b) for a random quotient q
        const double q = fabs(a);
        const double half_ulp = __longlong_as_double(__double_as_longlong(q) & 0x7ff0000000000000LL) * 1.1102230246251565e-16;
        a = fma(q, b, half_ulp * b);
        if (k & 16) a = -a;
      }
      const double want = a / b;
      const double got = mode == 0 ? div_small_int(a, bb, y) : div_known_recip(a, bb, y);
      if (__double_as_longlong(want) != __double_as_longlong(got)) ++bad;
    }
  }
  if (bad) atomicAdd(mismatches, bad);
}

int strict_selftest_division(const double *d_divisors, int n_div, int mode, int per_thread,
                             unsigned long long seed, int span, unsigned long long *d_mismatches,
                             void *stream) {
  selftest_division_kernel<<<148 * 4, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      d_divisors, n_div, mode, per_thread, seed, span, d_mismatches);
  return static_cast<int>(cudaGetLastError());
}
#endif
}  // namespace xlb
