// Fast variants: FMA contraction on, pack-time constant folding (XLB_STRICT 0).
//
// One translation unit per kernel FAMILY, selected by three compile-time switches:
//   XLB_BEAMFIELDS  0 = thin lenses only, 1 = + BeamBeam4D and space charge, 2 = + BeamBeam6D.
//                   The 6D lens is compiled into its own set of kernels: its register appetite
//                   makes ptxas spill in the dispatch loop of every kernel that contains it,
//                   whether or not a lattice has such a lens (ncu on the PS Booster: 6 % of all
//                   executed instructions were LDL/STL).
//   XLB_NOCHI       1 = every particle has chi == 1 (xlb_particles_t::chi == NULL, the reference's
//                   default: one species): chi is not carried in registers, its products are
//                   dropped (bit-identical: fma(-1, a, b) == b - a).  Eight registers per four
//                   particles that buy a fourth particle per thread at the same occupancy.
//   XLB_MAXORDER    3 = every multipole of the lattice has order <= 3 (XLB_F_LOW_ORDER): the
//                   Horner evaluation is straight-line, no coefficient ring, no loop.
// The host (cabi.cu, pick_variant) takes the most specialised family the call admits.
#define XLB_STRICT 0
#ifndef XLB_BEAMFIELDS
#define XLB_BEAMFIELDS 0
#endif
#ifndef XLB_NOCHI
#define XLB_NOCHI 0
#endif
#ifndef XLB_MAXORDER
#define XLB_MAXORDER 0
#endif
// Synchrotron radiation (MULTIPOLE_RAD, track_kernel_radiation): the one-species thin-lens families.
#if XLB_NOCHI && !XLB_BEAMFIELDS
#define XLB_RADIATION 1
#endif

// Beam-field kernels keep the warps of a CTA in step: one CTA barrier per lattice chunk.  Their
// hot code (field maps, Faddeeva loop, the thin-lens records in between) is several times the L0
// instruction cache of an SM sub-partition, and warps that run through the same records at the
// same time share every fetched line (PS Booster, C5: 2.78e8 -> 3.0e8 particle-turns/s; LHC with
// 74 lenses and the thin-lens families, whose loop fits the cache: no change -- measured,
// profiles/r2d_c5_sync_probe.json).
#if XLB_BEAMFIELDS && !defined(XLB_SYNC_CHUNK)
#define XLB_SYNC_CHUNK 1
#endif

#if XLB_BEAMFIELDS == 2
#define XLB_NS fast_bf6
#define XLB_FAMILY "/beamfields6d"
#elif XLB_BEAMFIELDS && XLB_NOCHI && XLB_MAXORDER
#define XLB_NS fast_bf_nc_lo
#define XLB_FAMILY "/beamfields/chi1/low-order"
#elif XLB_BEAMFIELDS
#define XLB_NS fast_bf
#define XLB_FAMILY "/beamfields"
#elif XLB_NOCHI && XLB_MAXORDER
#define XLB_NS fast_lean_nc_lo
#define XLB_FAMILY "/lean/chi1/low-order"
#elif XLB_NOCHI
#define XLB_NS fast_lean_nc
#define XLB_FAMILY "/lean/chi1"
#else
#define XLB_NS fast_lean
#define XLB_FAMILY "/lean"
#endif
#include "track_impl.cuh"
#include "variants.inc"

namespace xlb {
using namespace XLB_NS;

// (particles per thread, launch-bounds threads, resident CTAs per SM asked for)
#if XLB_BEAMFIELDS == 2
// Same launch bounds as the lean kernels: the thin-lens records dominate even a beam-beam
// lattice (74 lenses among 5 500 records on C3), so the register budget is set by them and
// the rarely executed beam-field code is allowed to spill.
#define XLB_SHAPES(X) X(1, 256, 2) X(2, 256, 2) X(3, 128, 3)
#elif XLB_BEAMFIELDS && XLB_NOCHI && defined(XLB_EXP_512)
#define XLB_SHAPES(X) X(1, 256, 2) X(2, 256, 2) X(2, 512, 1) X(3, 128, 3) X(4, 128, 3)
#elif XLB_BEAMFIELDS && XLB_NOCHI
#define XLB_SHAPES(X) X(1, 256, 2) X(2, 256, 2) X(3, 128, 3) X(4, 128, 3)
#elif XLB_BEAMFIELDS
#define XLB_SHAPES(X) X(1, 256, 2) X(2, 256, 2) X(3, 128, 3)
#elif XLB_NOCHI && XLB_MAXORDER
// four particles per thread at three CTAs per SM (168 registers): 1 536 particles per SM in
// flight against 1 152 for 3 x 128 x 3 -- C4 (PETRA IV) +23 %
#define XLB_SHAPES(X) X(1, 128, 5) X(2, 128, 3) X(3, 128, 4) X(4, 128, 3)
#elif XLB_NOCHI
#define XLB_SHAPES(X) X(1, 128, 5) X(1, 256, 3) X(1, 512, 2) X(2, 128, 3) X(2, 256, 2) X(3, 128, 3) X(4, 128, 3)
#else
#define XLB_SHAPES(X) X(1, 128, 5) X(1, 256, 3) X(1, 512, 2) X(2, 128, 3) X(2, 256, 2) X(3, 128, 3) X(4, 128, 2)
#endif

#define XLB_X_ENTRY(P, T, M) XLB_VARIANT_ENTRY("fast/ppt" #P "/t" #T XLB_FAMILY, P, T, M),
#define XLB_X_POLYGON_ENTRY(P, T, M) XLB_POLYGON_VARIANT_ENTRY("fast/ppt" #P "/t" #T XLB_FAMILY "/polygons", P, T, M),
#define XLB_X_RADIATION_ENTRY(P, T, M) \
  XLB_RADIATION_VARIANT_ENTRY("fast/ppt" #P "/t" #T XLB_FAMILY "/radiation", P, T, M),
static const Variant family_table[] = {
    XLB_SHAPES(XLB_X_ENTRY)
    XLB_TRACE_ENTRY("fast/trace" XLB_FAMILY),
    XLB_SHAPES(XLB_X_POLYGON_ENTRY)
    XLB_POLYGON_TRACE_ENTRY("fast/trace" XLB_FAMILY "/polygons"),
#if XLB_RADIATION
    XLB_SHAPES(XLB_X_RADIATION_ENTRY)
    XLB_RADIATION_TRACE_ENTRY("fast/trace" XLB_FAMILY "/radiation"),
#endif
};

#define XLB_CAT2(a, b) a##b
#define XLB_CAT(a, b) XLB_CAT2(a, b)
const Variant *XLB_CAT(XLB_NS, _variants)(int *n) {
  *n = static_cast<int>(sizeof(family_table) / sizeof(family_table[0]));
  return family_table;
}

#if XLB_BEAMFIELDS == 2
void fast_bb6d_launch(const KArgs &a, const unsigned long long *rec, int blocks, int threads, void *stream) {
  bf::bb6d_kernel<<<blocks, threads, 0, static_cast<cudaStream_t>(stream)>>>(
      a, reinterpret_cast<const double2 *>(rec));
}
#endif
}  // namespace xlb
