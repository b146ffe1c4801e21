// Kernel argument block shared by the tracking kernels and the host orchestration.
#pragma once
#include <stdint.h>

#ifndef XLB_STAGES
#define XLB_STAGES 3  // shared-memory ring depth for the lattice chunks
#endif

namespace xlb {

struct KArgs {
  const uint64_t *lat;  // packed lattice, device
  int chunk_words;
  int n_chunks;
  int num_turns;
  long long n;     // number of entries this launch covers (idx entries, or particles)
  const int *idx;  // optional survivor index list (device); nullptr = identity
  double *x, *px, *y, *py, *zeta, *delta, *rpp, *rvv, *s;
  const double *chi, *qr;
  long long *state, *at_element, *at_turn;
  const long long *pid;
  double q0, p0c, beta0, energy0;
  // q0^2 (1 - beta0^2) / (p0c beta0): the particle-independent factor of every space-charge kick
  // (be_beamfields/spacecharge.py:38-40), evaluated once per call on the host
  double sc_common;
  long long *loss_tally;
  double *mon;
  long long mon_words;
  unsigned int *n_lost;  // device counter, incremented per lost particle
  // work queue (nullptr = one item per CTA): [0] = next ticket, [1] = entries written, then a ring
  // of 64-bit READY entries (valid << 63 | segment << 32 | block) for the tickets beyond the first
  // n_blocks; zeroed before every launch.  n_items = n_blocks * ceil(num_turns / turns_per_item).
  unsigned int *queue;
  unsigned int n_blocks, n_items;
  int turns_per_item;
  // added to the per-particle turn counter at every END_TURN: 1, except for the passes over
  // the leading segments of a segmented lattice (xlb_lattice_t::segments), where it is 0
  int count_turns;
  int elem_off;  // added to the element index written to at_element (xlb_track_options_t)
  // element-by-element trace (debug kernels only): [n_elements][6][trace_n] fp64
  double *trace;
  long long trace_n;
};

struct Variant {
  const char *name;
  int strict, beamfields, ppt, threads, trace;
  int nochi;     // 1 = compiled for chi == 1 throughout (xlb_particles_t::chi == NULL)
  int maxorder;  // 0 = any multipole order; else the highest order the kernel evaluates (XLB_F_LOW_ORDER)
  int polygons;  // 1 = track_kernel_polygons: for the lattices flagged XLB_F_POLYGONS or XLB_F_EXCITER, only those
  int radiation;  // 1 = track_kernel_radiation (with the polygon case too): for XLB_F_RADIATION, and only those
  const void *func;  // the kernel's host stub
};

// The 6D beam-beam lens as a kernel of its own (segmented lattices): one particle per thread,
// `rec` = the BEAMBEAM6D record in the device copy of the lattice.
void fast_bb6d_launch(const KArgs &a, const unsigned long long *rec, int blocks, int threads, void *stream);

// Device self-test of the strict kernels' division sequences (track_strict.cu).
int strict_selftest_division(const double *d_divisors, int n_div, int mode, int per_thread,
                             unsigned long long seed, int span, unsigned long long *d_mismatches,
                             void *stream);

// Beam moments of slots 0..n-1 into the XLB_MOMENT_WORDS words at `out` (moments.cu); `scratch`
// holds beam_moments_scratch_words(n) doubles.
size_t beam_moments_scratch_words(long long n);
cudaError_t beam_moments_launch(const double *x, const double *px, const double *y, const double *py,
                                const double *zeta, const double *delta, const long long *state, long long n,
                                double *scratch, double *out, cudaStream_t st);

// NAFF tune and amplitude of n turn-major signals (naff.cu): sample t of signal j at
// u[t * stride + j] (and pu[..], nullptr for real signals); arguments checked by the caller.
cudaError_t naff_launch(const double *u, const double *pu, long long n, int num_turns, long long stride,
                        double beta, double alpha, double *tune, double *amplitude, cudaStream_t st);

namespace tangent {
// What the tangent-map kernel body carries (tangent.cu; include/xline_b200.h, "Tangent map"):
//   TANGENT   J, no radiating records (tangent_kernel);
//   TANGENT_R J, with mean-mode MULTIPOLE_RAD records (tangent_kernel_radiation);
//   ENVELOPE  Sigma <- J_e Sigma J_e^T per element, plus the quantum diffusion of every radiating half
//             (envelope_kernel).
enum Mode { TANGENT = 0, TANGENT_R = 1, ENVELOPE = 2 };
}  // namespace tangent

// Tangent-map tracking of the a.n particles (tangent.cu) in the kernel of `mode`: one particle per
// thread, `threads` per CTA, all a.num_turns turns in one launch; arguments checked by the caller.
// `jac` is J, or Sigma for ENVELOPE, [n][6][6]; log2_scale and fli are used by the tangent kernels,
// energy_loss by the envelope (the others may be null).
cudaError_t tangent_launch(tangent::Mode mode, const KArgs &a, double *jac, long long *log2_scale, double *fli,
                           double *energy_loss, int threads, cudaStream_t st);

// variant tables, one per translation unit (kernel family)
const Variant *fast_lean_variants(int *n);
const Variant *fast_lean_nc_variants(int *n);
const Variant *fast_lean_nc_lo_variants(int *n);
const Variant *fast_bf_variants(int *n);
const Variant *fast_bf_nc_lo_variants(int *n);
const Variant *fast_bf6_variants(int *n);
const Variant *strict_variants(int *n);
const Variant *strict_bf_variants(int *n);

}  // namespace xlb
