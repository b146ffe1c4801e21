// Launch policy of the tracking calls (cabi.cu): how many turns a launch takes, what shape the
// kernels are asked for, how many persistent CTAs run the work queue, and on which turns beam
// moments are stored.  Pure functions of sizes and options, free of CUDA, so that a plain C++
// compiler can build and test them (tests/test_launch_plan.py).
#pragma once
#include <algorithm>

#include "../../include/xline_b200.h"

namespace xlb {

// Turns per launch, at most: `turns_per_launch` 0 = automatic: long jobs are cut into launches of
// 100 turns so that survivors get re-compacted now and then; < 0 = one launch whatever the length
// (the kernel counts the chunks of a launch in 32 bits: a launch never exceeds 2^31 / n_chunks turns)
inline int launch_cap(int turns_per_launch, int num_turns, int n_chunks) {
  const int cap = std::max(1, static_cast<int>(0x7fffffffLL / std::max(1, n_chunks)));
  return std::min(cap, (turns_per_launch > 0) ? turns_per_launch
                       : (turns_per_launch == 0 && num_turns > 150 ? 100 : num_turns));
}

// Launch length for a loss rate: lanes of lost particles idle until the next launch boundary,
// on average rate * length / 2 of the lanes over a launch -- keep that near 3 %.
inline int launch_length_for_rate(double rate_per_turn, int longest) {
  if (!(rate_per_turn > 0)) return longest;
  const double len = 0.06 / rate_per_turn;
  if (len >= longest) return longest;
  return len < 1.0 ? 1 : static_cast<int>(len);
}

// The launch after one of `previous` turns that lost `rate_per_turn` of its particles per turn:
// the length for that rate, but at most twice the previous one.
inline int ramp_step(double rate_per_turn, int longest, int previous) {
  return static_cast<int>(std::min<long long>(launch_length_for_rate(rate_per_turn, longest), 2LL * previous));
}

// Particles per thread and threads per block asked of the variant tables for a launch over
// `n_now` particles on `sms` SMs; the caller's values (xlb_track_options_t) where they are > 0.
// Defaults from the B200 sweeps (scripts/probe_variants.py, scripts/probe_strict.py).  Thin-lens
// lattices of one species (chi == NULL): 4 particles per thread in 128-thread CTAs, 3 CTAs/SM at
// 168 registers = 1 536 particles in flight per SM (C2 +5 %, C4 +23 % over 3 x 128 x 3); with a
// chi column 3 x 128 (162 registers, no spills).  Strict C2: 1.08e7 particle-turns/s with 3 x 128
// against 9.1e6 (2 x 128), 7.3e6 (1 x 256), 6.7e6 (2 x 256).  Beam-field lattices: 2 x 256 unless
// the caller knows the lenses are sparse (xline_b200/line.py decides from the record counts).
struct LaunchRequest {
  int ppt, threads;
};
inline LaunchRequest launch_request(int particles_per_thread, int threads_per_block, bool strict, bool beamfields,
                                    bool chi, long long n_now, int sms) {
  int ppt = particles_per_thread;
  if (ppt <= 0) {
    if (beamfields) ppt = 2;
    else if (strict || chi) ppt = 3;
    else ppt = 4;
    if (!beamfields && threads_per_block <= 0) {
      // (below 2 only for beams that cannot give every SM one 128-thread CTA: one particle per
      // thread doubles the warps but also the per-record instructions issued, and loses on the
      // C2 lattice from 30 000 particles on -- profiles/r2_sweep_n.json; C1's 10 000 particles
      // on 79 CTAs instead of 40: 3.3e9 against 2.3e9 particle-turns/s)
      // (three per thread wins nowhere in the closing sweep, profiles/r2c_sweep_n.json: 200 k
      // particles 2.45e7 with two, 2.38e7 with three, 2.11e7 with four)
      if (ppt > 2 && n_now < static_cast<long long>(ppt) * 128 * 3 * sms) ppt = 2;
      if (ppt == 2 && n_now < 128LL * sms) ppt = 1;
    }
  }
  return {ppt, threads_per_block > 0 ? threads_per_block : (beamfields && ppt < 3 ? 256 : 128)};
}

// CTAs of a persistent launch over `blocks` particle blocks, of which the device holds `resident`
// at once on `sms` SMs.  Fewer CTAs than blocks (unless the blocks load every SM equally): the
// blocks beyond the grid wait in the ring, whose FIFO order then rotates the blocks over the CTAs,
// and all of them advance at the average speed.  (With every block resident on a CTA of its own a
// finishing CTA finds only its own block in the ring -- a static assignment, as slow as the CTAs of
// the fullest SMs: C2 at 125 k particles 1.9e7 against 2.2e7.)  Preferably the same number of CTAs
// on every SM; when that would idle more than 15 % of the CTAs, a backlog of 1/16 of the blocks.
inline int persistent_grid(int blocks, int resident, int sms) {
  const int q = std::min(blocks, resident), rem = q % sms;
  return (rem * 100 <= q * 15) ? q - rem : q - std::max(1, q / 16);
}

// Turn of store k of `spec` (after start + k * skip turns), or num_turns + 1 when there is none
// left in a call of num_turns turns.
inline long long moment_store_turn(const xlb_moments_spec_t &spec, long long k, long long num_turns) {
  if (k >= spec.num_stores || spec.start > num_turns) return num_turns + 1;
  if (k > 0 && spec.skip > (num_turns - spec.start) / k) return num_turns + 1;
  return spec.start + k * spec.skip;
}

}  // namespace xlb
