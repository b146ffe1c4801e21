// Beam moments (include/xline_b200.h, XLB_MOMENT_*): particle count and the first and second
// moments of (x, px, y, py, zeta, delta) over the surviving beam, as exact double-double sums
// in a summation order that depends on the slot index alone.
//
// Shape of the sum: a perfect binary tree over the slots 0 .. n-1, padded with zeros.  A tile of
// MO_TILE = 2048 consecutive slots is one CTA: each thread adds its 8 consecutive slots pairwise,
// a warp folds its 32 threads by shuffles (lane i takes lane i + d, d = 1, 2, .. 16), and the
// CTA folds its 8 warps pairwise.  The tile sums go to scratch, and the same tree folds groups of
// 2048 tile sums until one is left.  Launch shapes are fixed, no atomics: the result depends on
// n and the columns only.  Every addition is AccurateDWPlusDW (Joldes, Muller, Popescu 2017),
// relative error <= 3 u^2 / (1 - 4 u), u = 2^-53; an addition with a zero operand is exact, so a
// root-to-leaf path of the tree holds at most ceil(log2 n) inexact additions.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/xline_b200.h"
#include "kargs.h"

namespace xlb {

constexpr int MO_THREADS = 256;
constexpr int MO_ITEMS = 8;
constexpr int MO_TILE = MO_THREADS * MO_ITEMS;
constexpr int MO_WARPS = MO_THREADS / 32;
static_assert(XLB_MOMENT_WORDS == 2 + 2 * XLB_MOMENT_PAIRS, "moment store layout");

struct DD {
  double hi, lo;
};

__device__ __forceinline__ DD two_sum(double a, double b) {
  const double s = __dadd_rn(a, b);
  const double bb = __dsub_rn(s, a);
  const double e = __dadd_rn(__dsub_rn(a, __dsub_rn(s, bb)), __dsub_rn(b, bb));
  return {s, e};
}
__device__ __forceinline__ DD fast_two_sum(double a, double b) {  // |a| >= |b| or a == 0
  const double s = __dadd_rn(a, b);
  return {s, __dsub_rn(b, __dsub_rn(s, a))};
}
__device__ __forceinline__ DD dd_add(DD a, DD b) {  // AccurateDWPlusDW
  const DD s = two_sum(a.hi, b.hi);
  const DD t = two_sum(a.lo, b.lo);
  DD v = fast_two_sum(s.hi, __dadd_rn(s.lo, t.hi));
  return fast_two_sum(v.hi, __dadd_rn(t.lo, v.lo));
}
__device__ __forceinline__ DD two_prod(double a, double b) {
  const double p = __dmul_rn(a, b);
  return {p, fma(a, b, -p)};
}
__device__ __forceinline__ DD shfl_down(DD v, int d) {
  return {__shfl_down_sync(0xffffffffu, v.hi, d), __shfl_down_sync(0xffffffffu, v.lo, d)};
}

// (u, v) of pair q >= XLB_MOMENT_FIRST: upper triangle of the 6 x 6 products, row-major
__host__ __device__ constexpr int pair_u(int q) {
  return q < 6 ? q : (q < 12 ? 0 : q < 17 ? 1 : q < 21 ? 2 : q < 24 ? 3 : q < 26 ? 4 : 5);
}
__host__ __device__ constexpr int pair_v(int q) {
  return q < 6 ? q : q - 6 - (pair_u(q) * (13 - pair_u(q))) / 2 + pair_u(q);
}
static_assert(pair_u(6) == 0 && pair_v(6) == 0 && pair_v(11) == 5 && pair_u(12) == 1 && pair_v(12) == 1 &&
                  pair_v(16) == 5 && pair_u(17) == 2 && pair_v(17) == 2 && pair_v(20) == 5 && pair_u(21) == 3 &&
                  pair_v(21) == 3 && pair_v(23) == 5 && pair_u(24) == 4 && pair_v(25) == 5 && pair_u(26) == 5 &&
                  pair_v(26) == 5,
              "pair table");

// Folds the per-thread leaf sum `v` of one pair over the CTA: lane 0 of every warp parks its
// warp's sum in sh[warp].
__device__ __forceinline__ void warp_fold(DD v, DD *sh) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const DD o = shfl_down(v, d);
    if ((threadIdx.x & (2 * d - 1)) == 0) v = dd_add(v, o);
  }
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
}

// The 8 warp sums of pair q, pairwise, into out[2 + 2q .. 3 + 2q]; out[0..1] from the counts.
__device__ __forceinline__ void cta_finish(DD (*sh)[MO_WARPS], const double (*cnt)[MO_WARPS], double *out) {
  const int q = threadIdx.x;
  if (q < XLB_MOMENT_PAIRS) {
    DD a[MO_WARPS];
#pragma unroll
    for (int w = 0; w < MO_WARPS; ++w) a[w] = sh[q][w];
#pragma unroll
    for (int d = 1; d < MO_WARPS; d <<= 1)
#pragma unroll
      for (int w = 0; w < MO_WARPS; w += 2 * d) a[w] = dd_add(a[w], a[w + d]);
    out[2 + 2 * q] = a[0].hi;
    out[3 + 2 * q] = a[0].lo;
  } else if (q < XLB_MOMENT_PAIRS + 2) {
    const int c = q - XLB_MOMENT_PAIRS;
    double t = 0.0;  // integers below 2^31: exact in any order
    for (int w = 0; w < MO_WARPS; ++w) t += cnt[c][w];
    out[c] = t;
  }
}

__device__ __forceinline__ double count_fold(double c) {
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) c += __shfl_down_sync(0xffffffffu, c, d);
  return c;
}

// One tile of slots per CTA -> 56 words at out + 56 * blockIdx.x.
__global__ void __launch_bounds__(MO_THREADS) beam_moments_tiles(
    const double *__restrict__ x, const double *__restrict__ px, const double *__restrict__ y,
    const double *__restrict__ py, const double *__restrict__ zeta, const double *__restrict__ delta,
    const long long *__restrict__ state, long long n, double *__restrict__ out) {
  __shared__ DD sh[XLB_MOMENT_PAIRS][MO_WARPS];
  __shared__ double cnt[2][MO_WARPS];
  const long long base = static_cast<long long>(blockIdx.x) * MO_TILE + threadIdx.x * MO_ITEMS;
  double c[6][MO_ITEMS];
  double n_ok = 0.0, n_bad = 0.0;
#pragma unroll
  for (int j = 0; j < MO_ITEMS; ++j) {
    const long long i = base + j;
    bool alive = false;
#pragma unroll
    for (int k = 0; k < 6; ++k) c[k][j] = 0.0;
    if (i < n) {
      alive = state[i] == 1;
      c[0][j] = x[i]; c[1][j] = px[i]; c[2][j] = y[i];
      c[3][j] = py[i]; c[4][j] = zeta[i]; c[5][j] = delta[i];
    }
    bool finite = true;
#pragma unroll
    for (int k = 0; k < 6; ++k) finite = finite && isfinite(c[k][j]);
    const bool ok = alive && finite;
    n_ok += ok ? 1.0 : 0.0;
    n_bad += (alive && !finite) ? 1.0 : 0.0;
#pragma unroll
    for (int k = 0; k < 6; ++k) c[k][j] = ok ? c[k][j] : 0.0;  // a zero term: exact, as if absent
  }
  n_ok = count_fold(n_ok);
  n_bad = count_fold(n_bad);
  if ((threadIdx.x & 31) == 0) {
    cnt[0][threadIdx.x >> 5] = n_ok;
    cnt[1][threadIdx.x >> 5] = n_bad;
  }
#pragma unroll
  for (int q = 0; q < XLB_MOMENT_PAIRS; ++q) {
    DD a[MO_ITEMS];
#pragma unroll
    for (int j = 0; j < MO_ITEMS; ++j)
      a[j] = q < 6 ? DD{c[q][j], 0.0} : two_prod(c[pair_u(q)][j], c[pair_v(q)][j]);
#pragma unroll
    for (int d = 1; d < MO_ITEMS; d <<= 1)
#pragma unroll
      for (int j = 0; j < MO_ITEMS; j += 2 * d) a[j] = dd_add(a[j], a[j + d]);
    warp_fold(a[0], sh[q]);
  }
  __syncthreads();
  cta_finish(sh, cnt, out + static_cast<size_t>(blockIdx.x) * XLB_MOMENT_WORDS);
}

// The same tree over groups of MO_TILE partial stores: `in` holds `m` stores of 56 words.
__global__ void __launch_bounds__(MO_THREADS) beam_moments_fold(const double *__restrict__ in, long long m,
                                                                 double *__restrict__ out) {
  __shared__ DD sh[XLB_MOMENT_PAIRS][MO_WARPS];
  __shared__ double cnt[2][MO_WARPS];
  const long long base = static_cast<long long>(blockIdx.x) * MO_TILE + threadIdx.x * MO_ITEMS;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    double t = 0.0;
    for (int j = 0; j < MO_ITEMS; ++j)
      if (base + j < m) t += in[(base + j) * XLB_MOMENT_WORDS + k];
    t = count_fold(t);
    if ((threadIdx.x & 31) == 0) cnt[k][threadIdx.x >> 5] = t;
  }
  for (int q = 0; q < XLB_MOMENT_PAIRS; ++q) {
    DD a[MO_ITEMS];
#pragma unroll
    for (int j = 0; j < MO_ITEMS; ++j) {
      const long long i = base + j;
      a[j] = i < m ? DD{in[i * XLB_MOMENT_WORDS + 2 + 2 * q], in[i * XLB_MOMENT_WORDS + 3 + 2 * q]} : DD{0.0, 0.0};
    }
#pragma unroll
    for (int d = 1; d < MO_ITEMS; d <<= 1)
#pragma unroll
      for (int j = 0; j < MO_ITEMS; j += 2 * d) a[j] = dd_add(a[j], a[j + d]);
    warp_fold(a[0], sh[q]);
  }
  __syncthreads();
  cta_finish(sh, cnt, out + static_cast<size_t>(blockIdx.x) * XLB_MOMENT_WORDS);
}

static long long tiles_of(long long n) { return n <= MO_TILE ? 1 : (n + MO_TILE - 1) / MO_TILE; }

size_t beam_moments_scratch_words(long long n) {
  // first level of tile sums, then every further level (ping-pong in two halves)
  const long long t0 = tiles_of(n);
  const long long t1 = t0 > 1 ? tiles_of(t0) : 0;
  return static_cast<size_t>(t0 + t1) * XLB_MOMENT_WORDS;
}

cudaError_t beam_moments_launch(const double *x, const double *px, const double *y, const double *py,
                                const double *zeta, const double *delta, const long long *state, long long n,
                                double *scratch, double *out, cudaStream_t st) {
  long long m = tiles_of(n);
  double *a = scratch, *b = scratch + static_cast<size_t>(m) * XLB_MOMENT_WORDS;
  beam_moments_tiles<<<static_cast<unsigned>(m), MO_THREADS, 0, st>>>(x, px, y, py, zeta, delta, state, n,
                                                                       m == 1 ? out : a);
  while (m > 1) {
    const long long g = tiles_of(m);
    beam_moments_fold<<<static_cast<unsigned>(g), MO_THREADS, 0, st>>>(a, m, g == 1 ? out : b);
    double *t = a;
    a = b;
    b = t;
    m = g;
  }
  return cudaGetLastError();
}

}  // namespace xlb
