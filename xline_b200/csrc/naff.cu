// NAFF tunes (include/xline_b200.h, xlb_naff_device): the frequency of the largest spectral line
// of every turn-by-turn signal of a BeamMonitor slab, and its amplitude.
//
// Shape: one warp per signal, W = 4 / 2 / 1 consecutive signals per CTA (M <= 1024 / 2048 /
// larger), so one turn's loads of a CTA fill a 32-byte sector where W = 4.  A warp owns M complex
// doubles of dynamic shared memory (16·M bytes, 64 KiB per CTA, 128 KiB at M = 8192):
//   1. load z_t (t = lane, lane + 32, ..), check finiteness, sum for the mean;
//   2. centre, window, zero-pad to M, bit-reverse in place, radix-2 DIT FFT; the twiddles
//      e^{-iπ j/h} come from sincospi, M - 1 of them per signal;
//   3. coarse peak: argmax |X_k|² over k = 1 .. M-1 (complex) or 1 .. M/2 (real), lowest k on ties;
//   4. reload the centred, windowed samples in natural order; Newton on D(ν) = Re(conj(Z)·Z')
//      with a bisection safeguard.  One pass over the samples gives S_p = Σ t_c^p·w_t·z_t·e_t,
//      p = 0, 1, 2, with t_c = t - T/2 and e_t = e^{-2πiν t_c}:  Z = S_0, Z' = -2πi·S_1,
//      Z'' = -4π²·S_2.  e_t follows a lane's turns by the rotation e^{-2πiν·32} and is re-seeded
//      exactly every NF_RESEED steps from sincospi of the reduced argument ν·t_c - rint(ν·t_c);
//   5. fold ν into [0, 1) (complex) or [0, 1/2] (real).
// Every sum runs over t in increasing order within a lane, then over the lanes by an xor
// butterfly, which leaves the same bits in all lanes: a signal's result depends on its samples,
// T, the real/complex choice and (β, α) only -- not on n, its column, the row stride or W.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/xline_b200.h"
#include "kargs.h"

namespace xlb {

constexpr int NF_MAX_ITER = 40;  // Newton / bisection steps (a bracket of 2/M halves to 1e-15 in 40)
constexpr int NF_RESEED = 8;     // lane steps (of 32 turns) between exact phase seeds
constexpr double NF_TOL = 1e-15;  // stop when a step is below this
constexpr unsigned NF_FULL = 0xffffffffu;

struct Cx {
  double re, im;
};
__device__ __forceinline__ Cx cmul(Cx a, Cx b) { return {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re}; }

// e^{-2πi x}, from the argument reduced to [-1/2, 1/2] (x - rint(x) is exact)
__device__ __forceinline__ Cx phase(double x) {
  double s, c;
  sincospi(2.0 * (x - rint(x)), &s, &c);
  return {c, -s};
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) v += __shfl_xor_sync(NF_FULL, v, d);  // a + b == b + a: same bits in all lanes
  return v;
}

struct NaffSignal {
  const double *u, *pu;  // pu == nullptr: real signal
  long long stride, j;
  double isb, alpha, beta;  // 1/√β, α, β
  // z_t (complex: u/√β - i·(α·u + β·pu)/√β); `finite` is cleared on a non-finite sample
  __device__ __forceinline__ Cx z(int t, bool &finite) const {
    const long long i = static_cast<long long>(t) * stride + j;
    const double a = u[i];
    if (!pu) {
      finite = finite && isfinite(a);
      return {a, 0.0};
    }
    const double b = pu[i];
    finite = finite && isfinite(a) && isfinite(b);
    // explicit roundings: both load sites (steps 1 and 4) give the same bits
    return {__dmul_rn(a, isb), -__dmul_rn(fma(alpha, a, __dmul_rn(beta, b)), isb)};
  }
};

// Hann window 1 - cos(2πt/T) = 2·sin²(πt/T)
__device__ __forceinline__ double hann(int t, int T) {
  const double s = sinpi(static_cast<double>(t) / T);
  return 2.0 * s * s;
}

__global__ void __launch_bounds__(128) naff_kernel(const double *__restrict__ u, const double *__restrict__ pu,
                                                   long long n, int T, int log2M, long long stride, double isb,
                                                   double alpha, double beta, double *__restrict__ tune,
                                                   double *__restrict__ amplitude) {
  extern __shared__ double2 naff_smem[];
  const int lane = threadIdx.x & 31;
  const int M = 1 << log2M;
  const long long j = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (j >= n) return;  // warp-uniform
  double2 *X = naff_smem + static_cast<size_t>(threadIdx.x >> 5) * M;
  const NaffSignal sig{u, pu, stride, j, isb, alpha, beta};

  // 1. samples, finiteness, mean
  bool finite = true;
  double mr = 0.0, mi = 0.0;
  for (int t = lane; t < T; t += 32) {
    const Cx v = sig.z(t, finite);
    X[t] = make_double2(v.re, v.im);
    mr += v.re;
    mi += v.im;
  }
  if (__any_sync(NF_FULL, !finite)) {
    if (lane == 0) tune[j] = amplitude[j] = __longlong_as_double(0x7ff8000000000000LL);
    return;
  }
  mr = warp_sum(mr) / T;
  mi = warp_sum(mi) / T;

  // 2. centre, window, zero-pad; FFT
  bool nonzero = false;
  for (int t = lane; t < M; t += 32) {
    double2 v = make_double2(0.0, 0.0);
    if (t < T) {
      v = X[t];
      v.x -= mr;
      v.y -= mi;
      nonzero = nonzero || v.x != 0.0 || v.y != 0.0;
      const double w = hann(t, T);
      v.x *= w;
      v.y *= w;
    }
    X[t] = v;
  }
  if (!__any_sync(NF_FULL, nonzero)) {
    if (lane == 0) {
      tune[j] = __longlong_as_double(0x7ff8000000000000LL);
      amplitude[j] = 0.0;
    }
    return;
  }
  __syncwarp();
  for (int i = lane; i < M; i += 32) {
    const int r = static_cast<int>(__brev(static_cast<unsigned>(i)) >> (32 - log2M));
    if (i < r) {
      const double2 a = X[i];
      X[i] = X[r];
      X[r] = a;
    }
  }
  __syncwarp();
  for (int lh = 0; lh < log2M; ++lh) {
    const int h = 1 << lh;
    if (h < 32) {  // lane's twiddle index j = lane mod h for all of its butterflies b = lane + 32m
      const int jj = lane & (h - 1);
      double s, c;
      sincospi(static_cast<double>(jj) / h, &s, &c);
      for (int b = lane; b < M / 2; b += 32) {
        const int i0 = ((b >> lh) << (lh + 1)) | jj, i1 = i0 + h;
        const double2 a = X[i0], e = X[i1];
        const double br = e.x * c + e.y * s, bi = e.y * c - e.x * s;  // e · (c - i s)
        X[i0] = make_double2(a.x + br, a.y + bi);
        X[i1] = make_double2(a.x - br, a.y - bi);
      }
    } else {
      for (int jj = lane; jj < h; jj += 32) {
        double s, c;
        sincospi(static_cast<double>(jj) / h, &s, &c);
        for (int g = 0; g < M; g += 2 * h) {
          const int i0 = g + jj, i1 = i0 + h;
          const double2 a = X[i0], e = X[i1];
          const double br = e.x * c + e.y * s, bi = e.y * c - e.x * s;
          X[i0] = make_double2(a.x + br, a.y + bi);
          X[i1] = make_double2(a.x - br, a.y - bi);
        }
      }
    }
    __syncwarp();
  }

  // 3. coarse peak
  const int kmax = pu ? M - 1 : M / 2;
  double best = -1.0;
  int bk = 0;
  for (int k = 1 + lane; k <= kmax; k += 32) {
    const double2 v = X[k];
    const double p = v.x * v.x + v.y * v.y;
    if (p > best) {
      best = p;
      bk = k;
    }
  }
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) {
    const double ob = __shfl_xor_sync(NF_FULL, best, d);
    const int ok = __shfl_xor_sync(NF_FULL, bk, d);
    if (ob > best || (ob == best && ok < bk)) {
      best = ob;
      bk = ok;
    }
  }
  __syncwarp();

  // 4. centred, windowed samples in natural order (the same operations as in 1 and 2)
  for (int t = lane; t < T; t += 32) {
    const Cx v = sig.z(t, finite);
    const double w = hann(t, T);
    X[t] = make_double2((v.re - mr) * w, (v.im - mi) * w);
  }
  __syncwarp();

  const double half = 0.5 * T;
  double lo = (bk - 1) / static_cast<double>(M), hi = (bk + 1) / static_cast<double>(M);
  double nu = bk / static_cast<double>(M);
  Cx s0{0.0, 0.0};
  for (int it = 0; it < NF_MAX_ITER; ++it) {
    Cx s1{0.0, 0.0}, s2{0.0, 0.0};
    s0 = Cx{0.0, 0.0};
    const Cx r = phase(32.0 * nu);
    for (int base = lane; base < T; base += 32 * NF_RESEED) {
      Cx e = phase(nu * (base - half));
#pragma unroll
      for (int q = 0; q < NF_RESEED; ++q) {
        const int t = base + 32 * q;
        if (t < T) {
          const double tc = t - half;
          const double2 v = X[t];
          const Cx a = cmul(Cx{v.x, v.y}, e);
          s0.re += a.re;
          s0.im += a.im;
          s1.re = fma(tc, a.re, s1.re);
          s1.im = fma(tc, a.im, s1.im);
          const double tc2 = tc * tc;
          s2.re = fma(tc2, a.re, s2.re);
          s2.im = fma(tc2, a.im, s2.im);
          e = cmul(e, r);
        }
      }
    }
    s0.re = warp_sum(s0.re);
    s0.im = warp_sum(s0.im);
    s1.re = warp_sum(s1.re);
    s1.im = warp_sum(s1.im);
    s2.re = warp_sum(s2.re);
    s2.im = warp_sum(s2.im);
    // D = 2π·Im(conj(S0)·S1),  D' = 4π²·(|S1|² - Re(conj(S0)·S2)) < 0 at a maximum of |Z|
    const double d = s0.re * s1.im - s0.im * s1.re;
    const double dd = (s1.re * s1.re + s1.im * s1.im) - (s0.re * s2.re + s0.im * s2.im);
    // D = 0 is the answer only at a maximum: a real signal has D(1/2) = 0 by symmetry, also when
    // 1/2 is the minimum between a line and its mirror image
    if (d == 0.0 && dd < 0.0) break;
    if (d > 0.0)
      lo = nu;
    else
      hi = nu;
    double next = nu - d / (2.0 * M_PI * dd);
    if (!(dd < 0.0) || !(next >= lo && next <= hi)) next = 0.5 * (lo + hi);  // inclusive: a converged step is 0
    const double step = fabs(next - nu);
    nu = next;
    if (step < NF_TOL) break;
  }
  // The brackets of k = M - 1 (complex) and k = M/2 (real) reach past the range: fold (exactly) into
  // [0, 1) and [0, 1/2] -- the same frequency, seen modulo 1 and, for a real signal, up to sign.
  if (pu ? nu >= 1.0 : nu > 0.5) nu = pu ? nu - 1.0 : 1.0 - nu;
  if (lane == 0) {
    tune[j] = nu;
    amplitude[j] = hypot(s0.re, s0.im) / T;  // Σ w_t = T
  }
}

cudaError_t naff_launch(const double *u, const double *pu, long long n, int num_turns, long long stride,
                        double beta, double alpha, double *tune, double *amplitude, cudaStream_t st) {
  int log2M = 0;
  while ((1 << log2M) < num_turns) ++log2M;
  const int w = log2M <= 10 ? 4 : log2M == 11 ? 2 : 1;  // signals per CTA: 64 KiB of shared memory or less
  const size_t smem = static_cast<size_t>(w) << (log2M + 4);
  cudaError_t e = cudaFuncSetAttribute(naff_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(smem));
  if (e != cudaSuccess) return e;
  const long long grid = (n + w - 1) / w;
  const double isb = pu ? 1.0 / sqrt(beta) : 1.0;
  naff_kernel<<<static_cast<unsigned>(grid), 32 * w, smem, st>>>(u, pu, n, num_turns, log2M, stride, isb, alpha,
                                                                 beta, tune, amplitude);
  return cudaGetLastError();
}

}  // namespace xlb
