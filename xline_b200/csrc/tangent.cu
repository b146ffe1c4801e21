// Tangent-map tracking (include/xline_b200.h, "Tangent map"; DESIGN.md §4.8): every particle is
// tracked as Line.track tracks it, and carries J = dz/dz0 over z = (x, px, y, py, zeta, delta),
// updated record by record as J <- J_elem(z before the element) . J.
//
// One particle per thread; the state, J (36 doubles) and the loop variables stay in registers.
// The lattice is the element-by-element packing (one record per element, no fused block records,
// Line.track_tangent), read straight from global memory through L1/L2: the records of a turn are
// the same for every thread, so after the first warp they are cache hits.
//
// The coordinates are advanced by the tracking kernels' own element functions (track_impl.cuh,
// beamfields.cuh, instantiated here for one particle per thread); the Jacobian of each element is
// written out next to them from the same definitions and applied as row updates (a thin kick only
// changes the px and py rows, a drift the x, y and zeta rows).  Through the energy bookkeeping
// rpp = 1/(1+delta) and rvv = beta/beta0 are functions of delta:
//   E = 1 + ptau*beta0 = (1+delta)/rvv,   d rvv / d delta = (1 - beta0^2) / E^3.
#define XLB_STRICT 0
#define XLB_BEAMFIELDS 1
#define XLB_NOCHI 0
#define XLB_MAXORDER 0
#define XLB_NS tangent
#include "track_impl.cuh"

namespace xlb {
namespace tangent {

using Jac = double[6][6];
enum { X = 0, PX = 1, Y = 2, PY = 3, ZETA = 4, DELTA = 5 };

// The kernel body is a template over what it carries, MODE (kargs.h: TANGENT, TANGENT_R, ENVELOPE).

__device__ __forceinline__ void transpose(Jac &J) {
#pragma unroll
  for (int q = 0; q < 6; ++q)
#pragma unroll
    for (int c = q + 1; c < 6; ++c) {
      const double t = J[q][c];
      J[q][c] = J[c][q];
      J[c][q] = t;
    }
}

// Applies the row update F(A) = J_e A of an element, a statement on J that reads the state before
// the element only: once to J, or as F(F(Sigma)^T) = J_e Sigma J_e^T to a symmetric Sigma (the
// envelope).  A macro rather than a function taking a lambda: the tangent kernel compiles to the
// same code as it did before the envelope existed.
#define TAN_ROWS(...)         \
  do {                        \
    __VA_ARGS__;              \
    if (MODE == ENVELOPE) {   \
      transpose(J);           \
      __VA_ARGS__;            \
    }                         \
  } while (0)

// row r of J += a * row s
__device__ __forceinline__ void axpy(Jac &J, int r, double a, int s) {
#pragma unroll
  for (int c = 0; c < 6; ++c) J[r][c] = fma(a, J[s][c], J[r][c]);
}

// sin and cos of x through sincospi of x/pi carried in two words (within ~2 ulp of sin, cos for the
// phases an RF element sees).  CUDA's sin / cos keep a 40-byte local array for the Payne-Hanek
// reduction of huge arguments, which would give this kernel a stack frame.
__device__ __forceinline__ void sincos_ns(double x, double &s, double &c) {
  const double ip_hi = 0.3183098861837907, ip_lo = -1.9678676675182486e-17;  // 1/pi
  const double t = x * ip_hi;
  const double tl = fma(x, ip_hi, -t) + x * ip_lo;
  double sp, cp;
  sincospi(t, &sp, &cp);
  const double d = 3.141592653589793 * tl;
  s = fma(d, cp, sp);
  c = fma(-d, sp, cp);
}

__device__ __forceinline__ double drvv_ddelta(double beta0, double delta, double rvv) {
  const double E = (1.0 + delta) / rvv;
  return (1.0 - beta0 * beta0) / (E * E * E);
}

// Expanded drift (el_drift; xline/elements.py:48-56).
__device__ __forceinline__ void jac_drift(Jac &J, const Regs<1> &r, double beta0, double L) {
  const double rpp = r.rpp[0], xp = r.px[0] * rpp, yp = r.py[0] * rpp;
  const double dxd = -xp * rpp * L, dyd = -yp * rpp * L;
  const double dzpx = -L * xp * rpp, dzpy = -L * yp * rpp;
  const double dzd = L * (drvv_ddelta(beta0, r.delta[0], r.rvv[0]) + (xp * xp + yp * yp) * rpp);
#pragma unroll
  for (int c = 0; c < 6; ++c) {
    const double jpx = J[PX][c], jpy = J[PY][c], jd = J[DELTA][c];
    J[X][c] += rpp * L * jpx + dxd * jd;
    J[Y][c] += rpp * L * jpy + dyd * jd;
    J[ZETA][c] += dzpx * jpx + dzpy * jpy + dzd * jd;
  }
}

// Exact drift (el_drift_exact; xline/elements.py:64-72).
__device__ __forceinline__ void jac_drift_exact(Jac &J, const Regs<1> &r, double beta0, double L) {
  const double opd = 1.0 + r.delta[0], px = r.px[0], py = r.py[0];
  const double pz = sqrt(opd * opd - px * px - py * py);
  const double lpzi = L / pz, g = lpzi / (pz * pz);  // g = L / pz^3
  const double rv1 = drvv_ddelta(beta0, r.delta[0], r.rvv[0]);
#pragma unroll
  for (int c = 0; c < 6; ++c) {
    const double jpx = J[PX][c], jpy = J[PY][c], jd = J[DELTA][c];
    const double dl = g * (px * jpx + py * jpy - opd * jd);  // d lpzi
    J[X][c] += lpzi * jpx + px * dl;
    J[Y][c] += lpzi * jpy + py * dl;
    J[ZETA][c] += L * rv1 * jd - lpzi * jd - opd * dl;
  }
}

// P' = dr + i di at z = x + i y of P(z) = sum (kn_i + i ks_i) z^i / i!, pairs[m] = (kn, ks)[order - m]
// / (order - m)!: the Horner sweep of P carrying its derivative along.
__device__ __forceinline__ void horner_prime(const double2 *pairs, int order, double x, double y, double &dr,
                                             double &di) {
  double pr = pairs[0].x, pi = pairs[0].y, qr = 0.0, qi = 0.0;
  for (int m = 1; m <= order; ++m) {
    const double2 k = pairs[m];
    const double tr = fma(qr, x, fma(-qi, y, pr)), ti = fma(qr, y, fma(qi, x, pi));
    qr = tr;
    qi = ti;
    const double ur = fma(pr, x, fma(-pi, y, k.x)), ui = fma(pr, y, fma(pi, x, k.y));
    pr = ur;
    pi = ui;
  }
  dr = qr;
  di = qi;
}

// Thin multipole, straight or curved (el_multipole, el_multipole_curved; xline/elements.py:120-156):
// dpx = -chi Re P, dpy = chi Im P.
__device__ __forceinline__ void jac_multipole(Jac &J, const Regs<1> &r, const double2 *pairs, int order,
                                              bool curved, double hxl, double hyl, double inv_len) {
  const double x = r.x[0], y = r.y[0], chi = r.chi[0];
  double dr, di;
  horner_prime(pairs, order, x, y, dr, di);
  // d(-chi Re P)/dx = -chi Re P', /dy = chi Im P';  d(chi Im P)/dx = chi Im P', /dy = chi Re P'
  double axx = -chi * dr, axy = chi * di, ayx = chi * di, ayy = chi * dr, axd = 0.0, ayd = 0.0;
  double zx = 0.0, zy = 0.0;
  if (curved) {
    const double2 k0 = pairs[order];  // knl[0], ksl[0]
    axx -= chi * k0.x * hxl * inv_len;
    ayy += chi * k0.y * hyl * inv_len;
    axd = hxl;
    ayd = -hyl;
    zx = -chi * hxl;
    zy = chi * hyl;
  }
#pragma unroll
  for (int c = 0; c < 6; ++c) {
    const double jx = J[X][c], jy = J[Y][c], jd = J[DELTA][c];
    J[PX][c] += axx * jx + axy * jy + axd * jd;
    J[PY][c] += ayx * jx + ayy * jy + ayd * jd;
    J[ZETA][c] += zx * jx + zy * jy;
  }
}

// The chain through Pyparticles.add_to_energy (track_impl.cuh) of an energy change W whose
// gradient over (x, y, zeta, delta) is (gx, gy, gz, gd).  delta and rvv after it are functions of
// P1 = 1 + ptau*beta0 after; zeta' = zeta rvv'/rvv.
struct EnergyChain {
  double opdn;                  // 1 + delta after
  double dd_dP, drvv_dP;        // d delta' / d P1, d rvv' / d P1
  double rr, zr, rv1;           // rvv'/rvv, zeta/rvv, d rvv / d delta before
  double px_, py_, pz_, pd_;    // gradient of P1 over (x, y, zeta, delta)

  __device__ __forceinline__ EnergyChain(const Regs<1> &r, double beta0, double energy0, double W, double gx,
                                         double gy, double gz, double gd) {
    const double delta = r.delta[0], rvv = r.rvv[0];
    const double E = (1.0 + delta) / rvv;               // 1 + ptau*beta0 before
    const double P1 = E + W / energy0;                  // 1 + ptau*beta0 after
    const double ptau = (P1 - 1.0) / beta0;
    opdn = sqrt(ptau * ptau + 2.0 * ptau / beta0 + 1.0);
    const double rvvn = opdn / P1;                      // rvv after
    dd_dP = P1 / (beta0 * beta0 * opdn);
    drvv_dP = dd_dP / P1 - opdn / (P1 * P1);
    rv1 = (1.0 - beta0 * beta0) / (E * E * E);
    px_ = gx / energy0;
    py_ = gy / energy0;
    pz_ = gz / energy0;
    pd_ = gd / energy0 + beta0 * beta0 * (1.0 + delta) / E;
    zr = r.zeta[0] / rvv;
    rr = rvvn / rvv;
  }

  // P1's entry in a column of J from the column's x, y, zeta, delta entries.  ZGRAD: W depends on
  // zeta.  Without it the term is absent, not multiplied by 0 (which would turn an infinite jz
  // into NaN).
  template <bool ZGRAD>
  __device__ __forceinline__ double dP(double jx, double jy, double jz, double jd) const {
    return ZGRAD ? px_ * jx + py_ * jy + pz_ * jz + pd_ * jd : px_ * jx + py_ * jy + pd_ * jd;
  }

  // The delta and zeta entries of column c after the change, from P1's entry dP and the old zeta
  // and delta entries; returns the new delta entry.
  __device__ __forceinline__ double rows(Jac &J, int c, double dP, double jz, double jd) const {
    const double jdn = dd_dP * dP;
    J[DELTA][c] = jdn;
    J[ZETA][c] = rr * jz + zr * drvv_dP * dP - zr * rr * rv1 * jd;
    return jdn;
  }
};

// The chain of an energy change, plus the px, py rows of a kick applied before it (kx*, ky*:
// gradients of the px and py increments over x, y, zeta, delta).  Old rows are read before any
// row is written.
__device__ __forceinline__ void jac_energy(Jac &J, const EnergyChain &e, const double (&kx)[4],
                                           const double (&ky)[4]) {
#pragma unroll
  for (int c = 0; c < 6; ++c) {
    const double jx = J[X][c], jy = J[Y][c], jz = J[ZETA][c], jd = J[DELTA][c];
    const double dP = e.dP<true>(jx, jy, jz, jd);
    J[PX][c] += kx[0] * jx + kx[1] * jy + kx[2] * jz + kx[3] * jd;
    J[PY][c] += ky[0] * jx + ky[1] * jy + ky[2] * jz + ky[3] * jd;
    e.rows(J, c, dP, jz, jd);
  }
}

// CAVITY / SAWTOOTH_CAVITY (el_cavity; xline/elements.py:239-263).
// J and the state (the tracker's el_cavity with sincos_ns for sin).
template <int MODE>
__device__ __forceinline__ void tan_cavity(Jac &J, const KArgs &a, Regs<1> &r, const double2 *rec,
                                           double V, bool sawtooth) {
  const double2 c = rec[1];  // k, lag_rad
  const double tau = r.zeta[0] / r.rvv[0] / a.beta0;
  const double phase = c.y - c.x * tau;
  const double C = charge_ratio_of<1>(a, r, 0) * a.q0 * V;
  double w, dw;
  if (!sawtooth) {
    sincos_ns(phase, w, dw);
  } else {
    const double pi = 3.141592653589793;
    double m = fmod(phase + pi, 2 * pi);
    if (m < 0) m += 2 * pi;
    w = m - pi;
    dw = 1.0;
  }
  // d phase / d zeta = -k / (rvv beta0);  d phase / d delta = k zeta rvv' / (rvv^2 beta0)
  const double rv1 = drvv_ddelta(a.beta0, r.delta[0], r.rvv[0]);
  const double gz = C * dw * (-c.x / (r.rvv[0] * a.beta0));
  const double gd = C * dw * (c.x * r.zeta[0] * rv1 / (r.rvv[0] * r.rvv[0] * a.beta0));
  const double none[4] = {0.0, 0.0, 0.0, 0.0};
  const EnergyChain e(r, a.beta0, a.energy0, C * w, 0.0, 0.0, gz, gd);
  TAN_ROWS(jac_energy(J, e, none, none));
  add_to_energy(C * w, a.beta0, a.energy0, r.delta[0], r.rpp[0], r.rvv[0], r.zeta[0]);
}

// RFMULTIPOLE (el_rfmultipole; xline/elements.py:182-227).  With Z_i = z^i / i!, z = x + i y,
// cn_i = cos(pn_i - ktau), sn_i = sin(pn_i - ktau), cs_i, ss_i the same with ps_i:
//   dpx + i dpy = Q = sum A_i Z_i,   A_i = cn_i kn_i + i cs_i ks_i,
//   dptr = Re sum B_i Z_(i+1),       B_i = sn_i kn_i + i ss_i ks_i,
// dZ_i/dx = Z_(i-1), dZ_i/dy = i Z_(i-1), dA_i/dktau = B_i, dB_i/dktau = -A_i.
// J and the state (the tracker's el_rfmultipole with sincos_ns for sincos).
template <int MODE>
__device__ __forceinline__ void tan_rfmultipole(Jac &J, const KArgs &a, Regs<1> &r, const double2 *rec,
                                                int order, double V) {
  const double2 c = rec[1];  // k, lag_rad
  const double x = r.x[0], y = r.y[0], chi = r.chi[0];
  const double ktau = c.x * (r.zeta[0] / r.rvv[0] / a.beta0);
  double zr = 1.0, zi = 0.0;      // Z_i
  double pzr = 0.0, pzi = 0.0;    // Z_(i-1)
  double qr = 0.0, qi = 0.0;      // dQ/dz = sum A_i Z_(i-1)
  double br = 0.0, bi = 0.0;      // sum B_i Z_i = dQ/dktau, and d dptr/dx + i (-d dptr/dy)
  double ar = 0.0;                // Re sum A_i Z_(i+1) = -d dptr/dktau
  double dptr = 0.0, dpx = 0.0, dpy = 0.0;
  for (int ii = 0; ii <= order; ++ii) {
    const double2 kk = rec[2 + 2 * ii], ph = rec[3 + 2 * ii];
    double sn, cn, ss, cs;
    sincos_ns(ph.x - ktau, sn, cn);
    sincos_ns(ph.y - ktau, ss, cs);
    dpx = dpx + (cn * kk.x * zr - cs * kk.y * zi);
    dpy = dpy + (cs * kk.y * zr + cn * kk.x * zi);
    const double Ar = cn * kk.x, Ai = cs * kk.y, Br = sn * kk.x, Bi = ss * kk.y;
    if (ii > 0) {
      qr += Ar * pzr - Ai * pzi;
      qi += Ar * pzi + Ai * pzr;
    }
    br += Br * zr - Bi * zi;
    bi += Br * zi + Bi * zr;
    const double inv = static_cast<double>(ii + 1);
    const double nzr = (zr * x - zi * y) / inv, nzi = (zi * x + zr * y) / inv;
    ar += Ar * nzr - Ai * nzi;
    dptr += Br * nzr - Bi * nzi;
    pzr = zr;
    pzi = zi;
    zr = nzr;
    zi = nzi;
  }
  const double rv1 = drvv_ddelta(a.beta0, r.delta[0], r.rvv[0]);
  const double kz = c.x / (r.rvv[0] * a.beta0);                                // d ktau / d zeta
  const double kd = -c.x * r.zeta[0] * rv1 / (r.rvv[0] * r.rvv[0] * a.beta0);  // d ktau / d delta
  // px -= chi Re Q, py += chi Im Q: gradients over (x, y, zeta, delta)
  const double kxv[4] = {-chi * qr, chi * qi, -chi * br * kz, -chi * br * kd};
  const double kyv[4] = {chi * qi, chi * qr, chi * bi * kz, chi * bi * kd};
  const double C = charge_ratio_of<1>(a, r, 0) * a.q0;
  double sl, cl;
  sincos_ns(c.y - ktau, sl, cl);
  const double W = C * (V * sl - a.p0c * c.x * dptr);
  const double dW_dktau = C * (-V * cl + a.p0c * c.x * ar);
  const double gx = -C * a.p0c * c.x * br, gy = C * a.p0c * c.x * bi;
  const EnergyChain e(r, a.beta0, a.energy0, W, gx, gy, dW_dktau * kz, dW_dktau * kd);
  TAN_ROWS(jac_energy(J, e, kxv, kyv));
  r.px[0] = fma(-chi, dpx, r.px[0]);
  r.py[0] = fma(chi, dpy, r.py[0]);
  add_to_energy(W, a.beta0, a.energy0, r.delta[0], r.rpp[0], r.rvv[0], r.zeta[0]);
}

// Field of a frozen Gaussian (field_fixed, fast encoding) and its derivatives over (x, y).
// Round: E = temp(r2) (x, y).  Elliptic (Bassetti-Erskine, first quadrant u along the big axis):
// F = w(z1) - e w(z2), with w'(z) = -2 z w(z) + 2i/sqrt(pi).
__device__ __forceinline__ void field_jac(const double2 *blk, double x, double y, double &Ex, double &Ey,
                                          double &exx, double &exy, double &eyx, double &eyy) {
  const double2 s = blk[0];
  const long long kind = reinterpret_cast<const long long *>(blk)[2];
  if (kind == 0) {
    const double sigma = 0.5 * (s.x + s.y), A = blk[2].x;
    const double r2 = x * x + y * y;
    if (r2 < 1e-20) {
      // the tracker's linearised branch is singular in its derivative at the origin; the field's
      // own derivative there is A / (2 sigma^2)
      const double temp = sqrt(r2) * A / sigma;
      Ex = temp * x;
      Ey = temp * y;
      exx = eyy = A / (2.0 * sigma * sigma);
      exy = eyx = 0.0;
    } else {
      const double q = 0.5 * r2 / (sigma * sigma);
      const double om = -expm1(-q);  // 1 - e^-q
      const double temp = om * A / r2;
      const double dtemp = A * ((1.0 - om) * 0.5 / (sigma * sigma) - om / r2) / r2;  // d temp / d r2
      Ex = temp * x;
      Ey = temp * y;
      exx = temp + 2.0 * x * x * dtemp;
      eyy = temp + 2.0 * y * y * dtemp;
      exy = eyx = 2.0 * x * y * dtemp;
    }
    return;
  }
  const bool wide = kind == 1;
  const double2 c3 = blk[3], c4 = blk[4], c5 = blk[5];  // [1/S, fact] [small/big, big/small] [hb, hs]
  const double abx = fabs(x), aby = fabs(y);
  const double u = wide ? abx : aby, v = wide ? aby : abx;
  const double us = u * c3.x, vs = v * c3.x;
  const double zx[2] = {us, c4.x * us}, zy[2] = {vs, c4.y * vs};
  double wr[2], wi[2];
  bf::wofz_multi_q1<2>(zx, zy, wr, wi);
  const double e = exp(-fma(u * u, c5.x, v * v * c5.y));
  const double tsp = 1.1283791670955126;  // 2 / sqrt(pi)
  // w' at z1 and z2
  const double d1r = -2.0 * (zx[0] * wr[0] - zy[0] * wi[0]), d1i = -2.0 * (zx[0] * wi[0] + zy[0] * wr[0]) + tsp;
  const double d2r = -2.0 * (zx[1] * wr[1] - zy[1] * wi[1]), d2i = -2.0 * (zx[1] * wi[1] + zy[1] * wr[1]) + tsp;
  const double deu = -2.0 * u * c5.x * e, dev = -2.0 * v * c5.y * e;
  // dF/du = w1' /S - e w2' (s/b)/S - w2 de/du ;  dF/dv = i w1' /S - e i w2' (b/s)/S - w2 de/dv
  const double fur = c3.x * d1r - e * c4.x * c3.x * d2r - wr[1] * deu;
  const double fui = c3.x * d1i - e * c4.x * c3.x * d2i - wi[1] * deu;
  const double fvr = -c3.x * d1i + e * c4.y * c3.x * d2i - wr[1] * dev;
  const double fvi = c3.x * d1r - e * c4.y * c3.x * d2r - wi[1] * dev;
  const double f_im = c3.y * (wi[0] - wi[1] * e), f_re = c3.y * (wr[0] - wr[1] * e);
  const double sxy = ((x < 0) != (y < 0)) ? -1.0 : 1.0;
  if (wide) {  // Ex = sgn(x) f_im(|x|, |y|), Ey = sgn(y) f_re
    Ex = x < 0 ? -f_im : f_im;
    Ey = y < 0 ? -f_re : f_re;
    exx = c3.y * fui;
    exy = sxy * c3.y * fvi;
    eyx = sxy * c3.y * fur;
    eyy = c3.y * fvr;
  } else {     // u = |y|, v = |x|: Ex = sgn(x) f_re, Ey = sgn(y) f_im
    Ex = x < 0 ? -f_re : f_re;
    Ey = y < 0 ? -f_im : f_im;
    exx = c3.y * fvr;
    exy = sxy * c3.y * fur;
    eyx = sxy * c3.y * fvi;
    eyy = c3.y * fui;
  }
}

// px += f Ex + ..., py += f Ey + ...: rows of a beam-field kick with factor f, whose gradient over
// (zeta, delta) is (fz, fd).
__device__ __forceinline__ void jac_field_kick(Jac &J, double f, double fz, double fd, double Ex, double Ey,
                                               double exx, double exy, double eyx, double eyy) {
#pragma unroll
  for (int c = 0; c < 6; ++c) {
    const double jx = J[X][c], jy = J[Y][c], jz = J[ZETA][c], jd = J[DELTA][c];
    J[PX][c] += f * (exx * jx + exy * jy) + Ex * (fz * jz + fd * jd);
    J[PY][c] += f * (eyx * jx + eyy * jy) + Ey * (fz * jz + fd * jd);
  }
}

// BEAMBEAM4D (bf::beambeam4d; be_beamfields/beambeam.py:45-82).
__device__ __forceinline__ void jac_beambeam4d(Jac &J, const KArgs &a, const Regs<1> &r, const double2 *rec) {
  const double2 off = rec[1], bc = rec[3 + XLB_FIELD_PAIRS];
  double Ex, Ey, exx, exy, eyx, eyy;
  field_jac(rec + 2, r.x[0] - off.x, r.y[0] - off.y, Ex, Ey, exx, exy, eyx, eyy);
  const double beta = a.beta0 / r.rvv[0];
  const double K = r.chi[0] * bc.y * (charge_ratio_of<1>(a, r, 0) * a.q0) / a.p0c;
  const double f = K * (1.0 + beta * bc.x) / (beta + bc.x);
  const double df_dbeta = K * (bc.x * bc.x - 1.0) / ((beta + bc.x) * (beta + bc.x));
  const double dbeta_dd = -a.beta0 * drvv_ddelta(a.beta0, r.delta[0], r.rvv[0]) / (r.rvv[0] * r.rvv[0]);
  jac_field_kick(J, f, 0.0, df_dbeta * dbeta_dd, Ex, Ey, exx, exy, eyx, eyy);
}

// SPACECHARGE, the four profile kinds (bf::spacecharge; be_beamfields/spacecharge.py).
__device__ __forceinline__ void jac_spacecharge(Jac &J, const KArgs &a, const Regs<1> &r, const double2 *rec,
                                                int kind) {
  const double2 co = rec[1];
  const double2 *tail = rec + 2 + XLB_FIELD_PAIRS;
  const double2 b = tail[0];
  const double *w = reinterpret_cast<const double *>(tail);
  const double zeta = r.zeta[0], rvv = r.rvv[0];
  double lam = 1.0, dlz = 0.0, dld = 0.0;  // lambda and its derivatives over zeta, delta
  if (kind == 1) {
    const double2 c8 = tail[1], c9 = tail[2];
    const long long gauss = reinterpret_cast<const long long *>(tail)[6];
    const double sg = zeta / rvv;
    const double arg = b.y * (sg * sg);
    double dl_darg;
    if (gauss) {
      lam = c8.x * exp(-arg);
      dl_darg = -lam;
    } else {
      double up = 1.0 + (-arg) * c8.y;
      if (up < 0) up = 0;
      lam = c8.x * pow(up, c9.x);
      dl_darg = up > 0 ? -c8.y * c9.x * c8.x * pow(up, c9.x - 1.0) : 0.0;
    }
    const double rv1 = drvv_ddelta(a.beta0, r.delta[0], rvv);
    dlz = dl_darg * 2.0 * b.y * sg / rvv;
    dld = dl_darg * 2.0 * b.y * sg * (-zeta * rv1 / (rvv * rvv));
  } else if (kind == 2 || kind == 3) {
    const double z0 = b.y, dz = w[2];
    const long long n = reinterpret_cast<const long long *>(tail)[4];
    long long i = static_cast<long long>(floor((zeta - z0) / dz));
    if (i < 0) i = 0;
    if (i > n - 2) i = n - 2;
    if (kind == 2) {
      const double *f = w + 6;
      if (zeta <= z0) {
        lam = f[0];
      } else if (zeta >= z0 + static_cast<double>(n - 1) * dz) {
        lam = f[n - 1];
      } else {
        const double xi = z0 + static_cast<double>(i) * dz;
        const double sl = (f[i + 1] - f[i]) / dz;
        lam = sl * (zeta - xi) + f[i];
        dlz = sl;
      }
    } else {
      const double *xk = w + 6;
      const double *c = xk + n;
      const double t = zeta - xk[i];
      const long long m = n - 1;
      lam = ((c[i] * t + c[m + i]) * t + c[2 * m + i]) * t + c[3 * m + i];
      dlz = (3.0 * c[i] * t + 2.0 * c[m + i]) * t + c[2 * m + i];
    }
  }
  double Ex, Ey, exx, exy, eyx, eyy;
  field_jac(rec + 2, r.x[0] - co.x, r.y[0] - co.y, Ex, Ey, exx, exy, eyx, eyy);
  const double g = r.chi[0] * charge_ratio_of<1>(a, r, 0) * a.sc_common * b.x;
  jac_field_kick(J, g * lam, g * dlz, g * dld, Ex, Ey, exx, exy, eyx, eyy);
}

// DRIFT / DRIFT_EXACT, and the drift fused into an aperture or space-charge record.
template <int MODE>
__device__ __forceinline__ void tan_drift(Jac &J, Regs<1> &r, double beta0, bool exact, double L) {
  if (exact) {
    TAN_ROWS(jac_drift_exact(J, r, beta0, L));
    el_drift_exact<1>(r, L);
  } else {
    TAN_ROWS(jac_drift(J, r, beta0, L));
    el_drift<1>(r, L);
  }
}

// The end of an aperture record (LIMIT_*; the inside-tests are the tracker's, run_chunk): the
// particle is lost unless `in`, with the s-word at cur[s_word] (apply_losses), then the record's
// fused drift of length L, if any.  J is unchanged by the test.
template <int MODE>
__device__ __forceinline__ void tan_limit(Jac &J, const KArgs &a, Regs<1> &r, const double2 *cur, int aux,
                                          bool in, int s_word, const double &L) {
  const bool lost[1] = {r.alive(0) && !in};
  apply_losses<1>(a, r, lost, cur, 1, s_word);
  if (aux & XLB_AUX_DRIFT) tan_drift<MODE>(J, r, a.beta0, aux & XLB_AUX_DRIFT_EXACT, L);
}

// ---------------------------------------------------------------- mean-mode radiation
// One radiating half of a MULTIPOLE_RAD record in mean mode (the tracker's radiate_half,
// track_impl.cuh, restated: that function lives behind XLB_RADIATION, which would bring the
// __constant__ photon table into this unit).  x and y do not change inside the element, so the
// field size fl and the path length lh of both halves are functions of the state before it; the
// caller passes fl^2's gradient (f2x, f2y) over (x, y).  With A = -(2/3) q0^2 K_e beta^3 gamma^4 / (L^2
// (1+delta)^2) the loss is W = A fl^2 lh, whose gradient is taken through fl^2 (smooth where fl = 0,
// unlike fl itself), and  d ln W / d delta = 1/(1+delta) + P p0c / E^2  (W ~ (1+delta) E).  Then
// add_to_energy(W) through EnergyChain, and px, py times f = (1+delta')/(1+delta):
//   row(px) <- f row(px) + px (row(delta') - f row(delta)) / (1+delta),  the same for py.
// ENVELOPE: Sigma += V_h g g^T with V_h = nbar (11/27) u_c^2, the variance of the quantum mode's
// loss over the half (nbar, u_c of include/xline_b200.h), and g = dz_after/dW; `eloss` -= W.
template <int MODE>
__device__ __forceinline__ void tan_radiate_half(Jac &J, const KArgs &a, Regs<1> &r, const double2 *rec,
                                                 double fl, double lh, double f2x, double f2y, double hxl,
                                                 double hyl, double &eloss) {
  const double2 len = rec[1], ke = rec[2], al = rec[3];  // [L,1/L][K_e,hbar_c][alpha,seed]
  const double m2 = (a.energy0 - a.p0c) * (a.energy0 + a.p0c);
  const double opd = 1.0 + r.delta[0];
  const double P = opd * a.p0c;
  const double E = sqrt(fma(P, P, m2));
  const double gamma = E / sqrt(m2);
  const double kappa = fl * len.y / opd;
  const double q2 = a.q0 * a.q0;
  if (kappa == 0.0) return;  // the particle untouched; fl = 0 makes fl^2's gradient 0 as well
  const double beta = P / E;
  const double g2 = gamma * gamma;
  const double dE = -(2.0 / 3.0) * q2 * ke.x * (beta * beta * beta) * (g2 * g2) * (kappa * kappa) * lh;
  // the gradient of dE over (x, y, delta)
  const double il = len.y / opd;
  const double A = -(2.0 / 3.0) * q2 * ke.x * (beta * beta * beta) * (g2 * g2) * (il * il);
  const double fl2 = fl * fl;
  const double gx = A * (f2x * lh + fl2 * (0.5 * hxl));
  const double gy = A * (f2y * lh - fl2 * (0.5 * hyl));
  const double gd = dE * (1.0 / opd + P * a.p0c / (E * E));
  // the chain of add_to_energy (no zeta gradient) with the scaling of px, py
  const EnergyChain e(r, a.beta0, a.energy0, dE, gx, gy, 0.0, gd);
  const double f = e.opdn / opd, xo = r.px[0] / opd, yo = r.py[0] / opd;
  TAN_ROWS(
      _Pragma("unroll")
      for (int c = 0; c < 6; ++c) {
        const double jx = J[X][c], jy = J[Y][c], jz = J[ZETA][c], jd = J[DELTA][c];
        const double jdn = e.rows(J, c, e.dP<false>(jx, jy, jz, jd), jz, jd);
        J[PX][c] = f * J[PX][c] + xo * (jdn - f * jd);
        J[PY][c] = f * J[PY][c] + yo * (jdn - f * jd);
      });
  if (MODE == ENVELOPE) {
    const double nbar = (5.0 / (2.0 * 1.7320508075688772)) * q2 * al.x * gamma * kappa * lh;
    const double uc = 1.5 * ke.y * (gamma * g2) * kappa;
    const double V = nbar * (11.0 / 27.0) * (uc * uc);
    const double gdw = e.dd_dP / a.energy0;
    const double g[6] = {0.0, xo * gdw, 0.0, yo * gdw, e.zr * e.drvv_dP / a.energy0, gdw};
#pragma unroll
    for (int q = 0; q < 6; ++q)
#pragma unroll
      for (int c = 0; c < 6; ++c) J[q][c] = fma(V * g[q], g[c], J[q][c]);
    eloss -= dE;
  }
  add_to_energy(dE, a.beta0, a.energy0, r.delta[0], r.rpp[0], r.rvv[0], r.zeta[0]);
  const double fs = (1.0 + r.delta[0]) / opd;
  r.px[0] = r.px[0] * fs;
  r.py[0] = r.py[0] * fs;
}

// MULTIPOLE_RAD in mean mode (el_multipole_rad): radiate, the embedded multipole, radiate.
template <int MODE>
__device__ __forceinline__ void tan_multipole_rad(Jac &J, const KArgs &a, Regs<1> &r, const double2 *rec,
                                                  int order, double &eloss) {
  const double2 len = rec[1];
  const double2 *sub = rec + 4;
  const bool curved = (*reinterpret_cast<const unsigned *>(sub) & 0xffu) == XLB_T_MULTIPOLE_CURVED;
  const double hxl = curved ? sub[0].y : 0.0;
  const double hyl = curved ? sub[1].x : 0.0;
  const double2 *pairs = curved ? sub + 3 : sub + 1;
  const double x = r.x[0], y = r.y[0];
  double dpx[1], dpy[1];
  horner<1>(r, pairs, order, dpx, dpy);  // the tracker's field kick, bit for bit
  double dr, di;
  horner_prime(pairs, order, x, y, dr, di);
  // fl^2 = (Re P)^2 + (Im P)^2:  d/dx = 2 (Re P Re P' + Im P Im P'),  d/dy = 2 (Im P Re P' - Re P Im P')
  const double f2x = 2.0 * (dpx[0] * dr + dpy[0] * di), f2y = 2.0 * (dpy[0] * dr - dpx[0] * di);
  const double fl = sqrt(fma(dpx[0], dpx[0], dpy[0] * dpy[0]));
  const double lh = 0.5 * fma(-hyl, y, fma(hxl, x, len.x));
  if (r.alive(0)) tan_radiate_half<MODE>(J, a, r, rec, fl, lh, f2x, f2y, hxl, hyl, eloss);
  if (curved) {
    const double2 c1 = sub[1], c2 = sub[2];  // [hyl, length] [1/length, 0]
    TAN_ROWS(jac_multipole(J, r, sub + 3, order, true, hxl, c1.x, c2.x));
    el_multipole_curved<1>(r, sub, order, hxl);
  } else {
    TAN_ROWS(jac_multipole(J, r, sub + 1, order, false, 0.0, 0.0, 0.0));
    el_multipole<1>(r, sub, order);
  }
  if (r.alive(0)) tan_radiate_half<MODE>(J, a, r, rec, fl, lh, f2x, f2y, hxl, hyl, eloss);
}

// One argument block for the three kernels; each uses the outputs of its mode.
struct TArgs {
  KArgs k;
  double *jac;            // [n][6][6]: J, or Sigma (ENVELOPE)
  long long *log2_scale;  // [n], TANGENT and TANGENT_R
  double *fli;            // [n], TANGENT and TANGENT_R
  double *energy_loss;    // [n], ENVELOPE
};

// J (or Sigma) of particle k (< n), and what the mode accumulates with it: the exponent and the
// FLI, or the energy lost (eV).  J's 36 words are addressed with k, the other arrays with int(k).
template <int MODE>
__device__ __forceinline__ void load(const TArgs &t, long long k, Jac &J, long long &l2s, double &fli, double &el) {
  const double *jin = t.jac + k * 36;
  const int i = static_cast<int>(k);
#pragma unroll
  for (int q = 0; q < 6; ++q)
#pragma unroll
    for (int c = 0; c < 6; ++c) J[q][c] = jin[q * 6 + c];
  if (MODE == ENVELOPE) {
    el = t.energy_loss[i];
  } else {
    l2s = t.log2_scale[i];
    fli = t.fli[i];
  }
}

template <int MODE>
__device__ __forceinline__ void store(const TArgs &t, int i, const Jac &J, long long l2s, double fli, double el) {
  double *o = t.jac + static_cast<long long>(i) * 36;
#pragma unroll
  for (int q = 0; q < 6; ++q)
#pragma unroll
    for (int c = 0; c < 6; ++c) o[q * 6 + c] = J[q][c];
  if (MODE == ENVELOPE) {
    t.energy_loss[i] = el;
  } else {
    t.log2_scale[i] = l2s;
    t.fli[i] = fli;
  }
}

// End of a turn: the exact overflow guard, then the FLI.
__device__ __forceinline__ void end_turn(Jac &J, long long &l2s, double &fli) {
  double m = 0.0;
#pragma unroll
  for (int q = 0; q < 6; ++q)
#pragma unroll
    for (int c = 0; c < 6; ++c) m = fmax(m, fabs(J[q][c]));
  if (!(m > 0.0) || !isfinite(m)) return;  // a NaN / inf J stays as it is
  int e = ilogb(m);
  if (m > 0x1p512) {
#pragma unroll
    for (int q = 0; q < 6; ++q)
#pragma unroll
      for (int c = 0; c < 6; ++c) J[q][c] = scalbn(J[q][c], -e);
    l2s += e;
    e = 0;
  }
  // ||J||_F = 2^e sqrt(sum (J 2^-e)^2), without overflow for any max|J| <= 2^512
  double ss = 0.0;
#pragma unroll
  for (int q = 0; q < 6; ++q)
#pragma unroll
    for (int c = 0; c < 6; ++c) {
      const double v = scalbn(J[q][c], -e);
      ss = fma(v, v, ss);
    }
  const double f = 0.5 * log10(ss) + static_cast<double>(l2s + e) * 0.30102999566398120;
  fli = fmax(fli, f);
}

// End of an envelope turn: Sigma made exactly symmetric (F(F(Sigma)^T) is symmetric up to rounding).
__device__ __forceinline__ void symmetrize(Jac &S) {
#pragma unroll
  for (int q = 0; q < 6; ++q)
#pragma unroll
    for (int c = q + 1; c < 6; ++c) S[q][c] = S[c][q] = 0.5 * (S[q][c] + S[c][q]);
}

template <int MODE>
__device__ __forceinline__ void tangent_body(const TArgs &t) {
  const KArgs &a = t.k;
  const long long k = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  Regs<1> r;
  Jac J;
  long long l2s = 0;
  double fli = 0.0;
  double el = 0.0;  // ENVELOPE: energy lost (eV)
  r.slot[0] = -1;
  if (k < a.n) {
    const int i = static_cast<int>(k);
    if (a.state[i] == 1) {
      r.slot[0] = i;
      r.x[0] = a.x[i];
      r.px[0] = a.px[i];
      r.y[0] = a.y[i];
      r.py[0] = a.py[i];
      r.zeta[0] = a.zeta[i];
      r.delta[0] = a.delta[i];
      r.rpp[0] = a.rpp[i];
      r.rvv[0] = a.rvv[i];
      r.chi[0] = a.chi ? a.chi[i] : 1.0;
      load<MODE>(t, k, J, l2s, fli, el);
    }
  }
  if (r.slot[0] < 0) {
    park<1>(r, 0);
    r.chi[0] = 1.0;
#pragma unroll
    for (int q = 0; q < 6; ++q)
#pragma unroll
      for (int c = 0; c < 6; ++c) J[q][c] = (q == c) ? 1.0 : 0.0;
  }
  r.s_acc = 0.0;
  r.turns_done = 0;
  const double2 *lat = reinterpret_cast<const double2 *>(a.lat);
  const int chunk_pairs = a.chunk_words >> 1;
  for (int turn = 0; turn < a.num_turns; ++turn) {
    if (!__any_sync(0xffffffffu, r.alive(0))) break;  // warp-uniform
    const double2 *rec = lat;
    int chunk = 0;
    for (;;) {
      const double2 *cur = rec;
      const unsigned lo = static_cast<unsigned>(hdr_of(cur[0]));
      const int tag = static_cast<int>(lo & 0xffu), aux = static_cast<int>((lo >> 8) & 0xffu);
      const double p0 = cur[0].y;
      rec += (lo >> 16) & 0x3fffu;
      const bool was_alive = r.alive(0);
      if (tag == XLB_T_END_CHUNK) {
        rec = lat + static_cast<long long>(++chunk) * chunk_pairs;
        continue;
      }
      if (tag == XLB_T_END_TURN) {
        r.s_acc += p0;
        break;
      }
      switch (tag) {
        case XLB_T_DRIFT:
          tan_drift<MODE>(J, r, a.beta0, false, p0);
          break;
        case XLB_T_DRIFT_EXACT:
          tan_drift<MODE>(J, r, a.beta0, true, p0);
          break;
        case XLB_T_MULTIPOLE:
          TAN_ROWS(jac_multipole(J, r, cur + 1, aux, false, 0.0, 0.0, 0.0));
          el_multipole<1>(r, cur, aux);
          break;
        case XLB_T_MULTIPOLE_CURVED: {
          const double2 c1 = cur[1], c2 = cur[2];  // [hyl, length] [1/length, 0]
          TAN_ROWS(jac_multipole(J, r, cur + 3, aux, true, p0, c1.x, c2.x));
          el_multipole_curved<1>(r, cur, aux, p0);
          break;
        }
        case XLB_T_CAVITY:
        case XLB_T_SAWTOOTH_CAVITY:
          tan_cavity<MODE>(J, a, r, cur, p0, tag == XLB_T_SAWTOOTH_CAVITY);
          break;
        case XLB_T_RFMULTIPOLE:
          tan_rfmultipole<MODE>(J, a, r, cur, aux, p0);
          break;
        case XLB_T_XYSHIFT:  // xline/elements.py:274-276: J unchanged
          r.x[0] = r.x[0] - p0;
          r.y[0] = r.y[0] - cur[1].x;
          break;
        case XLB_T_SROTATION: {  // xline/elements.py:379-390: the same rotation of the rows
          const double cz = p0, sz = cur[1].x;
          TAN_ROWS(
              _Pragma("unroll")
              for (int c = 0; c < 6; ++c) {
                const double jx = J[X][c], jy = J[Y][c], jpx = J[PX][c], jpy = J[PY][c];
                J[X][c] = fma(cz, jx, sz * jy);
                J[Y][c] = fma(-sz, jx, cz * jy);
                J[PX][c] = fma(cz, jpx, sz * jpy);
                J[PY][c] = fma(-sz, jpx, cz * jpy);
              });
          const double xn = fma(cz, r.x[0], sz * r.y[0]), yn = fma(-sz, r.x[0], cz * r.y[0]);
          const double pxn = fma(cz, r.px[0], sz * r.py[0]), pyn = fma(-sz, r.px[0], cz * r.py[0]);
          r.x[0] = xn;
          r.y[0] = yn;
          r.px[0] = pxn;
          r.py[0] = pyn;
          break;
        }
        case XLB_T_DIPOLE_EDGE: {  // xline/elements.py:538-548
          const double r43 = cur[1].x;
          TAN_ROWS(axpy(J, PX, p0, X); axpy(J, PY, r43, Y));
          r.px[0] = r.px[0] + p0 * r.x[0];
          r.py[0] = r.py[0] + r43 * r.y[0];
          break;
        }
        case XLB_T_LIMIT_RECT: {  // the tracker's tests (run_chunk); J unchanged
          const double2 c1 = cur[1], c2 = cur[2];
          bool in;
          if (aux & 1)
            in = (fabs(r.x[0]) <= c1.x) & (fabs(r.y[0]) <= c2.x);
          else
            in = (r.x[0] >= p0) & (r.x[0] <= c1.x) & (r.y[0] >= c1.y) & (r.y[0] <= c2.x);
          tan_limit<MODE>(J, a, r, cur, aux, in, 5, cur[3].x);
          break;
        }
        case XLB_T_LIMIT_ELLIPSE: {
          const double2 c1 = cur[1], c2 = cur[2];
          const double q = fma(r.x[0] * r.x[0], c1.y, (r.y[0] * r.y[0]) * c2.x);
          tan_limit<MODE>(J, a, r, cur, aux, q <= 1.0, 5, cur[3].x);
          break;
        }
        case XLB_T_LIMIT_RECT_ELLIPSE: {
          const double mx = p0;
          const double2 c1 = cur[1], c2 = cur[2], c3 = cur[3];
          const double q = fma(r.x[0] * r.x[0], c2.y, (r.y[0] * r.y[0]) * c3.x);
          const bool in = (r.x[0] >= -mx) & (r.x[0] <= mx) & (r.y[0] >= -c1.x) & (r.y[0] <= c1.x) & (q <= 1.0);
          tan_limit<MODE>(J, a, r, cur, aux, in, 7, cur[4].x);
          break;
        }
        case XLB_T_LIMIT_POLYGON: {
          const int n_edges = static_cast<int>(__double_as_longlong(p0));
          const double2 *e = cur + 2;
          bool odd = false;
          for (int q = 0; q < n_edges; ++q, e += 2) odd ^= polygon_edge_crossed(r.x[0], r.y[0], e[0], e[1]);
          tan_limit<MODE>(J, a, r, cur, aux, odd, 2, cur[1].y);
          break;
        }
        case XLB_T_BEAMBEAM4D:
          TAN_ROWS(jac_beambeam4d(J, a, r, cur));
          bf::beambeam4d<1>(a, r, cur);
          break;
        case XLB_T_SPACECHARGE:
          TAN_ROWS(jac_spacecharge(J, a, r, cur, aux & 0xf));
          bf::spacecharge<1>(a, r, cur, aux & 0xf);
          if (aux & XLB_AUX_DRIFT) tan_drift<MODE>(J, r, a.beta0, aux & XLB_AUX_DRIFT_EXACT, p0);
          break;
        default:  // XLB_T_MONITOR: the identity, nothing stored.  The host refuses every other tag.
          if (MODE != TANGENT && tag == XLB_T_MULTIPOLE_RAD) tan_multipole_rad<MODE>(J, a, r, cur, aux, el);
          break;
      }
      if (was_alive && !r.alive(0)) store<MODE>(t, static_cast<int>(k), J, l2s, fli, el);  // frozen where lost
    }
    if (r.alive(0)) {
      if (MODE == ENVELOPE)
        symmetrize(J);
      else
        end_turn(J, l2s, fli);
    }
    r.turns_done += a.count_turns;
  }
  if (r.alive(0)) {
    const int i = r.slot[0];
    a.x[i] = r.x[0];
    a.px[i] = r.px[0];
    a.y[i] = r.y[0];
    a.py[i] = r.py[0];
    a.zeta[i] = r.zeta[0];
    a.delta[i] = r.delta[0];
    a.rpp[i] = r.rpp[0];
    a.rvv[i] = r.rvv[0];
    a.s[i] = a.s[i] + r.s_acc;
    a.at_turn[i] = a.at_turn[i] + r.turns_done;
    a.at_element[i] = 0;
    store<MODE>(t, i, J, l2s, fli, el);
  }
}

__global__ void __launch_bounds__(256) tangent_kernel(const __grid_constant__ TArgs t) { tangent_body<TANGENT>(t); }

__global__ void __launch_bounds__(256) tangent_kernel_radiation(const __grid_constant__ TArgs t) {
  tangent_body<TANGENT_R>(t);
}

__global__ void __launch_bounds__(256) envelope_kernel(const __grid_constant__ TArgs t) { tangent_body<ENVELOPE>(t); }

}  // namespace tangent

cudaError_t tangent_launch(tangent::Mode mode, const KArgs &a, double *jac, long long *log2_scale, double *fli,
                           double *energy_loss, int threads, cudaStream_t st) {
  const tangent::TArgs t = {a, jac, log2_scale, fli, energy_loss};
  const unsigned blocks = static_cast<unsigned>((a.n + threads - 1) / threads);
  if (mode == tangent::ENVELOPE)
    tangent::envelope_kernel<<<blocks, threads, 0, st>>>(t);
  else if (mode == tangent::TANGENT_R)
    tangent::tangent_kernel_radiation<<<blocks, threads, 0, st>>>(t);
  else
    tangent::tangent_kernel<<<blocks, threads, 0, st>>>(t);
  return cudaGetLastError();
}

}  // namespace xlb
