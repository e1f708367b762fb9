// Ascent dynamics, hand-derived first and second derivatives (FP64).
//
// Reference equations (LO:n = /root/reference/Launch_Optimiser.py line n):
//   differential rows  LO:114-123, algebraic accelerations LO:127-136,
//   terminal rows LO:161, 169, 173.  The circular variant (PDF p.27 src 76-96) uses the
//   same acceleration expressions with the pitch angle as the manipulated variable.
//
// Formulation used on the device (equivalent NLP, see DESIGN.md "Transcription"):
//   * ydoubledot / xdoubledot are substituted into the velocity rows (they are explicit
//     functions of y, x, angle, mass);
//   * mass obeys mass' = mflow*T*tf with mass(0)=0 (LO:123, LO:151), hence
//     mass_k = mflow*T*tf*tau_k exactly under any collocation scheme that is exact for
//     constants -- it is eliminated and re-materialised on output;
//   * tf (one global FV, LO:39) is carried as a stage state so that the KKT system is
//     block tridiagonal with no dense border.
//
// This header is compiled by nvcc for the product.  It is also compilable by g++ for
// tools/hostsim (a developer-only debugging harness, never loaded by the package).
#pragma once
#include <math.h>

#include "../../include/lmato_b200.h"

#if defined(__CUDACC__)
#define LM_HD __host__ __device__ __forceinline__
#define LM_D __device__ __forceinline__
#define LM_NOINLINE __host__ __device__ __noinline__
// The three sweeps have one call site each and are inlined into the kernel: as ABI functions every
// global access paid two R2UR moves for its memory descriptor and scalar arguments travelled through
// the local-memory stack.
#ifndef LM_SWEEP
#define LM_SWEEP __host__ __device__ __forceinline__
#endif
#else
#define LM_HD inline
#define LM_D inline
#define LM_NOINLINE
#define LM_SWEEP inline
#endif

namespace lmato {

// Per-problem derived constants (LO:50-75, 107-109).
struct Params {
  double GM;      // G*M                         LO:50-51
  double R0;      // lunar radius                LO:52
  double Ft;      // thrust                      LO:61
  double M0;      // wet mass                    LO:62
  double S;       // distance scale = r_periapsis LO:73,107
  double ms;      // mass scale in dynamics      LO:108 (2576 in the PDF original)
  double mflow;   // M_dot / fuel_mass           LO:65
  double asc;     // angle_doubledot_max / 3     LO:109
  double T;       // final_time                  LO:38
  double a_ub;    // angle upper bound           LO:94
  double u_ub;    // |angledoubledot| bound      LO:96
  double vt2;     // (periapsis_v / S)^2         LO:75,169
  double rt;      // (R0 + S) / S                LO:161
  double R0S;     // R0 / S                      LO:161
  double tf_ub;   // min(1, 1/(mflow*T)): tf<=1 (LO:39) and mass<=1 (LO:83) at the last node
  double fuel;    // fuel_mass (for final-mass output)
  double Sinv;    // 1 / S
  // Model switch.  coup5 = 1: Launch_Optimiser.py (angledot_k - angledot_{k-1} = beta*u_k, LO:121).
  // coup5 = 0: the circular "IB-document" model (PDF p.27 src 69-73), where the pitch angle itself
  // is the MV: the angledot row loses its link to the previous node (angledot_k = beta*u_k with u
  // unbounded), which makes angle_k = angle_{k-1} + alpha*angledot_k a free variable per step.
  // coup5 = 0 AND asc = 0: the circular model WITH its move-suppression term (PDF p.27 src 69-73: DCOST on the
  // MV `angle`), cooperative kernel only: the MV slot of the 8-state formulation IS the pitch angle
  // (angle_k - u_k = 0 instead of angle_k - angle_{k-1} - alpha*angledot_k = 0, angledot pinned at 0), so that the
  // slack pair of the move u_k - u_{k-1} carries |angle_k - angle_{k-1}|.  See mv_is_angle().
  double coup5;
  double mT;      // mflow * T: mass(tau) = mT * tau * tf (LO:123); read per stage, kept here so that it is a
                  // shared-memory load and not a spilled register
};

// Params of problem b from the raw parameter block [LMATO_NPARAM][B] of include/lmato_b200.h.  move: the circular
// model with its move-suppression term (see coup5 above).
LM_HD Params derive_params(const double* __restrict__ p, long B, long b, int model, bool move = false) {
  // LO:50-75, 107-109
  Params P;
  const double G = p[LMATO_P_G * B + b], Mm = p[LMATO_P_M * B + b];
  const double R0 = p[LMATO_P_R0 * B + b];
  const double fuel = p[LMATO_P_FUEL_MASS * B + b];
  const double rp = p[LMATO_P_R_PERIAPSIS * B + b], ra = p[LMATO_P_R_APOAPSIS * B + b];
  P.GM = G * Mm;
  P.R0 = R0;
  P.Ft = p[LMATO_P_FT * B + b];
  P.M0 = p[LMATO_P_M0 * B + b];
  P.S = rp;
  P.ms = p[LMATO_P_MASS_SCALAR * B + b];
  P.mflow = p[LMATO_P_M_DOT * B + b] / fuel;
  P.asc = p[LMATO_P_ANGLE_DOUBLEDOT_MAX * B + b] / 3.0;
  P.T = p[LMATO_P_FINAL_TIME * B + b];
  P.a_ub = p[LMATO_P_ANGLE_UB * B + b];
  P.u_ub = p[LMATO_P_U_BOUND * B + b];
  const double vt = sqrt(P.GM / (R0 + 0.5 * (rp + ra)));
  P.vt2 = (vt / P.S) * (vt / P.S);
  P.rt = (R0 + P.S) / P.S;
  P.R0S = R0 / P.S;
  P.tf_ub = fmin(1.0, 1.0 / (P.mflow * P.T));
  P.fuel = fuel;
  P.Sinv = 1.0 / P.S;
  P.coup5 = 1.0;
  P.mT = P.mflow * P.T;
  if (model == LMATO_MODEL_CIRCULAR) {
    // PDF p.27 src 69-73: the MV is the pitch angle itself; no rate or acceleration limit exists
    P.coup5 = 0.0;
    P.asc = move ? 0.0 : 1.0;     // with the move term the MV slot holds the pitch angle itself (mv_is_angle())
    P.u_ub = 1e20;
  }
  return P;
}

// Partial derivatives of a function of Params (the Lagrangian of the NLP, ascent_result.cuh) with respect to the
// fields it reads.  S is the distance scale where the dynamics read it (X = x*S, Y = y*S + R0, Sinv = 1/S); the
// terminal rows read R0S, rt and vt2 instead.  mT = mflow*T and tf_ub = min(1, 1/(mflow*T)) depend on mflow and T
// alone, so their partials are carried in mflow and T (mflow: through the mass mT*tau*tf and tf_ub; T: through the
// step h*T*tf, the mass and tf_ub).
struct ParamsGrad {
  double GM, R0, Ft, M0, S, ms, mflow, asc, T, a_ub, u_ub, vt2, rt, R0S;
};

// The chain rule through derive_params: out[r * ostride] = d / d p[r] for every row r of problem b's raw parameter
// column, given g = the partials with respect to the derived fields.  The circular model does not read
// angle_doubledot_max and u_bound (derive_params overrides asc and u_ub): those two rows are NaN.
LM_HD void derive_params_grad(const double* __restrict__ p, long B, long b, int model, const ParamsGrad& g,
                              double* __restrict__ out, long ostride) {
  const double G = p[LMATO_P_G * B + b], Mm = p[LMATO_P_M * B + b];
  const double R0 = p[LMATO_P_R0 * B + b];
  const double fuel = p[LMATO_P_FUEL_MASS * B + b];
  const double rp = p[LMATO_P_R_PERIAPSIS * B + b], ra = p[LMATO_P_R_APOAPSIS * B + b];
  const double GM = G * Mm;
  const double D = R0 + 0.5 * (rp + ra);
  const double vt2 = GM / D / (rp * rp);                  // vt2 = GM / (D S^2), D = R0 + (rp + ra)/2, S = rp
  const double gGM = g.GM + g.vt2 * vt2 / GM;             // GM = G*M
  const double gD = -g.vt2 * vt2 / D;                     // d vt2 / d D = -vt2 / D
  const double gR0S = g.rt + g.R0S;                       // rt = R0S + 1, R0S = R0 / S
  const bool circ = model == LMATO_MODEL_CIRCULAR;
  out[LMATO_P_G * ostride] = gGM * Mm;
  out[LMATO_P_M * ostride] = gGM * G;
  out[LMATO_P_R0 * ostride] = g.R0 + gR0S / rp + gD;
  out[LMATO_P_FT * ostride] = g.Ft;
  out[LMATO_P_M0 * ostride] = g.M0;
  out[LMATO_P_M_DOT * ostride] = g.mflow / fuel;                                     // mflow = M_dot / fuel_mass
  out[LMATO_P_FUEL_MASS * ostride] = -g.mflow * (p[LMATO_P_M_DOT * B + b] / fuel) / fuel;
  out[LMATO_P_ANGLE_DOUBLEDOT_MAX * ostride] = circ ? NAN : g.asc / 3.0;           // asc = angle_doubledot_max / 3
  out[LMATO_P_R_PERIAPSIS * ostride] = g.S - gR0S * R0 / (rp * rp) + gD * 0.5 - 2.0 * g.vt2 * vt2 / rp;
  out[LMATO_P_R_APOAPSIS * ostride] = gD * 0.5;
  out[LMATO_P_FINAL_TIME * ostride] = g.T;
  out[LMATO_P_MASS_SCALAR * ostride] = g.ms;
  out[LMATO_P_ANGLE_UB * ostride] = g.a_ub;
  out[LMATO_P_U_BOUND * ostride] = circ ? NAN : g.u_ub;
}

// 1 in the circular model with the move term (the MV slot holds the pitch angle), else 0
LM_HD double mv_is_angle(const Params& P) { return (P.coup5 == 0.0 && P.asc == 0.0) ? 1.0 : 0.0; }

// ---------------------------------------------------------------------------------------
// Branch-free FP64 math for the inner loops.  Every argument in the sweeps is a normal, positive,
// bounded number (slacks, radii, masses) or an angle in [0, pi], so the library routines'
// special-case branches (denormals, infinities, huge-argument reduction) are dead weight: they
// split every stage body into dozens of small basic blocks (one BSSY/BSYNC pair per rcp / rsqrt /
// sincos), which starves the two warps per scheduler of instruction-level parallelism.  These
// versions are straight-line code: hardware seed (MUFU) + Newton, or fdlibm's kernels.
//
// The polynomial coefficients of lm_sincos_small (k_sin.c, k_cos.c) and lm_log_pos (e_log.c) are
// those of fdlibm, the Freely Distributable LIBM -- third-party, not from the reference repository.
// Its notice, preserved as its licence asks:
//   ====================================================
//   Copyright (C) 1993 by Sun Microsystems, Inc. All rights reserved.
//
//   Developed at SunSoft, a Sun Microsystems, Inc. business.
//   Permission to use, copy, modify, and distribute this
//   software is freely granted, provided that this notice
//   is preserved.
//   ====================================================
// ---------------------------------------------------------------------------------------
LM_HD double lm_rcp(double x) {
#if defined(__CUDA_ARCH__)
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  // seed error <= 2^-23, squared by every Newton step: two steps reach the FP64 rounding level
  // (measured against 1/x over 2^18 arguments: 1.1e-16, the same as with three)
  double e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  e = fma(-x, r, 1.0);
  return fma(r, e, r);
#else
  return 1.0 / x;
#endif
}

LM_HD double lm_rsqrt(double x) {
#if defined(__CUDA_ARCH__)
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  const double h = 0.5 * x;
  double e = fma(-h * y, y, 0.5);
  y = fma(y, e, y);
  e = fma(-h * y, y, 0.5);
  return fma(y, e, y);
#else
  return 1.0 / sqrt(x);
#endif
}

// sin and cos for |a| <= ~3.5 (here: 3*angle in [0, pi]).  Quadrant reduction with a two-term
// Cody-Waite split of pi/2, then the fdlibm kernels on [-pi/4, pi/4] (error < 1 ulp each).
LM_HD void lm_sincos_small(double a, double* sn, double* cs) {
#if defined(__CUDA_ARCH__)
  const double kq = rint(a * 0.63661977236758138);          // a * 2/pi
  double r = fma(-kq, 1.5707963267948966, a);               // pi/2 hi
  r = fma(-kq, 6.123233995736766e-17, r);                   // pi/2 lo
  const double z = r * r;
  // sin kernel
  double ps = fma(z, 1.58969099521155010221e-10, -2.50507602534068634195e-08);
  ps = fma(ps, z, 2.75573137070700676789e-06);
  ps = fma(ps, z, -1.98412698298579493134e-04);
  ps = fma(ps, z, 8.33333333332248946124e-03);
  ps = fma(ps, z, -1.66666666666666324348e-01);
  const double s = fma(r * z, ps, r);
  // cos kernel
  double pc = fma(z, -1.13596475577881948265e-11, 2.08757232129817482790e-09);
  pc = fma(pc, z, -2.75573143513906633035e-07);
  pc = fma(pc, z, 2.48015872894767294178e-05);
  pc = fma(pc, z, -1.38888888888741095749e-03);
  pc = fma(pc, z, 4.16666666666666019037e-02);
  const double c = fma(z * z, pc, fma(-0.5, z, 1.0));
  const int q = (int)kq & 3;
  const double s1 = (q & 1) ? c : s;
  const double c1 = (q & 1) ? s : c;
  *sn = (q & 2) ? -s1 : s1;
  *cs = ((q + 1) & 2) ? -c1 : c1;
#else
  *sn = sin(a);
  *cs = cos(a);
#endif
}

// Natural logarithm of a positive normal double (fdlibm e_log.c core, straight-line).
LM_HD double lm_log_pos(double x) {
#if defined(__CUDA_ARCH__)
  int hx = __double2hiint(x);
  const int lx = __double2loint(x);
  int k = (hx >> 20) - 1023;
  hx &= 0x000fffff;
  const int i = (hx + 0x95f64) & 0x100000;                  // mantissa >= sqrt(2): halve it
  const double m = __hiloint2double(hx | (i ^ 0x3ff00000), lx);
  k += (i >> 20);
  const double f = m - 1.0;
  const double sden = lm_rcp(2.0 + f);
  const double s = f * sden;
  const double dk = (double)k;
  const double z = s * s;
  const double w = z * z;
  double t1 = fma(w, 1.531383769920937332e-01, 2.222219843214978396e-01);   // Lg6, Lg4
  t1 = fma(t1, w, 3.999999999940941908e-01);                                 // Lg2
  t1 *= w;
  double t2 = fma(w, 1.479819860511658591e-01, 1.818357216161805012e-01);   // Lg7, Lg5
  t2 = fma(t2, w, 2.857142874366239149e-01);                                 // Lg3
  t2 = fma(t2, w, 6.666666666666735130e-01);                                 // Lg1
  const double R = fma(t2, z, t1);
  const double hfsq = 0.5 * f * f;
  // log(x) = k*ln2_hi - ((hfsq - (s*(hfsq+R) + k*ln2_lo)) - f)
  return fma(dk, 6.93147180369123816490e-01, -((hfsq - fma(s, hfsq + R, dk * 1.90821492927058770002e-10)) - f));
#else
  return log(x);
#endif
}

LM_HD void lm_sincos(double a, double* s, double* c) {
#if defined(__CUDA_ARCH__)
  sincos(a, s, c);
#else
  *s = sin(a);
  *c = cos(a);
#endif
}

// First-order quantities of the acceleration field at one node.
struct Accel1 {
  double ay, ax;                 // LO:127-136 (scaled: divided by S)
  double ay_y, ay_x, ay_a, ay_m; // d ay / d (y, x, angle, mass), scaled coordinates
  double ax_y, ax_x, ax_a, ax_m;
  // retained intermediates for the second-order pass
  double nx, ny, rinv, Tx, Ty, AT, eta, g3;
};

LM_HD void accel_first(const Params& P, double y, double x, double a, double m, Accel1& o) {
  const double X = x * P.S;
  const double Y = fma(y, P.S, P.R0);
  const double r2 = fma(X, X, Y * Y);
  const double rinv = lm_rsqrt(r2);
  const double nx = X * rinv, ny = Y * rinv;
  double s3, c3;
  lm_sincos_small(3.0 * a, &s3, &c3);
  const double Ty = fma(ny, c3, nx * s3);      // cos(psi - 3a)
  const double Tx = fma(nx, c3, -ny * s3);     // sin(psi - 3a)
  const double mden = lm_rcp(P.M0 - P.ms * m);
  const double AT = P.Ft * mden;               // thrust acceleration [m/s^2]
  const double eta = P.ms * mden;              // d ln(AT) / d mass
  const double g2 = P.GM * rinv * rinv;        // GM / r^2
  const double g3 = g2 * rinv;                 // GM / r^3
  const double Sinv = P.Sinv;
  o.ay = (AT * Ty - g2 * ny) * Sinv;
  o.ax = (AT * Tx - g2 * nx) * Sinv;
  const double ATr = AT * rinv;
  const double cross = 3.0 * g3 * nx * ny;
  o.ay_y = ATr * nx * Tx - g3 * (1.0 - 3.0 * ny * ny);
  o.ay_x = -ATr * ny * Tx + cross;
  o.ax_y = -ATr * nx * Ty + cross;
  o.ax_x = ATr * ny * Ty - g3 * (1.0 - 3.0 * nx * nx);
  o.ay_a = 3.0 * AT * Tx * Sinv;
  o.ax_a = -3.0 * AT * Ty * Sinv;
  o.ay_m = AT * eta * Ty * Sinv;
  o.ax_m = AT * eta * Tx * Sinv;
  o.nx = nx; o.ny = ny; o.rinv = rinv; o.Tx = Tx; o.Ty = Ty; o.AT = AT; o.eta = eta; o.g3 = g3;
}

// Acceleration values only (LO:127-136), used by the start-point roll-out and the output pass.
LM_HD void accel_value(const Params& P, double y, double x, double a, double m, double& ay, double& ax) {
  const double X = x * P.S;
  const double Y = fma(y, P.S, P.R0);
  const double r2 = fma(X, X, Y * Y);
  const double rinv = lm_rsqrt(r2);
  const double nx = X * rinv, ny = Y * rinv;
  double s3, c3;
  lm_sincos_small(3.0 * a, &s3, &c3);
  const double AT = P.Ft * lm_rcp(P.M0 - P.ms * m);
  const double g2 = P.GM * rinv * rinv;
  ay = (AT * fma(ny, c3, nx * s3) - g2 * ny) * P.Sinv;
  ax = (AT * fma(nx, c3, -ny * s3) - g2 * nx) * P.Sinv;
}

// Second derivatives of  Psi = l1*ay + l3*ax  w.r.t. (y, x, angle, mass), scaled coordinates.
struct Accel2 {
  double yy, yx, xx, ya, xa, aa, ym, xm, am, mm;
};

LM_HD void accel_second(const Params& P, const Accel1& f, double l1, double l3, Accel2& h) {
  const double nx = f.nx, ny = f.ny, ri = f.rinv;
  const double LT = fma(l1, f.Ty, l3 * f.Tx);    // lambda . thrust direction
  const double LP = fma(l1, f.Tx, -l3 * f.Ty);   // -dLT/dbeta
  // beta = psi - 3a ;  grad beta wrt (X, Y, a) = (ny/r, -nx/r, -3)
  const double bX = ny * ri, bY = -nx * ri;
  const double ri2 = ri * ri;
  // thrust part of S*Psi : AT * LT(beta)
  const double A = f.AT;
  const double pXX = -2.0 * nx * ny * ri2, pYY = -pXX, pXY = (nx * nx - ny * ny) * ri2;
  double HXX = A * (-LT * bX * bX - LP * pXX);
  double HYY = A * (-LT * bY * bY - LP * pYY);
  double HXY = A * (-LT * bX * bY - LP * pXY);
  const double HXa = A * (3.0 * LT * bX);
  const double HYa = A * (3.0 * LT * bY);
  const double Haa = A * (-9.0 * LT);
  // gravity part of S*Psi : -(GM)(l1*Y + l3*X)/r^3
  const double ln = fma(l3, nx, l1 * ny);
  const double k = 3.0 * f.g3 * ri;               // 3 GM / r^4
  HXX += k * (2.0 * l3 * nx + ln - 5.0 * ln * nx * nx);
  HYY += k * (2.0 * l1 * ny + ln - 5.0 * ln * ny * ny);
  HXY += k * (l3 * ny + l1 * nx - 5.0 * ln * nx * ny);
  const double S = P.S, Sinv = P.Sinv;
  h.yy = HYY * S; h.yx = HXY * S; h.xx = HXX * S;
  h.ya = HYa;     h.xa = HXa;     h.aa = Haa * Sinv;
  const double Ae = A * f.eta;
  h.ym = -Ae * LP * bY;
  h.xm = -Ae * LP * bX;
  h.am = 3.0 * Ae * LP * Sinv;
  h.mm = 2.0 * Ae * f.eta * LT * Sinv;
}

// Terminal constraint values and gradients at the last node (LO:161, 169, 173; the
// orthogonality row is divided by S^2, which leaves its zero set unchanged).
struct Terminal {
  double g1, g2, g3;     // radius - rt ; speed^2 - vt2 ; r.v / S^2
  double rT;             // scaled radius
  double Yb;             // y + R0/S
};

LM_HD void terminal_eval(const Params& P, double y, double vy, double x, double vx, Terminal& t) {
  t.Yb = y + P.R0S;
  t.rT = sqrt(fma(t.Yb, t.Yb, x * x));
  t.g1 = t.rT - P.rt;
  t.g2 = fma(vx, vx, vy * vy) - P.vt2;
  t.g3 = fma(t.Yb, vy, x * vx);
}

}  // namespace lmato
