// The flight of one solved problem: its control flown through the continuous ascent dynamics (LO:114-136).
//
// Every answer of the solver is the optimum of the TRANSCRIBED problem (backward Euler for NODES = 2, Lobatto
// collocation for NODES = 3..6).  This integrates the ODEs themselves with that control, so that a user sees where
// the vehicle really ends up: classical RK4 in normalised time tau with `substeps` equal sub-steps per mesh step,
// the MV of node k held on (tau_{k-1}, tau_k] as both transcriptions hold it (MV_TYPE = 0, LO:29), from the pinned
// zeros of node 0 (LO:145-151).  The accelerations are the solver's own (accel_value, LO:127-136); mass is linear in
// tau (LO:123) and taken exactly, mass(tau) = mflow*T*tf*tau, as the result writer re-materialises it.
//
// Compiled by nvcc (fly_control_kernel, ascent_cabi.cu) and by g++ (tools/hostsim, hostsim_fly).  No solve kernel
// includes it.
#pragma once
#include "ascent_model.cuh"

namespace lmato {

// Rows of the flight's summary [LMATO_NFLY][B] (include/lmato_b200.h).
enum FlyRow { FLY_Y = 0, FLY_YDOT, FLY_X, FLY_XDOT, FLY_ANGLE, FLY_ANGLEDOT, FLY_MASS, FLY_RADIUS_MISS,
              FLY_SPEED_MISS, FLY_FPA };
static_assert(FLY_FPA + 1 == LMATO_NFLY, "LMATO_NFLY rows");

// d/dtau of (y, ydot, x, xdot, angle, angledot) at normalised time tau under the held MV u.  c = T*tf.
// Elliptical model (LO:114-121): u is angledoubledot.  Circular model (PDF p.27 src 76-83): u is the pitch angle
// itself, so the angle rows do not move (s[4] holds u, s[5] stays 0).
LM_HD void fly_rhs(const Params& P, bool elliptical, double c, double tf, double tau, double u, const double s[6],
                   double d[6]) {
  double ay, ax;
  accel_value(P, s[0], s[2], s[4], P.mT * tf * tau, ay, ax);
  d[0] = c * s[1];
  d[1] = c * ay;
  d[2] = c * s[3];
  d[3] = c * ax;
  d[4] = elliptical ? c * s[5] : 0.0;
  d[5] = elliptical ? c * P.asc * u : 0.0;
}

// Flies problem b of a batch of B.  traj: the solve's output [LMATO_NVAR][nt][B], of which the MV row is read
// (angledoubledot, or angle for the circular model).  fin: [LMATO_NFLY][B].  out (or null): the flown trajectory in the
// same layout; node 0 is zero in every row, as the solve writes it, the acceleration rows are evaluated at the flown
// nodes, the MV row is copied from traj, and rows the model does not have (the circular model's angledot and
// angledoubledot) are zero.
LM_HD void fly_one(const Params& P, int model, const double* __restrict__ tau, int nt, const double* __restrict__ traj,
                   double tf, int substeps, long B, long b, double* __restrict__ fin, double* __restrict__ out) {
  const bool ell = model == LMATO_MODEL_ELLIPTICAL;
  const int mv_row = ell ? LMATO_V_ANGLEDOUBLEDOT : LMATO_V_ANGLE;
  const double c = P.T * tf;
  double s[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  if (out)
    for (int v = 0; v < LMATO_NVAR; ++v) out[((long)v * nt) * B + b] = 0.0;
  for (int k = 1; k < nt; ++k) {
    const double u = traj[((long)mv_row * nt + k) * B + b];
    if (!ell) s[4] = u;
    const double t0 = tau[k - 1], hk = tau[k] - t0;
    const double h = hk / substeps;
    for (int j = 0; j < substeps; ++j) {
      const double t = t0 + hk * j / substeps;
      double k1[6], k2[6], k3[6], k4[6], w[6];
      fly_rhs(P, ell, c, tf, t, u, s, k1);
      for (int i = 0; i < 6; ++i) w[i] = fma(0.5 * h, k1[i], s[i]);
      fly_rhs(P, ell, c, tf, t + 0.5 * h, u, w, k2);
      for (int i = 0; i < 6; ++i) w[i] = fma(0.5 * h, k2[i], s[i]);
      fly_rhs(P, ell, c, tf, t + 0.5 * h, u, w, k3);
      for (int i = 0; i < 6; ++i) w[i] = fma(h, k3[i], s[i]);
      fly_rhs(P, ell, c, tf, t + h, u, w, k4);
      for (int i = 0; i < 6; ++i) s[i] = fma(h / 6.0, (k1[i] + k4[i]) + 2.0 * (k2[i] + k3[i]), s[i]);
    }
    if (out) {
      const double m = P.mT * tf * tau[k];
      double ay, ax;
      accel_value(P, s[0], s[2], s[4], m, ay, ax);
      const double row[LMATO_NVAR] = {s[0], s[1], ay, s[2], s[3], ax, s[4], s[5], m, ell ? u : 0.0};
      for (int v = 0; v < LMATO_NVAR; ++v) out[((long)v * nt + k) * B + b] = row[v];
    }
  }
  // terminal quantities (LO:161, 169, 173) in SI
  Terminal T;
  terminal_eval(P, s[0], s[1], s[2], s[3], T);
  const double speed = sqrt(fma(s[3], s[3], s[1] * s[1]));
  const double f[LMATO_NFLY] = {s[0], s[1], s[2], s[3], s[4], s[5], P.mT * tf * tau[nt - 1], T.g1 * P.S,
                                (speed - sqrt(P.vt2)) * P.S, asin(T.g3 / (T.rT * speed))};
  for (int r = 0; r < LMATO_NFLY; ++r) fin[(long)r * B + b] = f[r];
}

}  // namespace lmato
