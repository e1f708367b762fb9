// Result write-back of one finished problem, shared by every solve kernel (ascent_cabi.cu) and the host build of
// the sweeps (tools/hostsim).  The kernels differ only in how node k of the converged iterate is read: each Sweeps
// policy provides that read as SW::node().
#pragma once
#include "ascent_coop.cuh"

namespace lmato {

// The output arrays of a batch of B problems, in the layout of include/lmato_b200.h.  traj, kkt and sens may be null.
struct ResultOut {
  double* traj;          // [NVAR][nt][B]
  double* tf;
  double* fmass;
  int* status;
  int* iters;
  double* kkt;
  double* sens;          // [LMATO_NSENS][B] d tf / d parameter
  long B;
};

// Results of problem b (LO:178-202: tf, the per-node values of all ten variables, final mass, status).  ydoubledot,
// xdoubledot and mass, which the device formulation eliminates, are recomputed (LO:123, 127-136).  The problem's G
// lanes (lane mask `mask`) share the work: lane g writes the scalars if g == 0, the node-0 rows g, g+G, ... and the
// nodes 1+g, 1+g+G, ...  Out of line on the device: the kernels that call it already use all 255 registers.
template <class SW, int G, class WS>
LM_NOINLINE void write_results(const ResultOut& R, const Params& P, const Mesh& M, double obj_scale, int model,
                               const WS& W, int g, unsigned mask, const IpmState& S, long b) {
  SolveOut out;
  ipm_result(S, out);
  const int nt = M.N + 1;
  const long B = R.B;
  if (g == 0) {
    R.tf[b] = out.tf;
    R.fmass[b] = P.M0 - P.fuel * (P.mflow * P.T * out.tf);   // mass(nt-1) = mflow*T*tf (LO:123)
    R.status[b] = out.status;
    R.iters[b] = out.iters;
    if (R.kkt) R.kkt[b] = out.kkt;
  }
  if (!R.traj && !R.sens) return;
  double* __restrict__ t = R.traj;
  if (t) {
    for (int v = g; v < LMATO_NVAR; v += G) t[((long)v * nt) * B + b] = 0.0;   // node 0 pinned
  }
  // Parametric sensitivity of the optimum (envelope theorem): d objective* / d theta = d Lagrangian / d theta
  // = sum_k lambda_k . d c_k / d theta at the solution, with c_k = s_k - s_{k-1} - h_k T tf F(s_k, u_k; theta).
  // theta enters only the velocity rows (through the thrust acceleration Ft / (M0 - ms*mass), LO:127-136,
  // and mass = mflow*T*tau*tf, LO:123) and the angledot row (angle_scalar, LO:121).
  double s_ft = 0.0, s_m0 = 0.0, s_mf = 0.0, s_asc = 0.0;
  for (int k = 1 + g; k <= M.N; k += G) {
    double z[7];                                   // the six states and the control u = z[6]
    SW::node(W, out.cur, k, z, nullptr);
    const double u = z[6];
    const double m = P.mflow * P.T * M.tau[k] * out.tf;
    double ay, ax;
    if (R.sens) {
      Accel1 f;
      accel_first(P, z[0], z[2], z[4], m, f);
      ay = f.ay; ax = f.ax;
      const double al = M.h[k] * P.T * out.tf;
      // the multipliers are read here and not with z: held across accel_first they spill in the thread kernel
      double lam[3];
      SW::node(W, out.cur, k, nullptr, lam);
      const double l1 = lam[0], l3 = lam[1], l5 = lam[2];                    // ydot, xdot and angledot rows
      const double thrust = l1 * (f.AT * f.Ty * P.Sinv) + l3 * (f.AT * f.Tx * P.Sinv);
      s_ft -= al * thrust / P.Ft;
      s_m0 += al * thrust * (f.AT / P.Ft);                                  // d AT / d M0 = -AT / (M0 - ms*mass)
      s_mf -= al * (l1 * f.ay_m + l3 * f.ax_m) * (P.T * M.tau[k] * out.tf);
      s_asc -= al * u * l5;
    } else {
      accel_value(P, z[0], z[2], z[4], m, ay, ax);
    }
    if (!t) continue;
    t[((long)LMATO_V_Y * nt + k) * B + b] = z[0];
    t[((long)LMATO_V_YDOT * nt + k) * B + b] = z[1];
    t[((long)LMATO_V_YDOUBLEDOT * nt + k) * B + b] = ay;
    t[((long)LMATO_V_X * nt + k) * B + b] = z[2];
    t[((long)LMATO_V_XDOT * nt + k) * B + b] = z[3];
    t[((long)LMATO_V_XDOUBLEDOT * nt + k) * B + b] = ax;
    t[((long)LMATO_V_ANGLE * nt + k) * B + b] = z[4];
    t[((long)LMATO_V_ANGLEDOT * nt + k) * B + b] = z[5];
    t[((long)LMATO_V_MASS * nt + k) * B + b] = m;
    t[((long)LMATO_V_ANGLEDOUBLEDOT * nt + k) * B + b] = u;
  }
  if (R.sens) {
    s_ft = coop::Grp<G>::sum(mask, s_ft); s_m0 = coop::Grp<G>::sum(mask, s_m0);
    s_mf = coop::Grp<G>::sum(mask, s_mf); s_asc = coop::Grp<G>::sum(mask, s_asc);
    // the mass bound 0 <= mass <= 1 (LO:83) is carried as tf <= tf_ub = 1 / (mflow T): where that is the binding
    // upper bound on tf, its multiplier contributes  -zUt * d tf_ub / d mflow = zUt / (mflow^2 T)
    if (P.tf_ub < 1.0) s_mf += S.cur.zUt / (P.mflow * P.mflow * P.T);
    if (g == 0) {
      // per unit of the RAW parameters of include/lmato_b200.h: M_dot = mflow * fuel_mass (LO:65),
      // angle_doubledot_max = 3 * angle_scalar (LO:109); tf in the reference's scaled units (0..1)
      const double inv = 1.0 / obj_scale;
      R.sens[(long)LMATO_S_FT * B + b] = s_ft * inv;
      R.sens[(long)LMATO_S_M0 * B + b] = s_m0 * inv;
      R.sens[(long)LMATO_S_M_DOT * B + b] = s_mf * inv / P.fuel;
      // the circular model has no pitch-acceleration limit (its MV is the angle): no such derivative exists there
      R.sens[(long)LMATO_S_ANGLE_DOUBLEDOT_MAX * B + b] = model == LMATO_MODEL_CIRCULAR ? NAN : s_asc * inv / 3.0;
    }
  }
}

}  // namespace lmato
