// Result write-back of one finished problem, shared by every solve kernel (ascent_cabi.cu) and the host build of
// the sweeps (tools/hostsim).  The kernels differ only in how node k of the converged iterate is read: each Sweeps
// policy provides that read as SW::node() (states, control, three multipliers) and SW::node_duals() (every multiplier
// the all-row sensitivity output needs).
#pragma once
#include "ascent_coop.cuh"

namespace lmato {

// The output arrays of a batch of B problems, in the layout of include/lmato_b200.h.  traj, kkt, sens and psens may be
// null.
struct ResultOut {
  double* traj;          // [NVAR][nt][B]
  double* tf;
  double* fmass;
  int* status;
  int* iters;
  double* kkt;
  double* sens;          // [LMATO_NSENS][B] d tf / d parameter
  long B;
  double* psens = nullptr;           // [LMATO_NPARAM][B] d tf / d params[p] for every row p
  const double* params = nullptr;    // [LMATO_NPARAM][B] the problems' raw parameters (read where psens is written)
};

// Sums of the sensitivity pass of write_results: d Lagrangian / d (Ft, M0, mflow, asc) for lmato_sens_t, and the other
// fields of ParamsGrad for the all-row output.
struct SensSums {
  double ft, m0, mf, asc;
  double gm, r0, sc, ms, t, aub, uub, vt2, rt, r0s;
};

// The terms of node k (state and control z, mass m, f = accel_first there) in the sums; the ParamsGrad fields other than
// the four of lmato_sens_t only if the all-row output is registered.
template <class SW, class WS>
LM_HD void sens_node(const ResultOut& R, const Params& P, const Mesh& M, const WS& W, const IpmState& S,
                     const SolveOut& out, int k, const double* z, double m, const Accel1& f, SensSums& a) {
  const double u = z[6];
  const double al = M.h[k] * P.T * out.tf;
  // the multipliers are read here and not with z: held across accel_first they spill in the thread kernel
  double lam[3];
  SW::node(W, out.cur, k, nullptr, lam);
  const double l1 = lam[0], l3 = lam[1], l5 = lam[2];                    // ydot, xdot and angledot rows
  const double thrust = l1 * (f.AT * f.Ty * P.Sinv) + l3 * (f.AT * f.Tx * P.Sinv);
  a.ft -= al * thrust / P.Ft;
  a.m0 += al * thrust * (f.AT / P.Ft);                                  // d AT / d M0 = -AT / (M0 - ms*mass)
  a.mf -= al * (l1 * f.ay_m + l3 * f.ax_m) * (P.T * M.tau[k] * out.tf);
  a.asc -= al * u * l5;
  if (!R.psens) return;
  double d[9];                               // read after the four sums above, for the same reason as lam
  SW::node_duals(W, out.cur, k, d);
  const double ht = M.h[k] * out.tf;         // d alpha / d T
  const double mt = P.mflow * M.tau[k] * out.tf;   // d mass / d T
  const double r1 = d[1] * P.Sinv, r3 = d[3] * P.Sinv;
  const double fl = d[0] * z[1] + d[1] * f.ay + d[2] * z[3] + d[3] * f.ax + d[4] * z[5] + d[5] * (P.asc * u);
  a.t -= ht * fl + al * (d[1] * f.ay_m + d[3] * f.ax_m) * mt;
  a.gm += al * (f.rinv * f.rinv) * (r1 * f.ny + r3 * f.nx);
  a.r0 -= al * (r1 * f.ay_y + r3 * f.ax_y);
  a.sc -= al * (r1 * (z[2] * f.ay_x + z[0] * f.ay_y - f.ay) + r3 * (z[2] * f.ax_x + z[0] * f.ax_y - f.ax));
  a.ms -= al * (d[1] * (f.AT * f.Ty) + d[3] * (f.AT * f.Tx)) * P.Sinv * (f.AT / P.Ft) * m;   // d AT / d ms
  a.aub -= d[6];
  a.uub -= d[7] + d[8];
  if (k == M.N) {
    // terminal rows: multipliers -zs1 (radius - rt), -zs2 (speed^2 - vt2) and nu3 (r.v / S^2)
    Terminal T;
    terminal_eval(P, z[0], z[1], z[2], z[3], T);
    a.rt += S.cur.zs1;
    a.vt2 += S.cur.zs2;
    a.r0s += S.cur.nu3 * z[1] - S.cur.zs1 * T.Yb / T.rT;
  }
}

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
  if (!R.traj && !R.sens && !R.psens) return;
  double* __restrict__ t = R.traj;
  if (t) {
    for (int v = g; v < LMATO_NVAR; v += G) t[((long)v * nt) * B + b] = 0.0;   // node 0 pinned
  }
  // Parametric sensitivity of the optimum (envelope theorem): d objective* / d theta = d Lagrangian / d theta
  // = sum_k lambda_k . d c_k / d theta at the solution, with c_k = s_k - s_{k-1} - h_k T tf F(s_k, u_k; theta).
  // theta enters only the velocity rows (through the thrust acceleration Ft / (M0 - ms*mass), LO:127-136,
  // and mass = mflow*T*tau*tf, LO:123) and the angledot row (angle_scalar, LO:121).
  // For psens, every field of ParamsGrad (ascent_model.cuh): T enters every defect row through alpha = h*T*tf and the
  // mass; GM, R0 and the distance scale S enter the velocity rows through gravity and the scaling (X = x*S,
  // Y = y*S + R0, 1/S); ms the thrust acceleration; a_ub and u_ub the bounds of node k (their multipliers); R0S, rt
  // and vt2 the terminal rows.  derive_params_grad maps these onto the raw rows.
  SensSums a{};
  for (int k = 1 + g; k <= M.N; k += G) {
    double z[7];                                   // the six states and the control u = z[6]
    SW::node(W, out.cur, k, z, nullptr);
    const double u = z[6];
    const double m = P.mflow * P.T * M.tau[k] * out.tf;
    // the trajectory's accelerations: from the derivative pass with lmato_sens_t's output (as it has always been
    // written), else from this one evaluation, with or without the all-row output
    double ay, ax;
    if (!R.sens) accel_value(P, z[0], z[2], z[4], m, ay, ax);
    if (R.sens || R.psens) {
      Accel1 f;
      accel_first(P, z[0], z[2], z[4], m, f);
      if (R.sens) { ay = f.ay; ax = f.ax; }
      sens_node<SW>(R, P, M, W, S, out, k, z, m, f, a);
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
  if (R.sens || R.psens) {
    a.ft = coop::Grp<G>::sum(mask, a.ft); a.m0 = coop::Grp<G>::sum(mask, a.m0);
    a.mf = coop::Grp<G>::sum(mask, a.mf); a.asc = coop::Grp<G>::sum(mask, a.asc);
    // the mass bound 0 <= mass <= 1 (LO:83) is carried as tf <= tf_ub = 1 / (mflow T): where that is the binding
    // upper bound on tf, its multiplier contributes  -zUt * d tf_ub / d mflow = zUt / (mflow^2 T)
    if (P.tf_ub < 1.0) a.mf += S.cur.zUt / (P.mflow * P.mflow * P.T);
    if (g == 0 && R.sens) {
      // per unit of the RAW parameters of include/lmato_b200.h: M_dot = mflow * fuel_mass (LO:65),
      // angle_doubledot_max = 3 * angle_scalar (LO:109); tf in the reference's scaled units (0..1)
      const double inv = 1.0 / obj_scale;
      R.sens[(long)LMATO_S_FT * B + b] = a.ft * inv;
      R.sens[(long)LMATO_S_M0 * B + b] = a.m0 * inv;
      R.sens[(long)LMATO_S_M_DOT * B + b] = a.mf * inv / P.fuel;
      // the circular model has no pitch-acceleration limit (its MV is the angle): no such derivative exists there
      R.sens[(long)LMATO_S_ANGLE_DOUBLEDOT_MAX * B + b] = model == LMATO_MODEL_CIRCULAR ? NAN : a.asc * inv / 3.0;
    }
  }
  if (R.psens) {
    a.gm = coop::Grp<G>::sum(mask, a.gm); a.r0 = coop::Grp<G>::sum(mask, a.r0); a.sc = coop::Grp<G>::sum(mask, a.sc);
    a.ms = coop::Grp<G>::sum(mask, a.ms); a.t = coop::Grp<G>::sum(mask, a.t); a.aub = coop::Grp<G>::sum(mask, a.aub);
    a.uub = coop::Grp<G>::sum(mask, a.uub); a.vt2 = coop::Grp<G>::sum(mask, a.vt2); a.rt = coop::Grp<G>::sum(mask, a.rt);
    a.r0s = coop::Grp<G>::sum(mask, a.r0s);
    // the binding mass bound tf <= tf_ub = 1 / (mflow T) (see a.mf above): -zUt * d tf_ub / d T = zUt / (mflow T^2)
    if (P.tf_ub < 1.0) a.t += S.cur.zUt / (P.mflow * P.T * P.T);
    if (g == 0) {
      // the derivative of the whole objective (with the move term), per unit of obj_scale; the four rows of sens are
      // the same values
      const double inv = 1.0 / obj_scale;
      const ParamsGrad pg{a.gm * inv, a.r0 * inv, a.ft * inv, a.m0 * inv, a.sc * inv, a.ms * inv, a.mf * inv,
                          a.asc * inv, a.t * inv, a.aub * inv, a.uub * inv, a.vt2 * inv, a.rt * inv, a.r0s * inv};
      derive_params_grad(R.params, B, b, model, pg, R.psens + b, B);
    }
  }
}

}  // namespace lmato
