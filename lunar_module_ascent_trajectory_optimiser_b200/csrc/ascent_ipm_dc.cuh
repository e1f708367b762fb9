// 8-state variant of the sweeps: the NLP with the reference's move-suppression term
//     + dcost * sum_k |MV_k - MV_{k-1}|        (angledoubledot.DCOST = 1e-5, LO:99; MV(0) = 0)
// on top of minimise tf (LO:176).  As in APMonitor (SURVEY B.3) the l1 term is written with a
// non-negative slack pair per step,  MV_k - MV_{k-1} = p_k - n_k,  cost w (p_k + n_k),  and the pair
// is treated primal-dually like every other bound: p, n and their multipliers z_p, z_n are part of
// the iterate; in the Newton system they condense into an effective quadratic cost of the move
//     R = Sp Sn / (Sp + Sn),   r = (gp Sn - gn Sp) / (Sp + Sn) + R c,      Sp = z_p/p, Sn = z_n/n,
//     gp = w - mu/p, gn = w - mu/n,  c = u_k - u_{k-1} - p + n.
// (A closed-form elimination of the pair from the barrier problem was tried first; it is a primal
// barrier method for these two variables and zig-zags once mu/w drops below the move sizes.)
// Because a move couples two consecutive controls, the previous control becomes an eighth stage state:
//     s = (y, vy, x, vx | angle, angledot, u, tf),   control v_k = u_k - u_{k-1},
//     angledot_k - angledot_{k-1} - beta u_k = 0,    u_k - u_{k-1} - v_k = 0  (multiplier lam_6)
// The tuned 7-state sweeps in ascent_ipm.cuh are used whenever dcost = 0.
#pragma once
#include "ascent_ipm.cuh"

namespace lmato {
namespace dc {

enum : int {
  // iterate, two ping-pong copies of 22 rows
  F_Z = 0, F_U = 6, F_LAM = 7 /* 7 rows: six defects + the u row */, F_ZLA = 14, F_ZUA = 15, F_ZLU = 16, F_ZUU = 17,
  F_PP = 18, F_PN = 19, F_ZPP = 20, F_ZPN = 21,     // move slack pair and its multipliers
  N_ITER = 22,
  R_STEP = 2 * N_ITER,
  F_DS = R_STEP + 0, F_DU = R_STEP + 6, F_PI = R_STEP + 7 /* 7 rows */, N_STEP = 14,
  R_FACT = R_STEP + N_STEP,
  F_K = R_FACT + 0 /* 8 gains */, F_KFF = R_FACT + 8, N_FACT = 9,
  N_FIELDS = 2 * N_ITER + N_STEP + N_FACT,   // 67
  REF_ROWS = N_ITER + 1
};

// Condensed move cost of one step and the recovery of the pair's Newton step from the move step.
struct Move {
  double R, r;          // effective Hessian / gradient of the move
  double Sp, Sn, gp, gn, sinv, c;
  double ip, in_;       // 1/p, 1/n (one division for both; reused by the callers)
  LM_HD void build(double pp, double pn, double zp, double zn, double v, double w, double mu, bool ls) {
    const double ipn = lm_rcp(pp * pn);
    ip = ipn * pn; in_ = ipn * pp;
    if (!ls) { Sp = zp * ip; Sn = zn * in_; gp = w - mu * ip; gn = w - mu * in_; c = v - pp + pn; }
    else     { Sp = 1.0; Sn = 1.0; gp = w - zp; gn = w - zn; c = 0.0; }
    sinv = lm_rcp(Sp + Sn);
    R = Sp * Sn * sinv;
    r = (gp * Sn - gn * Sp) * sinv + R * c;
  }
  // dp - dn = dv + c
  LM_HD void steps(double dv, double& dp, double& dn) const {
    dn = -(Sp * (dv + c) + gp + gn) * sinv;
    dp = dv + c + dn;
  }
};

// v <- E^{-1} v (8 states)
LM_HD void solveE8(const StageJac& J, double* v) {
  const double v7 = v[7], v6 = v[6];
  const double v5 = v[5] + J.beta * v6 + J.e5 * v7;
  const double v4 = v[4] + J.al * v5 + J.e4 * v7;
  const double r0 = fma(J.e0, v7, v[0]);
  const double r2 = fma(J.e2, v7, v[2]);
  const double r1 = v[1] + J.ga1 * v4 + J.e1 * v7;
  const double r3 = v[3] + J.ga3 * v4 + J.e3 * v7;
  const double t1 = r1 + J.ala * r0 + J.alb * r2;
  const double t3 = r3 + J.alc * r0 + J.ald * r2;
  const double v1 = J.m11 * t1 + J.m13 * t3;
  const double v3 = J.m31 * t1 + J.m33 * t3;
  v[0] = fma(J.al, v1, r0); v[1] = v1; v[2] = fma(J.al, v3, r2); v[3] = v3; v[4] = v4; v[5] = v5;
}

// g <- E^{-T} g (8 states)
LM_HD void solveET8(const StageJac& J, double* g) {
  double w0 = g[0], w1 = g[1], w2 = g[2], w3 = g[3];
  applyA11T(J, w0, w1, w2, w3);
  const double gaw = J.ga1 * w1 + J.ga3 * w3;
  const double gew = J.e0 * w0 + J.e1 * w1 + J.e2 * w2 + J.e3 * w3;
  const double w4 = g[4] + gaw;
  const double w5 = g[5] + J.al * w4;
  const double w6 = g[6] + J.beta * w5;
  const double w7 = g[7] + gew + J.e4 * w4 + J.e5 * w5;
  g[0] = w0; g[1] = w1; g[2] = w2; g[3] = w3; g[4] = w4; g[5] = w5; g[6] = w6; g[7] = w7;
}

static_assert((int)F_LAM == NODE_LAM && (int)F_ZLA == NODE_ZLA && (int)F_ZUU == NODE_ZUU && (int)F_PP == NODE_PP &&
              (int)F_ZPN == NODE_ZPN && (int)N_ITER == NODE_N, "the 8-state rows are the rows of a start node (ascent_ipm.cuh)");

// ---------------------------------------------------------------------------------------
// Staging tiles (see ascent_ipm.cuh: tl_*): which rows each sweep reads per stage and where they sit
// in the tile.  "CUR" = rows F_LAM .. N_ITER-1 of the source iterate at stage k (multipliers and the
// slack pair), "PZ"/"PDS" = (s, u) and their steps at stage k-1.
// ---------------------------------------------------------------------------------------
enum : int {
  N_CUR = N_ITER - F_LAM,                          // 15
  EV_CUR = 0, EV_PI = EV_CUR + N_CUR, EV_PZ = EV_PI + 7, EV_PDS = EV_PZ + 7, EV_ROWS = EV_PDS + 7,
  BK_CUR = 0, BK_PZ = BK_CUR + N_CUR, BK_ROWS = BK_PZ + 7,
  FW_Z = 0, FW_ZB = FW_Z + 7, FW_K = FW_ZB + (N_ITER - F_ZLA), FW_ROWS = FW_K + N_FACT
};
static_assert(EV_ROWS <= TILE_DATA && BK_ROWS <= TILE_DATA && FW_ROWS <= TILE_DATA, "tile too small");
#define TL_CUR(tb, base, f) tl_ld(tb, (base) + (f) - F_LAM)      // row f (>= F_LAM) of the source iterate

LM_HD void ev_stage_copy(const Mesh& M, const Ws& W, int k, int so, bool read_pi) {
  const TileRef tb = tl_buf(W, k);
  tl_copy_mesh(tb, M, k);
  const double* sp = W.stage(k);
  const double* sm = ws_opaque(sp - W.SS);
  const double* spo = ws_opaque(sp + so * LANES);
  const double* smo = ws_opaque(sm + so * LANES);
  tl_copy_rows<EV_CUR, N_CUR>(tb, spo, F_LAM);
  if (read_pi) tl_copy_rows<EV_PI, 7>(tb, sp, F_PI);
  tl_copy_rows<EV_PZ, 7>(tb, smo, F_Z);
  tl_copy_rows<EV_PDS, 7>(tb, sm, F_DS);
  tl_commit();
}
// Inside the stage loops the same copies are issued in two halves, each its own commit group: (a) at the top of the
// stage body, (b) in the middle of it.  As one burst the 24-38 LDGSTS of a stage filled the load/store unit's queue
// (the source view showed 39 % "lg_throttle" and 16 % "mio_throttle" stall samples on the copy blocks); split, config 4
// runs 85.2 -> 82.7 ms.  Three parts are slower again (85.4).  The wait is unchanged: before stage k is consumed
// everything but the newest group -- part (a) of stage k-1, just issued -- has landed.
LM_HD void ev_stage_copy_a(const Mesh& M, const Ws& W, int k, int so, bool read_pi) {
  const TileRef tb = tl_buf(W, k);
  tl_copy_mesh(tb, M, k);
  const double* sp = W.stage(k);
  tl_copy_rows<EV_CUR, N_CUR>(tb, ws_opaque(sp + so * LANES), F_LAM);
  if (read_pi) tl_copy_rows<EV_PI, 7>(tb, sp, F_PI);
  tl_commit();
}
LM_HD void ev_stage_copy_b(const Ws& W, int k, int so) {
  const TileRef tb = tl_buf(W, k);
  const double* sm = ws_opaque(W.stage(k) - W.SS);
  tl_copy_rows<EV_PZ, 7>(tb, ws_opaque(sm + so * LANES), F_Z);
  tl_copy_rows<EV_PDS, 7>(tb, sm, F_DS);
  tl_commit();
}
LM_HD void bk_stage_copy_a(const Mesh& M, const Ws& W, int k, int so) {
  const TileRef tb = tl_buf(W, k);
  tl_copy_mesh(tb, M, k);
  tl_copy_rows<BK_CUR, N_CUR>(tb, ws_opaque(W.stage(k) + so * LANES), F_LAM);
  tl_commit();
}
LM_HD void bk_stage_copy_b(const Ws& W, int k, int so) {
  const TileRef tb = tl_buf(W, k);
  tl_copy_rows<BK_PZ, 7>(tb, ws_opaque(W.stage(k) + so * LANES - W.SS), F_Z);
  tl_commit();
}
LM_HD void fw_stage_copy_a(const Mesh& M, const Ws& W, int k, int so) {
  const TileRef tb = tl_buf(W, k);
  tl_copy_mesh(tb, M, k);
  const double* spo = ws_opaque(W.stage(k) + so * LANES);
  tl_copy_rows<FW_Z, 7>(tb, spo, F_Z);
  tl_copy_rows<FW_ZB, N_ITER - F_ZLA>(tb, spo, F_ZLA);
  tl_commit();
}
LM_HD void fw_stage_copy_b(const Ws& W, int k) {
  const TileRef tb = tl_buf(W, k);
  tl_copy_rows<FW_K, N_FACT>(tb, W.stage(k), F_K);
  tl_commit();
}

LM_HD void bk_stage_copy(const Mesh& M, const Ws& W, int k, int so) {
  const TileRef tb = tl_buf(W, k);
  tl_copy_mesh(tb, M, k);
  const double* spo = ws_opaque(W.stage(k) + so * LANES);
  tl_copy_rows<BK_CUR, N_CUR>(tb, spo, F_LAM);
  tl_copy_rows<BK_PZ, 7>(tb, ws_opaque(spo - W.SS), F_Z);
  tl_commit();
}
LM_HD void fw_stage_copy(const Mesh& M, const Ws& W, int k, int so) {
  const TileRef tb = tl_buf(W, k);
  tl_copy_mesh(tb, M, k);
  const double* sp = W.stage(k);
  const double* spo = ws_opaque(sp + so * LANES);
  tl_copy_rows<FW_Z, 7>(tb, spo, F_Z);
  tl_copy_rows<FW_ZB, N_ITER - F_ZLA>(tb, spo, F_ZLA);
  tl_copy_rows<FW_K, N_FACT>(tb, sp, F_K);
  tl_commit();
}

// ---------------------------------------------------------------------------------------
// evaluation pass (see ascent_ipm.cuh: eval_pass); differences: u is a state of the node, the u row
// and its multiplier lam_6, the move slack pair (p, n, z_p, z_n) in the merit and the residuals.
// ---------------------------------------------------------------------------------------
LM_SWEEP void eval_pass(const Params& P, const Mesh& M, const Options& O, const Ws& W, int src, int dst,
                           const Scal& c0, const TermStep& ts, double mu, double dw, double alpha,
                           double alpha_z, double alpha_lam, int mode, Scal& t, double* pimax_out) {
  const int N = M.N;
  const int so = src * N_ITER, dd = dst * N_ITER;
  tl_begin();
  ev_stage_copy(M, W, N, so, mode == EV_READ_PI);
  const double tf0 = c0.tf, dtf = ts.dtf;
  t.tf = tf0 + alpha * dtf;
  const double tf = t.tf;
  const bool ls = (mode == EV_LSQ);
  const double wdc = O.w_dcost;
  double theta = 0, prim = 0, dual = 0, sumlog = 0, cmin = 1e300, cmax = 0, slam = 0, sz = 0;
  double gtf = 0, pimax = 0, movecost = 0;
  bool bad = false;
  t.sg1 = c0.sg1 + alpha * ts.dsg1;
  t.sg2 = c0.sg2 + alpha * ts.dsg2;
  t.nu3 = c0.nu3 + alpha_lam * ts.dnu3;
  t.zs1 = c0.zs1 + alpha_z * ts.dzs1;
  t.zs2 = c0.zs2 + alpha_z * ts.dzs2;
  t.zLt = c0.zLt + alpha_z * ts.dzLt;
  t.zUt = c0.zUt + alpha_z * ts.dzUt;
  {
    const double dLt = tf, dUt = P.tf_ub - tf;
    if (!(t.sg1 > 0 && t.sg2 > 0 && dLt > 0 && dUt > 0)) bad = true;
    t.zs1 = clip_mult(t.zs1, t.sg1, mu);
    t.zs2 = clip_mult(t.zs2, t.sg2, mu);
    t.zLt = clip_mult(t.zLt, dLt, mu);
    t.zUt = clip_mult(t.zUt, dUt, mu);
    sumlog += log((t.sg1 * t.sg2) * (dLt * dUt));
    const double q1 = t.sg1 * t.zs1, q2 = t.sg2 * t.zs2, q3 = dLt * t.zLt, q4 = dUt * t.zUt;
    cmin = dmin(cmin, dmin(dmin(q1, q2), dmin(q3, q4)));
    cmax = dmax(cmax, dmax(dmax(q1, q2), dmax(q3, q4)));
    sz += t.zs1 + t.zs2 + t.zLt + t.zUt;
    slam += t.zs1 + t.zs2 + fabs(t.nu3);
    gtf += O.obj_scale - t.zLt + t.zUt;
  }
  // node k (old point + step); node k-1 is loaded while node k is processed
  double zo[7], ds[7];      // index 6 = u
  {
    const double* sp = W.stage(N);
#pragma unroll
    for (int i = 0; i < 6; ++i) { zo[i] = WS_AT(sp, so + F_Z + i); ds[i] = WS_AT(sp, F_DS + i); }
    zo[6] = WS_AT(sp, so + F_U); ds[6] = WS_AT(sp, F_DU);
  }
  double lam_next[7] = {0, 0, 0, 0, 0, 0, 0};
  double pi_next[7] = {0, 0, 0, 0, 0, 0, 0};
  for (int k = N; k >= 1; --k) {
    double* sp = W.stage(k);
    if (k > 1) ev_stage_copy_a(M, W, k - 1, so, mode == EV_READ_PI); else tl_commit();
    tl_wait_prev();
    const TileRef tb = tl_buf(W, k);
    double z[7], zpo[7], dsp[7], zp[7], lam[7];
#pragma unroll
    for (int i = 0; i < 7; ++i) z[i] = fma(alpha, ds[i], zo[i]);
#pragma unroll
    for (int i = 0; i < 7; ++i) {                 // node k-1 (node 0 rows are zeros)
      zpo[i] = tl_ld(tb, EV_PZ + i); dsp[i] = tl_ld(tb, EV_PDS + i);
      zp[i] = fma(alpha, dsp[i], zpo[i]);
    }
    const double u_old = zo[6], du = ds[6], u = z[6];
    double lam_old[7];
#pragma unroll
    for (int i = 0; i < 7; ++i) lam_old[i] = TL_CUR(tb, EV_CUR, F_LAM + i);
    double zla = TL_CUR(tb, EV_CUR, F_ZLA), zua = TL_CUR(tb, EV_CUR, F_ZUA);
    double zlu = TL_CUR(tb, EV_CUR, F_ZLU), zuu = TL_CUR(tb, EV_CUR, F_ZUU);
    const double kap = tl_ld(tb, TL_H) * P.T;
    const double taum = P.mT * tl_ld(tb, TL_TAU);
    // ---- new multipliers pi_k ----
    double pi[7];
    if (mode != EV_READ_PI) {
      Accel1 f0;
      accel_first(P, zo[0], zo[2], zo[4], taum * tf0, f0);
      StageJac J0;
      stagejac_build(P, kap, tf0, taum, f0, zo[1], zo[3], zo[5], u_old, J0);
      stagejac_invert(J0);
      StageQ q;
      stage_hessian(P, f0, J0, kap, taum, lam_old, zo[4], u_old, zla, zua, zlu, zuu, mu, dw, ls, q);
      // Stationarity of the Newton QP wrt s_k:  E_k^T pi_k = D pi_{k+1} - (Q_k ds_k + q_k).  The move
      // cost does not appear here: it sits in the stationarity of the move, pi_6,k = r + R dv_k, which
      // the solution of this recursion satisfies by construction.
      double g[8];
      g[0] = pi_next[0] - (q.q00 * ds[0] + q.q02 * ds[2] + q.q04 * ds[4] + q.q06 * dtf);
      g[1] = pi_next[1] - (q.d * ds[1] + q.q16 * dtf);
      g[2] = pi_next[2] - (q.q02 * ds[0] + q.q22 * ds[2] + q.q24 * ds[4] + q.q26 * dtf);
      g[3] = pi_next[3] - (q.d * ds[3] + q.q36 * dtf);
      g[4] = pi_next[4] - (q.q04 * ds[0] + q.q24 * ds[2] + q.q44 * ds[4] + q.q46 * dtf + q.q4);
      g[5] = pi_next[5] - (q.d * ds[5] + q.q56 * dtf);
      // u as a state: bound barrier (q.R - dw, q.r hold Sigma_u and its gradient), u-tf cross term
      g[6] = pi_next[6] - (q.R * du + q.sig * dtf + q.r);
      g[7] = 0.0;
      if (k == N) {
        TermQP tq;
        terminal_qp(P, O, c0, zo, mu, dw, ls, tq);
#pragma unroll
        for (int i = 0; i < 4; ++i)
          g[i] -= tq.H[i][0] * ds[0] + tq.H[i][1] * ds[1] + tq.H[i][2] * ds[2] + tq.H[i][3] * ds[3] + tq.g[i];
      }
      solveET8(J0, g);
#pragma unroll
      for (int i = 0; i < 7; ++i) { pi[i] = g[i]; WS_AT(sp, F_PI + i) = g[i]; pimax = dmax(pimax, fabs(g[i])); }
    } else {
#pragma unroll
      for (int i = 0; i < 7; ++i) pi[i] = tl_ld(tb, EV_PI + i);
    }
#pragma unroll
    for (int i = 0; i < 7; ++i) lam[i] = fma(alpha_lam, pi[i] - lam_old[i], lam_old[i]);
    if (k > 1) ev_stage_copy_b(W, k - 1, so); else tl_commit();      // second half of the next stage's tile
    // ---- bound multipliers ----
    {
      double rLa, rUa, rLu, rUu;
      recip4(zo[4], P.a_ub - zo[4], u_old + P.u_ub, P.u_ub - u_old, rLa, rUa, rLu, rUu);
      const double da = ds[4];
      zla += alpha_z * ((mu - zla * da) * rLa - zla);
      zua += alpha_z * ((mu + zua * da) * rUa - zua);
      zlu += alpha_z * ((mu - zlu * du) * rLu - zlu);
      zuu += alpha_z * ((mu + zuu * du) * rUu - zuu);
    }
    const double dLa = z[4], dUa = P.a_ub - z[4], dLu = u + P.u_ub, dUu = P.u_ub - u;
    if (!(dLa > 0 && dUa > 0 && dLu > 0 && dUu > 0)) bad = true;
    {
      const double c1 = dLa * zla, c2 = dUa * zua, c3 = dLu * zlu, c4 = dUu * zuu;
      const double hi = 1e10 * mu, lo = 1e-10 * mu;
      if (dmax(dmax(c1, c2), dmax(c3, c4)) > hi || dmin(dmin(c1, c2), dmin(c3, c4)) < lo) {
        zla = clip_mult(zla, dLa, mu); zua = clip_mult(zua, dUa, mu);
        zlu = clip_mult(zlu, dLu, mu); zuu = clip_mult(zuu, dUu, mu);
      }
    }
    const double slack4 = (dLa * dUa) * (dLu * dUu);      // its logarithm is taken together with the pair's below
    {
      const double c1 = dLa * zla, c2 = dUa * zua, c3 = dLu * zlu, c4 = dUu * zuu;
      cmin = dmin(cmin, dmin(dmin(c1, c2), dmin(c3, c4)));
      cmax = dmax(cmax, dmax(dmax(c1, c2), dmax(c3, c4)));
    }
    sz += (zla + zua) + (zlu + zuu);
    // ---- move slack pair: p, n follow the move step, their multipliers the dual step ----
    double pp = TL_CUR(tb, EV_CUR, F_PP), pn = TL_CUR(tb, EV_CUR, F_PN);
    double zpp = TL_CUR(tb, EV_CUR, F_ZPP), zpn = TL_CUR(tb, EV_CUR, F_ZPN);
    {
      Move mv;
      mv.build(pp, pn, zpp, zpn, u_old - zpo[6], wdc, mu, false);
      double dp, dn;
      mv.steps(du - dsp[6], dp, dn);
      const double ip = mv.ip, in_ = mv.in_;
      zpp += alpha_z * ((mu - zpp * dp) * ip - zpp);
      zpn += alpha_z * ((mu - zpn * dn) * in_ - zpn);
      pp = fma(alpha, dp, pp);
      pn = fma(alpha, dn, pn);
    }
    if (!(pp > 0 && pn > 0)) bad = true;
    {
      const double c1 = pp * zpp, c2 = pn * zpn;
      if (dmax(c1, c2) > 1e10 * mu || dmin(c1, c2) < 1e-10 * mu) { zpp = clip_mult(zpp, pp, mu); zpn = clip_mult(zpn, pn, mu); }
    }
    sumlog += lm_log_pos(slack4 * (pp * pn));             // six slacks in (0, ~2): no underflow
    {
      const double c1 = pp * zpp, c2 = pn * zpn;
      cmin = dmin(cmin, dmin(c1, c2));
      cmax = dmax(cmax, dmax(c1, c2));
    }
    sz += zpp + zpn;
    movecost += pp + pn;
    // ---- dynamics at the trial point ----
    Accel1 f;
    accel_first(P, z[0], z[2], z[4], taum * tf, f);
    StageJac J;
    stagejac_build(P, kap, tf, taum, f, z[1], z[3], z[5], u, J);
    const double al = J.al;
    double c[6];
    c[0] = z[0] - zp[0] - al * z[1];
    c[1] = z[1] - zp[1] - al * f.ay;
    c[2] = z[2] - zp[2] - al * z[3];
    c[3] = z[3] - zp[3] - al * f.ax;
    c[4] = z[4] - zp[4] - al * z[5];
    c[5] = z[5] - zp[5] - J.beta * u;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      const double ac = fabs(c[i]);
      theta += ac;
      prim = dmax(prim, ac);
      slam += fabs(lam[i]);
    }
    slam += fabs(lam[6]);
    {
      const double c6 = fabs((u - zp[6]) - pp + pn);            // move row: u_k - u_{k-1} = p - n
      theta += c6;
      prim = dmax(prim, c6);
    }
    // ---- Lagrangian gradient wrt (s_k, u_k) and wrt the move v_k ----
    double res[7];
    applyET6(J, lam, res);
    res[4] += zua - zla;
    res[6] = -J.beta * lam[5] + lam[6] - zlu + zuu;        // column u of E: -beta (angledot row), 1 (u row)
    if (k == N) {
      Terminal T;
      terminal_eval(P, z[0], z[1], z[2], z[3], T);
      const double c1 = T.g1 - t.sg1, c2 = T.g2 - t.sg2, c3 = T.g3;
      theta += fabs(c1) + fabs(c2) + fabs(c3);
      prim = dmax(prim, dmax(fabs(c1), dmax(fabs(c2), fabs(c3))));
      const double rinv = 1.0 / T.rT;
      res[0] += -t.zs1 * T.Yb * rinv + t.nu3 * z[1];
      res[2] += -t.zs1 * z[2] * rinv + t.nu3 * z[3];
      res[1] += -t.zs2 * 2.0 * z[1] + t.nu3 * T.Yb;
      res[3] += -t.zs2 * 2.0 * z[3] + t.nu3 * z[2];
    } else {
#pragma unroll
      for (int i = 0; i < 5; ++i) res[i] -= lam_next[i];
      res[5] -= lam_next[5];
      res[6] -= lam_next[6];
    }
#pragma unroll
    for (int i = 0; i < 7; ++i) dual = dmax(dual, fabs(res[i]));
    dual = dmax(dual, dmax(fabs(wdc - lam[6] - zpp), fabs(wdc + lam[6] - zpn)));   // d L / d p_k, d L / d n_k
    gtf -= J.e0 * lam[0] + J.e1 * lam[1] + J.e2 * lam[2] + J.e3 * lam[3] + J.e4 * lam[4] + J.e5 * lam[5];
    // ---- write the trial iterate, shift the pipeline ----
double* spd = ws_opaque(sp + dd * LANES);
#pragma unroll
    for (int i = 0; i < 6; ++i) WS_AT(spd, F_Z + i) = z[i];
#pragma unroll
    for (int i = 0; i < 7; ++i) {
      WS_AT(spd, F_LAM + i) = lam[i];
      lam_next[i] = lam[i]; pi_next[i] = pi[i]; zo[i] = zpo[i]; ds[i] = dsp[i];
    }
    WS_AT(spd, F_U) = u;
    WS_AT(spd, F_ZLA) = zla; WS_AT(spd, F_ZUA) = zua;
    WS_AT(spd, F_ZLU) = zlu; WS_AT(spd, F_ZUU) = zuu;
    WS_AT(spd, F_PP) = pp; WS_AT(spd, F_PN) = pn;
    WS_AT(spd, F_ZPP) = zpp; WS_AT(spd, F_ZPN) = zpn;
  }
  dual = dmax(dual, fabs(gtf));
  t.theta = theta;
  t.fobj = O.obj_scale * tf + wdc * movecost;
  t.sumlog = bad ? -1e300 : sumlog;
  t.prim_inf = prim; t.dual_inf = dual; t.cmin = cmin; t.cmax = cmax; t.sum_lam = slam; t.sum_z = sz;
  if (bad || !(theta == theta)) t.theta = 1e300;
  if (pimax_out) *pimax_out = pimax;
}

// ---------------------------------------------------------------------------------------
// backward Riccati sweep, 8 states: p = (y,vy,x,vx), q = (angle, angledot, u, tf); the control is the
// move v (enters the u row with coefficient 1; its cost is the condensed slack pair, struct Move).
// ---------------------------------------------------------------------------------------
LM_SWEEP bool riccati_backward(const Params& P, const Mesh& M, const Options& O, const Ws& W, int src,
                                  const Scal& c0, double mu, double dw, bool ls_arg, double* dtf_out) {
  const bool ls = ls_arg;
  const int N = M.N;
  const double tf = c0.tf;
  const int so = src * N_ITER;
  tl_begin();
  bk_stage_copy(M, W, N, so);
  const double wdc = O.w_dcost;
  double A[4][4], Bm[4][4], C[4][4];     // C: q x q, full storage (kept symmetric)
  double pv[8];
  double zn[7];
  {
    const double* sp = W.stage(N);
#pragma unroll
    for (int i = 0; i < 6; ++i) zn[i] = WS_AT(sp, so + F_Z + i);
    zn[6] = WS_AT(sp, so + F_U);
  }
  {
    TermQP tq;
    terminal_qp(P, O, c0, zn, mu, dw, ls, tq);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int j = 0; j < 4; ++j) { A[i][j] = tq.H[i][j]; Bm[i][j] = 0.0; C[i][j] = 0.0; }
      pv[i] = tq.g[i];
    }
    C[3][3] = tq.H66;
    pv[4] = 0.0; pv[5] = 0.0; pv[6] = 0.0; pv[7] = tq.g6;
  }
  bool ok = true;
  for (int k = N; k >= 1; --k) {
    double* sp = W.stage(k);
    if (k > 1) bk_stage_copy_a(M, W, k - 1, so); else tl_commit();
    tl_wait_prev();
    const TileRef tb = tl_buf(W, k);
    const bool ls = W.ls_flag != 0;      // shadows the argument: a shared-memory load per stage
    double lam[6], zm[7];
#pragma unroll
    for (int i = 0; i < 6; ++i) lam[i] = TL_CUR(tb, BK_CUR, F_LAM + i);
#pragma unroll
    for (int i = 0; i < 7; ++i) zm[i] = tl_ld(tb, BK_PZ + i);
    const double u = zn[6];
    const double zla = TL_CUR(tb, BK_CUR, F_ZLA), zua = TL_CUR(tb, BK_CUR, F_ZUA);
    const double zlu = TL_CUR(tb, BK_CUR, F_ZLU), zuu = TL_CUR(tb, BK_CUR, F_ZUU);
    const double kap = tl_ld(tb, TL_H) * P.T;
    const double taum = P.mT * tl_ld(tb, TL_TAU);
    Accel1 f;
    accel_first(P, zn[0], zn[2], zn[4], taum * tf, f);
    StageJac J;
    stagejac_build(P, kap, tf, taum, f, zn[1], zn[3], zn[5], u, J);
    stagejac_invert(J);
    const double al = J.al;
    StageQ q;
    stage_hessian(P, f, J, kap, taum, lam, zn[4], u, zla, zua, zlu, zuu, mu, dw, ls, q);
    // ---- W = Q_k + P_k; q-indices: 0 angle, 1 angledot, 2 u, 3 tf ----
    A[0][0] += q.q00;
    A[2][0] += q.q02; A[0][2] += q.q02;
    A[2][2] += q.q22;
    A[1][1] += q.d; A[3][3] += q.d;
    Bm[0][0] += q.q04; Bm[2][0] += q.q24;
    Bm[0][3] += q.q06; Bm[1][3] += q.q16; Bm[2][3] += q.q26; Bm[3][3] += q.q36;
    C[0][0] += q.q44; C[1][1] += q.d;
    C[2][2] += q.R;                              // Sigma_u + delta_w (u is a bounded state here)
    C[0][3] += q.q46; C[3][0] += q.q46;
    C[1][3] += q.q56; C[3][1] += q.q56;
    C[2][3] += q.sig; C[3][2] += q.sig;
    C[3][3] += q.q66;
    pv[4] += q.q4;
    pv[6] += q.r;
    Move mv;
    mv.build(TL_CUR(tb, BK_CUR, F_PP), TL_CUR(tb, BK_CUR, F_PN), TL_CUR(tb, BK_CUR, F_ZPP), TL_CUR(tb, BK_CUR, F_ZPN),
             u - zm[6], wdc, mu, ls);
    const double R = mv.R + (ls ? 0.0 : dw);
    const double r = mv.r;
    double c[6];
    if (!ls) {
      c[0] = zn[0] - zm[0] - al * zn[1];
      c[1] = zn[1] - zm[1] - al * f.ay;
      c[2] = zn[2] - zm[2] - al * zn[3];
      c[3] = zn[3] - zm[3] - al * f.ax;
      c[4] = zn[4] - zm[4] - al * zn[5];
      c[5] = zn[5] - zm[5] - J.beta * u;
    } else {
#pragma unroll
      for (int i = 0; i < 6; ++i) c[i] = 0.0;
    }
    // ---- T1 ----
#pragma unroll
    for (int j = 0; j < 4; ++j) applyA11T(J, A[0][j], A[1][j], A[2][j], A[3][j]);
#pragma unroll
    for (int i = 0; i < 4; ++i) applyA11T(J, A[i][0], A[i][1], A[i][2], A[i][3]);
#pragma unroll
    for (int j = 0; j < 4; ++j) applyA11T(J, Bm[0][j], Bm[1][j], Bm[2][j], Bm[3][j]);
    if (k > 1) bk_stage_copy_b(W, k - 1, so); else tl_commit();      // second half of the next stage's tile
    // ---- T2: (angle, tf) couple into the velocity rows: C_T2 = [ga | 0 | 0 | e] ----
    {
      double ACa[4], ACt[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        ACa[i] = A[i][1] * J.ga1 + A[i][3] * J.ga3;
        ACt[i] = A[i][0] * J.e0 + A[i][1] * J.e1 + A[i][2] * J.e2 + A[i][3] * J.e3;
      }
      double CtBa[4], CtBt[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        CtBa[j] = J.ga1 * Bm[1][j] + J.ga3 * Bm[3][j];
        CtBt[j] = J.e0 * Bm[0][j] + J.e1 * Bm[1][j] + J.e2 * Bm[2][j] + J.e3 * Bm[3][j];
      }
      const double aa = J.ga1 * ACa[1] + J.ga3 * ACa[3];
      const double at = J.ga1 * ACt[1] + J.ga3 * ACt[3];
      const double tt = J.e0 * ACt[0] + J.e1 * ACt[1] + J.e2 * ACt[2] + J.e3 * ACt[3];
      // C += Ct B + (Ct B)^T + Ct A C, rows/cols 0 (angle) and 3 (tf) of Ct are the non-zero ones
#pragma unroll
      for (int j = 0; j < 4; ++j) { C[0][j] += CtBa[j]; C[j][0] += CtBa[j]; C[3][j] += CtBt[j]; C[j][3] += CtBt[j]; }
      C[0][0] += aa; C[0][3] += at; C[3][0] += at; C[3][3] += tt;
#pragma unroll
      for (int i = 0; i < 4; ++i) { Bm[i][0] += ACa[i]; Bm[i][3] += ACt[i]; }
    }
    // ---- T3: A22 = elementary column operations  w += al*a ; u += beta*w ; tf += e4*a + e5*w ----
    {
      const double be = J.beta, e4 = J.e4, e5 = J.e5;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        Bm[i][1] = fma(al, Bm[i][0], Bm[i][1]);
        Bm[i][2] = fma(be, Bm[i][1], Bm[i][2]);
        Bm[i][3] += e4 * Bm[i][0] + e5 * Bm[i][1];
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {      // columns
        C[i][1] = fma(al, C[i][0], C[i][1]);
        C[i][2] = fma(be, C[i][1], C[i][2]);
        C[i][3] += e4 * C[i][0] + e5 * C[i][1];
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {      // rows
        C[1][j] = fma(al, C[0][j], C[1][j]);
        C[2][j] = fma(be, C[1][j], C[2][j]);
        C[3][j] += e4 * C[0][j] + e5 * C[1][j];
      }
    }
    solveET8(J, pv);
    // ---- condense the move (enters the u row, q-index 2, with coefficient 1) ----
    const double Ruu = R + C[2][2];
    double Rux[8];
#pragma unroll
    for (int i = 0; i < 4; ++i) Rux[i] = Bm[i][2];
#pragma unroll
    for (int j = 0; j < 4; ++j) Rux[4 + j] = 0.5 * (C[2][j] + C[j][2]);
    double rx[8];
#pragma unroll
    for (int i = 0; i < 4; ++i)
      rx[i] = pv[i] - (A[i][0] * c[0] + A[i][1] * c[1] + A[i][2] * c[2] + A[i][3] * c[3] + Bm[i][0] * c[4] + Bm[i][1] * c[5]);
#pragma unroll
    for (int j = 0; j < 4; ++j)
      rx[4 + j] = pv[4 + j] - (Bm[0][j] * c[0] + Bm[1][j] * c[1] + Bm[2][j] * c[2] + Bm[3][j] * c[3] + C[j][0] * c[4] + C[j][1] * c[5]);
    const double ru = r + rx[6];
    // (these sweeps serve the elliptical model only -- coup5 = 1, d defect_k / d s_{k-1} = -I: the circular model
    //  runs the 7-state sweeps, and with its move term the cooperative kernel)
    if (!(Ruu > 0.0) || !(Ruu < 1e300)) ok = false;
    const double Rinv = lm_rcp(Ruu);
    double RuxS[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { RuxS[i] = Rux[i] * Rinv; WS_AT(sp, F_K + i) = -RuxS[i]; }
    WS_AT(sp, F_KFF) = -ru * Rinv;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int j = 0; j <= i; ++j) {
        const double v = 0.5 * (A[i][j] + A[j][i]) - Rux[i] * RuxS[j];
        A[i][j] = v; A[j][i] = v;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) Bm[i][j] -= Rux[i] * RuxS[4 + j];
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int j = 0; j <= i; ++j) {
        const double v = 0.5 * (C[i][j] + C[j][i]) - Rux[4 + i] * RuxS[4 + j];
        C[i][j] = v; C[j][i] = v;
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) pv[i] = rx[i] - RuxS[i] * ru;
#pragma unroll
    for (int i = 0; i < 7; ++i) zn[i] = zm[i];
    if (!ok) return false;
  }
  // node 0: everything pinned except tf (u_0 = 0 is pinned, LO:96 + GEKKO's node-0 rule)
  if (!(C[3][3] > 0.0)) return false;
  *dtf_out = -pv[7] / C[3][3];
  return true;
}

// ---------------------------------------------------------------------------------------
// forward sweep, 8 states
// ---------------------------------------------------------------------------------------
LM_SWEEP void riccati_forward(const Params& P, const Mesh& M, const Options& O, const Ws& W, int src,
                                 const Scal& c0, double mu, double tau, double dtf, bool ls_arg, TermStep& ts,
                                 StepInfo& si) {
  const bool ls = ls_arg;
  const int N = M.N;
  const double tf = c0.tf;
  const int so = src * N_ITER;
  const double wdc = O.w_dcost;
  tl_begin();
  fw_stage_copy(M, W, 1, so);
  double ds[8] = {0, 0, 0, 0, 0, 0, 0, dtf};      // (y,vy,x,vx,a,w,u,tf) of the previous node
  double zm[7] = {0, 0, 0, 0, 0, 0, 0};
  double dphi = 0.0, dxmax = fabs(dtf);
  RatioMax rp, rz;
  rp.init(); rz.init();
  const double cw = ls ? 0.0 : 1.0;
  for (int k = 1; k <= N; ++k) {
    double* sp = W.stage(k);
    if (k < N) fw_stage_copy_a(M, W, k + 1, so); else tl_commit();
    tl_wait_prev();
    const TileRef tb = tl_buf(W, k);
    const bool ls = W.ls_flag != 0;      // shadows the argument: a shared-memory load per stage
    double zn[7];
#pragma unroll
    for (int i = 0; i < 7; ++i) zn[i] = tl_ld(tb, FW_Z + i);
    const double u = zn[6];
    const double kap = tl_ld(tb, TL_H) * P.T;
    const double taum = P.mT * tl_ld(tb, TL_TAU);
    Accel1 f;
    accel_first(P, zn[0], zn[2], zn[4], taum * tf, f);
    StageJac J;
    stagejac_build(P, kap, tf, taum, f, zn[1], zn[3], zn[5], u, J);
    stagejac_invert(J);
    const double al = J.al;
    double dv = tl_ld(tb, FW_K + 8);
#pragma unroll
    for (int i = 0; i < 8; ++i) dv = fma(tl_ld(tb, FW_K + i), ds[i], dv);
    double xi[8];
    xi[0] = ds[0] - cw * (zn[0] - zm[0] - al * zn[1]);
    xi[1] = ds[1] - cw * (zn[1] - zm[1] - al * f.ay);
    xi[2] = ds[2] - cw * (zn[2] - zm[2] - al * zn[3]);
    xi[3] = ds[3] - cw * (zn[3] - zm[3] - al * f.ax);
    xi[4] = ds[4] - cw * (zn[4] - zm[4] - al * zn[5]);
    xi[5] = ds[5] - cw * (zn[5] - zm[5] - J.beta * u);
    xi[6] = ds[6] + dv;                       // u row: du_k = du_{k-1} + dv_k (its defect is identically 0)
    xi[7] = dtf;
    solveE8(J, xi);
    if (k < N) fw_stage_copy_b(W, k + 1); else tl_commit();          // second half of the next stage's tile
    {
      // slack pair: primal and dual steps, fraction to the boundary, merit slope
      const double pp = tl_ld(tb, FW_ZB + F_PP - F_ZLA), pn = tl_ld(tb, FW_ZB + F_PN - F_ZLA);
      const double zpp = tl_ld(tb, FW_ZB + F_ZPP - F_ZLA), zpn = tl_ld(tb, FW_ZB + F_ZPN - F_ZLA);
      Move mv;
      mv.build(pp, pn, zpp, zpn, u - zm[6], wdc, mu, ls);
      double dp, dn;
      mv.steps(dv, dp, dn);
      const double ip = mv.ip, in_ = mv.in_;
      rp.push(-dp, pp); rp.push(-dn, pn);
      rz.push(-((mu - zpp * dp) * ip - zpp), zpp);
      rz.push(-((mu - zpn * dn) * in_ - zpn), zpn);
      dphi += (wdc - mu * ip) * dp + (wdc - mu * in_) * dn;
      dxmax = dmax(dxmax, dmax(fabs(dp), fabs(dn)) * dmin(1.0, dmax(ip, in_)));
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) { ds[i] = xi[i]; WS_AT(sp, F_DS + i) = xi[i]; dxmax = dmax(dxmax, fabs(xi[i])); }
    ds[6] = xi[6];
    const double du = xi[6];
    WS_AT(sp, F_DU) = du;
    dxmax = dmax(dxmax, fabs(du));
#pragma unroll
    for (int i = 0; i < 7; ++i) zm[i] = zn[i];
    const double da = ds[4];
    const double dLa = zn[4], dUa = P.a_ub - zn[4], dLu = u + P.u_ub, dUu = P.u_ub - u;
    rp.push(-da, dLa); rp.push(da, dUa); rp.push(-du, dLu); rp.push(du, dUu);
    const double zla = tl_ld(tb, FW_ZB + 0), zua = tl_ld(tb, FW_ZB + 1);
    const double zlu = tl_ld(tb, FW_ZB + 2), zuu = tl_ld(tb, FW_ZB + 3);
    double rLa, rUa, rLu, rUu;
    recip4(dLa, dUa, dLu, dUu, rLa, rUa, rLu, rUu);
    const double d1 = (mu - zla * da) * rLa - zla;
    const double d2 = (mu + zua * da) * rUa - zua;
    const double d3 = (mu - zlu * du) * rLu - zlu;
    const double d4 = (mu + zuu * du) * rUu - zuu;
    rz.push(-d1, zla); rz.push(-d2, zua); rz.push(-d3, zlu); rz.push(-d4, zuu);
    dphi += mu * ((rUa - rLa) * da + (rUu - rLu) * du);
  }
  {
    Terminal T;
    terminal_eval(P, zm[0], zm[1], zm[2], zm[3], T);
    const double rinv = 1.0 / T.rT;
    const double dg1 = T.Yb * rinv * ds[0] + zm[2] * rinv * ds[2];
    const double dg2 = 2.0 * zm[1] * ds[1] + 2.0 * zm[3] * ds[3];
    const double dg3 = zm[1] * ds[0] + T.Yb * ds[1] + zm[3] * ds[2] + zm[2] * ds[3];
    ts.dtf = dtf;
    ts.dsg1 = dg1 + cw * (T.g1 - c0.sg1);
    ts.dsg2 = dg2 + cw * (T.g2 - c0.sg2);
    ts.dnu3 = (dg3 + cw * T.g3) / O.delta_c;
    if (!ls) {
      ts.dzs1 = mu / c0.sg1 - c0.zs1 - c0.zs1 / c0.sg1 * ts.dsg1;
      ts.dzs2 = mu / c0.sg2 - c0.zs2 - c0.zs2 / c0.sg2 * ts.dsg2;
    } else {
      ts.dzs1 = 0.0; ts.dzs2 = 0.0;
    }
    const double dLt = tf, dUt = P.tf_ub - tf;
    ts.dzLt = mu / dLt - c0.zLt - c0.zLt / dLt * dtf;
    ts.dzUt = mu / dUt - c0.zUt + c0.zUt / dUt * dtf;
    rp.push(-ts.dsg1, c0.sg1); rp.push(-ts.dsg2, c0.sg2); rp.push(-dtf, dLt); rp.push(dtf, dUt);
    rz.push(-ts.dzs1, c0.zs1); rz.push(-ts.dzs2, c0.zs2); rz.push(-ts.dzLt, c0.zLt); rz.push(-ts.dzUt, c0.zUt);
    dphi += (O.obj_scale - mu / dLt + mu / dUt) * dtf - mu / c0.sg1 * ts.dsg1 - mu / c0.sg2 * ts.dsg2;
    dxmax = dmax(dxmax, dmax(fabs(ts.dsg1), fabs(ts.dsg2)));
  }
  si.a_max = (rp.n > tau * rp.d) ? tau * rp.d / rp.n : 1.0;
  si.a_z = (rz.n > tau * rz.d) ? tau * rz.d / rz.n : 1.0;
  si.dphi = dphi; si.dxmax = dxmax;
}

}  // namespace dc

// Sweeps policy of the 8-state (DCOST) formulation.
struct Sweeps8 {
  enum : int { NFIELDS = dc::N_FIELDS, NITER = dc::N_ITER, FZ = dc::F_Z, FU = dc::F_U, FLAM = dc::F_LAM, FZLA = dc::F_ZLA,
               REFROWS = dc::REF_ROWS, MOVE_TERM = 1, LANES_PER_PROBLEM = 1, STORES_REF = 0 };
  LM_HD static int n_eq(const Ws&, int N) { return 7 * N + 3; }
  LM_HD static int n_bd(const Ws&, int N) { return 6 * N + 4; }
  LM_HD static bool backward(const Params& P, const Mesh& M, const Options& O, const Ws& W, int src, const Scal& c0,
                             double mu, double dw, bool ls, double* dtf) {
    return dc::riccati_backward(P, M, O, W, src, c0, mu, dw, ls, dtf);
  }
  LM_HD static void forward(const Params& P, const Mesh& M, const Options& O, const Ws& W, int src, const Scal& c0,
                            double mu, double tau, double dtf, bool ls, TermStep& ts, StepInfo& si) {
    dc::riccati_forward(P, M, O, W, src, c0, mu, tau, dtf, ls, ts, si);
  }
  LM_HD static void eval(const Params& P, const Mesh& M, const Options& O, const Ws& W, int src, int dst,
                         const Scal& c0, const TermStep& ts, double mu, double dw, double alpha, double alpha_z,
                         double alpha_lam, int mode, Scal& t, double* pimax) {
    dc::eval_pass(P, M, O, W, src, dst, c0, ts, mu, dw, alpha, alpha_z, alpha_lam, mode, t, pimax);
  }
  // start points (ascent_ipm.cuh: start_rollout, ...): node k into the 8-state rows; node 0 pinned at zero, MV(0) = 0
  LM_HD static void store_node(const Ws& W, int k, const double* x) {
    double* sp = W.stage(k);
#pragma unroll
    for (int f = 0; f < NODE_N; ++f) WS_AT(sp, f) = x[f];
#pragma unroll
    for (int i = 0; i < dc::N_STEP; ++i) WS_AT(sp, dc::R_STEP + i) = 0.0;
  }
  LM_HD static void zero_node0(const Ws& W) {
    double* s0 = W.stage(0);
#pragma unroll
    for (int i = 0; i < 7; ++i) { WS_AT(s0, dc::F_Z + i) = 0.0; WS_AT(s0, dc::N_ITER + dc::F_Z + i) = 0.0; WS_AT(s0, dc::F_DS + i) = 0.0; }
  }
  LM_HD static void node(const Ws& W, int cur, int k, double* x, double* lam) { ws_node<Sweeps8>(W, cur, k, x, lam); }
  LM_HD static void node_duals(const Ws& W, int cur, int k, double* d) { ws_node_duals<Sweeps8>(W, cur, k, d); }
  LM_HD static void remerit(const Mesh&, const Options&, const Ws&, int, double, Scal&) {}
};

}  // namespace lmato
