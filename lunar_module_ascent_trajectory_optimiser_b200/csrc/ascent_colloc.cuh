// Higher-order collocation on the device: GEKKO NODES = 3 ... 6 (LO:25; SURVEY Appendix B.2).
//
// APMonitor's transcription for NODES = n: every mesh step carries m = n-1 collocation points (Lobatto
// points tau_1 < ... < tau_m = 1, the last one is the mesh node) and the rows
//     z_i - z_0 - h T tf sum_j N_ij F(z_j, u, t_j) = 0,   i = 1..m        (z_0 = the previous mesh node)
// with the MV held over the step (MV_TYPE = 0, LO:29).  NODES = 2 (m = 1, N = [1]) is backward Euler, which the
// two tuned kernels solve; this header is the general path, organised like ascent_coop.cuh:
//   * STAGE-PARALLEL (GP lanes per problem): at every trial point each step is condensed on its own.  Its
//     6m x 6m Jacobian E_k = I - h T tf (N (x) I) blkdiag(F_z(z_j)) is LU-factorised (partial pivoting, in the
//     workspace) and the step's unknowns become an affine map of what couples the steps,
//         (dz_1 .. dz_m) = Phi_k (dz_0, du, dtf, 1),                       Phi_k: 6m x 9,
//     and the step's Lagrangian Hessian (block diagonal over the points, plus the tf / u couplings) becomes the
//     9 x 9 matrix Qh_k = Phibar^T H Phibar in those coordinates;
//   * SEQUENTIAL (one lane): a dense Riccati recursion on the 7 coupling unknowns (the six states of the mesh
//     node and tf) with the scalar control du; inertia from its pivots as before; the value function of every
//     node is kept, because the costate sigma_k = sum_i pi_{k,i} that links the steps' multipliers is its gradient;
//   * STAGE-PARALLEL again: the steps of all collocation points (Phi_k times the coupling step), bound
//     multipliers, fraction-to-boundary ratios, and the new row multipliers from E_k^T pi_k = e_m (x) sigma_{k+1}
//     - (H d + g) with the stored LU factors.
// Same IPM driver (ipm_iterate_t), same model functions (ascent_model.cuh), same terminal rows.  The l1 move
// term (LO:99) is not carried here (the oracle drops it for NODES > 2 as well).  GP = 1 is the host build.
#pragma once
#include "ascent_coop.cuh"

namespace lmato {
namespace colloc {

constexpr int MAXM = 5;              // NODES <= 6
constexpr int MAXN6 = 6 * MAXM;

// Collocation rule of one NODES value (computed on the host, include/lmato_b200.h: lmato_create).
struct Coll {
  int m;                             // points per step = NODES - 1
  double N[MAXM][MAXM];              // h N f_{1..m} = z_{1..m} - z_0
  double tau[MAXM];                  // tau_i in (0, 1], tau_m = 1
};

using coop::Grp;

// record sizes / offsets (doubles) for m points per step
struct Lay {
  int m, n6;
  int XR, DR, MR;
  // X: z[m][6] | u | lam[m][6] | zla[m] | zua[m] | zlu | zuu
  int x_u, x_lam, x_zla, x_zua, x_zlu, x_zuu;
  // D: dz[m][6] | du | pi[m][6] | xprev[6] (step of the previous mesh node)
  int d_du, d_pi, d_xp;
  // M: Phi[6m][9] | Qh[81] | beta[9] | Gd[81] | LU[6m][6m] | piv[6m] | Hp[m][16] (per-point Hessian pieces) | sc[4]
  int m_qh, m_beta, m_gd, m_lu, m_piv, m_hp, m_sc;
  LM_HD void init(int m_) {
    m = m_; n6 = 6 * m;
    x_u = n6; x_lam = n6 + 1; x_zla = 2 * n6 + 1; x_zua = x_zla + m; x_zlu = x_zua + m; x_zuu = x_zlu + 1;
    XR = x_zuu + 1;
    d_du = n6; d_pi = n6 + 1; d_xp = 2 * n6 + 1; DR = d_xp + 6;
    m_qh = n6 * 9; m_beta = m_qh + 81; m_gd = m_beta + 9; m_lu = m_gd + 81; m_piv = m_lu + n6 * n6;
    m_hp = m_piv + n6; m_sc = m_hp + 16 * m; MR = m_sc + 4;
  }
};
constexpr int KR_ = 8, PR_ = 64;     // feedback law (x[6], dtf, 1) ; value function of a node: 8 x 8 homogeneous
enum : int { H_00 = 0, H_02, H_22, H_04, H_24, H_44, H_D, H_T0 /* 6: z-tf cross */, H_TT = H_T0 + 6, H_G4A, H_G4B, H_N = 16 };
enum : int { SC_RU = 0, SC_SIG, SC_RUA, SC_RUB };      // per-step u pieces: Sigma_u, u-tf cross, gradient A + mu B

struct Nws {
  double* base;
  int N1;
  Lay L;
  const Coll* C;         // the collocation rule (shared by the whole launch)
  int g;                 // lane inside the group (0 .. GP-1)
  unsigned mask;
  mutable double dw;
  mutable double pimax;
  mutable int ls_flag;
  LM_HD long per_stage() const { return 2L * L.XR + L.DR + 2L * L.MR + KR_ + PR_; }
  LM_HD double* X(int buf, int k) const { return base + ((long)buf * N1 + k) * L.XR; }
  LM_HD double* D(int k) const { return base + 2L * N1 * L.XR + (long)k * L.DR; }
  LM_HD double* Mo(int buf, int k) const { return base + 2L * N1 * L.XR + (long)N1 * L.DR + ((long)buf * N1 + k) * L.MR; }
  LM_HD double* K(int k) const { return base + 2L * N1 * L.XR + (long)N1 * L.DR + 2L * N1 * L.MR + (long)k * KR_; }
  LM_HD double* Pn(int k) const { return base + 2L * N1 * L.XR + (long)N1 * L.DR + 2L * N1 * L.MR + (long)N1 * KR_ + (long)k * PR_; }
};
LM_HD long colloc_doubles_per_problem(int nt, int m) {
  Lay L; L.init(m);
  return (long)nt * (2L * L.XR + L.DR + 2L * L.MR + KR_ + PR_);
}

// dense LU with partial pivoting, in place (n <= 30), and the two solves
LM_HD bool lu_factor(double* A, double* piv, int n) {
  for (int c = 0; c < n; ++c) {
    int p = c; double best = fabs(A[c * n + c]);
    for (int r = c + 1; r < n; ++r) { const double v = fabs(A[r * n + c]); if (v > best) { best = v; p = r; } }
    piv[c] = (double)p;
    if (!(best > 0.0)) return false;
    if (p != c) for (int j = 0; j < n; ++j) { const double t = A[c * n + j]; A[c * n + j] = A[p * n + j]; A[p * n + j] = t; }
    const double inv = 1.0 / A[c * n + c];
    for (int r = c + 1; r < n; ++r) {
      const double l = A[r * n + c] * inv;
      A[r * n + c] = l;
      if (l != 0.0) for (int j = c + 1; j < n; ++j) A[r * n + j] -= l * A[c * n + j];
    }
  }
  return true;
}
// b (stride ldb, one column) <- A^-1 b
LM_HD void lu_solve(const double* A, const double* piv, int n, double* b, int ldb) {
  for (int c = 0; c < n; ++c) { const int p = (int)piv[c]; if (p != c) { const double t = b[c * ldb]; b[c * ldb] = b[p * ldb]; b[p * ldb] = t; } }
  for (int r = 1; r < n; ++r) { double s = b[r * ldb]; for (int j = 0; j < r; ++j) s -= A[r * n + j] * b[j * ldb]; b[r * ldb] = s; }
  for (int r = n - 1; r >= 0; --r) { double s = b[r * ldb]; for (int j = r + 1; j < n; ++j) s -= A[r * n + j] * b[j * ldb]; b[r * ldb] = s / A[r * n + r]; }
}
// b <- A^-T b      (P A = L U  =>  A^T = U^T L^T P)
LM_HD void lu_solve_t(const double* A, const double* piv, int n, double* b) {
  for (int r = 0; r < n; ++r) { double s = b[r]; for (int j = 0; j < r; ++j) s -= A[j * n + r] * b[j]; b[r] = s / A[r * n + r]; }
  for (int r = n - 2; r >= 0; --r) { double s = b[r]; for (int j = r + 1; j < n; ++j) s -= A[j * n + r] * b[j]; b[r] = s; }
  for (int c = n - 1; c >= 0; --c) { const int p = (int)piv[c]; if (p != c) { const double t = b[c]; b[c] = b[p]; b[p] = t; } }
}

// ---------------------------------------------------------------------------------------
// Condense one step at one point of the iteration: E, LU, Phi, Qh, beta, Gd, per-point Hessian pieces.
// Returns the step's defects in `cdef` (6m) -- evaluated before E is overwritten by its factors.
// ---------------------------------------------------------------------------------------
LM_HD void build_step(const Params& P, const Coll& C, const Lay& L, double hk, double tau0, double tf, bool ls,
                      const double* x /* X record */, const double* z0 /* previous mesh node, 6 */, double* mrec,
                      double* cdef /* 6m, may be null */, double* Fpt /* 6m: F(z_j), may be null */) {
  const int m = L.m, n6 = L.n6;
  const double kap = hk * P.T;
  const double al = kap * tf;
  double* Phi = mrec;                 // 6m x 9, first used as the right-hand sides
  double* E = mrec + L.m_lu;
  double* piv = mrec + L.m_piv;
  double* Hp = mrec + L.m_hp;
  double* sc = mrec + L.m_sc;
  const double u = x[L.x_u];
  for (int i = 0; i < n6 * n6; ++i) E[i] = 0.0;
  for (int i = 0; i < n6; ++i) E[i * n6 + i] = 1.0;
  // per point: dynamics, first derivatives; E blocks; e column pieces
  double Fj[MAXM][6], Ftf[MAXM][6];        // F(z_j) and d F / d tf (through the mass)
  for (int j = 0; j < m; ++j) {
    const double* z = x + 6 * j;
    const double tj = tau0 + C.tau[j] * hk;
    const double taum = P.mT * tj;
    Accel1 f;
    accel_first(P, z[0], z[2], z[4], taum * tf, f);
    Fj[j][0] = z[1]; Fj[j][1] = f.ay; Fj[j][2] = z[3]; Fj[j][3] = f.ax; Fj[j][4] = z[5]; Fj[j][5] = P.asc * u;
    Ftf[j][0] = 0; Ftf[j][1] = f.ay_m * taum; Ftf[j][2] = 0; Ftf[j][3] = f.ax_m * taum; Ftf[j][4] = 0; Ftf[j][5] = 0;
    for (int i = 0; i < m; ++i) {
      const double cN = al * C.N[i][j];
      double* Eb = E + (6 * i) * n6 + 6 * j;
      Eb[0 * n6 + 1] -= cN;
      Eb[1 * n6 + 0] -= cN * f.ay_y; Eb[1 * n6 + 2] -= cN * f.ay_x; Eb[1 * n6 + 4] -= cN * f.ay_a;
      Eb[2 * n6 + 3] -= cN;
      Eb[3 * n6 + 0] -= cN * f.ax_y; Eb[3 * n6 + 2] -= cN * f.ax_x; Eb[3 * n6 + 4] -= cN * f.ax_a;
      Eb[4 * n6 + 5] -= cN;
    }
    // Hessian pieces of this point: multiplier of F(z_j) is lamt_j = sum_i N_ij lam_i
    double lamt[6] = {0, 0, 0, 0, 0, 0};
    for (int i = 0; i < m; ++i)
      for (int r = 0; r < 6; ++r) lamt[r] += C.N[i][j] * x[L.x_lam + 6 * i + r];
    StageJac J;
    J.al = al;
    StageQ q;
    stage_hessian(P, f, J, kap, taum, lamt, z[4], u, x[L.x_zla + j], x[L.x_zua + j], x[L.x_zlu], x[L.x_zuu], 1.0, 0.0, ls, q);
    double* h = Hp + H_N * j;
    h[H_00] = q.q00; h[H_02] = q.q02; h[H_22] = q.q22; h[H_04] = q.q04; h[H_24] = q.q24; h[H_44] = q.q44; h[H_D] = q.d;
    h[H_T0 + 0] = q.q06; h[H_T0 + 1] = q.q16; h[H_T0 + 2] = q.q26; h[H_T0 + 3] = q.q36; h[H_T0 + 4] = q.q46; h[H_T0 + 5] = q.q56;
    h[H_TT] = q.q66;
    h[H_G4A] = ls ? q.q4 : 0.0; h[H_G4B] = ls ? 0.0 : q.q4;
    if (j == 0) { sc[SC_RU] = q.R; sc[SC_RUA] = ls ? q.r : 0.0; sc[SC_RUB] = ls ? 0.0 : q.r; sc[SC_SIG] = 0.0; }
    sc[SC_SIG] += q.sig;
  }
  // right-hand sides: [1 (x) I6 | b | e | -c]
  for (int i = 0; i < m; ++i) {
    double NF[6] = {0, 0, 0, 0, 0, 0}, NFt[6] = {0, 0, 0, 0, 0, 0};
    double rs = 0.0;
    for (int j = 0; j < m; ++j) {
      rs += C.N[i][j];
      for (int r = 0; r < 6; ++r) { NF[r] += C.N[i][j] * Fj[j][r]; NFt[r] += C.N[i][j] * Ftf[j][r]; }
    }
    for (int r = 0; r < 6; ++r) {
      double* row = Phi + (6 * i + r) * 9;
      for (int c = 0; c < 6; ++c) row[c] = (c == r) ? 1.0 : 0.0;
      row[6] = (r == 5) ? al * rs * P.asc : 0.0;                       // d / d u
      row[7] = kap * (NF[r] + tf * NFt[r]);                            // d / d tf
      const double cd = x[6 * i + r] - z0[r] - al * NF[r];
      row[8] = ls ? 0.0 : -cd;
      if (cdef) cdef[6 * i + r] = cd;
    }
  }
  if (Fpt) for (int j = 0; j < m; ++j) for (int r = 0; r < 6; ++r) Fpt[6 * j + r] = Fj[j][r];
  lu_factor(E, piv, n6);
  for (int c = 0; c < 9; ++c) lu_solve(E, piv, n6, Phi + c, 9);
  // Qh = Phibar^T H Phibar (9 x 9, homogeneous), beta = mu-coefficient of its affine column, Gd = Phi^T Phi + e6 e6^T
  double* Qh = mrec + L.m_qh;
  double* beta = mrec + L.m_beta;
  double* Gd = mrec + L.m_gd;
  for (int i = 0; i < 81; ++i) { Qh[i] = 0.0; Gd[i] = 0.0; }
  for (int c = 0; c < 9; ++c) beta[c] = 0.0;
  for (int j = 0; j < m; ++j) {
    const double* h = Hp + H_N * j;
    const double* Pj = Phi + (6 * j) * 9;
    for (int c = 0; c < 9; ++c) {
      const double p0 = Pj[0 * 9 + c], p1 = Pj[1 * 9 + c], p2 = Pj[2 * 9 + c], p3 = Pj[3 * 9 + c], p4 = Pj[4 * 9 + c], p5 = Pj[5 * 9 + c];
      // T = Hzz Phi_j (column c)
      const double t0 = h[H_00] * p0 + h[H_02] * p2 + h[H_04] * p4;
      const double t1 = h[H_D] * p1;
      const double t2 = h[H_02] * p0 + h[H_22] * p2 + h[H_24] * p4;
      const double t3 = h[H_D] * p3;
      const double t4 = h[H_04] * p0 + h[H_24] * p2 + h[H_44] * p4;
      const double t5 = h[H_D] * p5;
      for (int r = 0; r < 9; ++r) {
        Qh[r * 9 + c] += Pj[0 * 9 + r] * t0 + Pj[1 * 9 + r] * t1 + Pj[2 * 9 + r] * t2 + Pj[3 * 9 + r] * t3 + Pj[4 * 9 + r] * t4 + Pj[5 * 9 + r] * t5;
        Gd[r * 9 + c] += Pj[0 * 9 + r] * p0 + Pj[1 * 9 + r] * p1 + Pj[2 * 9 + r] * p2 + Pj[3 * 9 + r] * p3 + Pj[4 * 9 + r] * p4 + Pj[5 * 9 + r] * p5;
      }
      // z - tf cross terms and the gradient of the angle barrier
      const double ht = h[H_T0 + 0] * p0 + h[H_T0 + 1] * p1 + h[H_T0 + 2] * p2 + h[H_T0 + 3] * p3 + h[H_T0 + 4] * p4 + h[H_T0 + 5] * p5;
      Qh[7 * 9 + c] += ht; Qh[c * 9 + 7] += ht;
      Qh[8 * 9 + c] += h[H_G4A] * p4; Qh[c * 9 + 8] += h[H_G4A] * p4;
      beta[c] += h[H_G4B] * p4;
    }
    Qh[7 * 9 + 7] += h[H_TT];
  }
  Qh[6 * 9 + 6] += sc[SC_RU];
  Qh[6 * 9 + 7] += sc[SC_SIG]; Qh[7 * 9 + 6] += sc[SC_SIG];
  Qh[6 * 9 + 8] += sc[SC_RUA]; Qh[8 * 9 + 6] += sc[SC_RUA];
  beta[6] += sc[SC_RUB];
  Gd[6 * 9 + 6] += 1.0;
}

LM_HD double xrec_u_prev(const Nws& W, int buf, int k) { return k > 0 ? W.X(buf, k)[W.L.x_u] : 0.0; }

template <int GP>
LM_SWEEP void colloc_build(const Params& P, const Mesh& M, const Coll& C, const Nws& W, int buf, double tf, bool ls) {
  const int N = M.N, m = W.L.m;
  for (int k = 1 + W.g; k <= N; k += GP) {
    double z0[6];
    const double* xp = W.X(buf, k - 1) + 6 * (m - 1);
    for (int r = 0; r < 6; ++r) z0[r] = k > 1 ? xp[r] : 0.0;
    build_step(P, C, W.L, M.h[k], M.tau[k - 1], tf, ls, W.X(buf, k), z0, W.Mo(buf, k), nullptr, nullptr);
  }
  Grp<GP>::sync(W.mask);
}

// ---------------------------------------------------------------------------------------
// backward: dense Riccati on (x = step of the mesh node (6), dtf), control du, homogeneous 9 x 9 forms.
// One lane; returns false on wrong inertia.
// ---------------------------------------------------------------------------------------
LM_HD bool colloc_backward_seq(const Params& P, const Mesh& M, const Options& O, const Nws& W, int src, const Scal& c0,
                               double mu, double dw, bool ls, double* dtf_out) {
  const int N = M.N, m = W.L.m;
  // value function of a node, homogeneous on (x[6], dtf, 1): 8 x 8 symmetric
  double V[8][8];
  for (int i = 0; i < 8; ++i) for (int j = 0; j < 8; ++j) V[i][j] = 0.0;
  {
    const double* zn = W.X(src, N) + 6 * (m - 1);
    TermQP tq;
    terminal_qp(P, O, c0, zn, mu, dw, ls, tq);
    for (int i = 0; i < 4; ++i) { for (int j = 0; j < 4; ++j) V[i][j] = tq.H[i][j]; V[i][7] = tq.g[i]; V[7][i] = tq.g[i]; }
    V[6][6] = tq.H66; V[6][7] = tq.g6; V[7][6] = tq.g6;
  }
  for (int k = N; k >= 1; --k) {
    double* pn = W.Pn(k);
    for (int i = 0; i < 8; ++i) for (int j = 0; j < 8; ++j) pn[i * 8 + j] = V[i][j];
    const double* mrec = W.Mo(src, k);
    const double* Psi = mrec + (6 * (m - 1)) * 9;       // last six rows of Phi: the mesh node as a function of (x, du, dtf, 1)
    const double* Qh = mrec + W.L.m_qh;
    const double* beta = mrec + W.L.m_beta;
    const double* Gd = mrec + W.L.m_gd;
    // M9 = Qh + mu sym(e8 beta^T) + dw Gd + Psibar^T V Psibar,  Psibar = [Psi; e7^T (dtf); e8^T (1)]
    double VP[8][9];
    for (int i = 0; i < 8; ++i)
      for (int c = 0; c < 9; ++c) {
        double s = 0.0;
        for (int j = 0; j < 6; ++j) s += V[i][j] * Psi[j * 9 + c];
        if (c == 7) s += V[i][6];
        if (c == 8) s += V[i][7];
        VP[i][c] = s;
      }
    double M9[9][9];
    for (int r = 0; r < 9; ++r)
      for (int c = 0; c < 9; ++c) {
        double s = Qh[r * 9 + c] + dw * Gd[r * 9 + c];
        if (r == 8) s += mu * beta[c];
        if (c == 8) s += mu * beta[r];
        for (int j = 0; j < 6; ++j) s += Psi[j * 9 + r] * VP[j][c];
        if (r == 7) s += VP[6][c];
        if (r == 8) s += VP[7][c];
        M9[r][c] = s;
      }
    const double Ruu = M9[6][6];
    if (!(Ruu > 0.0) || !(Ruu < 1e300)) return false;
    const double Rinv = 1.0 / Ruu;
    double* kk = W.K(k);
    static const int idx[8] = {0, 1, 2, 3, 4, 5, 7, 8};
    double row6[8];
    for (int a = 0; a < 8; ++a) { row6[a] = 0.5 * (M9[6][idx[a]] + M9[idx[a]][6]); kk[a] = -row6[a] * Rinv; }
    for (int a = 0; a < 8; ++a)
      for (int b = 0; b <= a; ++b) {
        const double v = 0.5 * (M9[idx[a]][idx[b]] + M9[idx[b]][idx[a]]) - row6[a] * row6[b] * Rinv;
        V[a][b] = v; V[b][a] = v;
      }
  }
  if (!(V[6][6] > 0.0)) return false;
  *dtf_out = -V[6][7] / V[6][6];
  return true;
}

template <int GP>
LM_SWEEP bool colloc_backward(const Params& P, const Mesh& M, const Options& O, const Nws& W, int src, const Scal& c0,
                              double mu, double dw, bool ls, double* dtf_out) {
  W.dw = dw;
  double dtf = 0.0;
  int ok = 0;
  if (W.g == 0) ok = colloc_backward_seq(P, M, O, W, src, c0, mu, dw, ls, &dtf) ? 1 : 0;
  Grp<GP>::sync(W.mask);
  if (GP > 1) { ok = Grp<GP>::bcast_int(W.mask, ok, 0); dtf = Grp<GP>::bcast(W.mask, dtf, 0); }
  *dtf_out = dtf;
  return ok != 0;
}

// ---------------------------------------------------------------------------------------
// forward: (1) coupling steps, one lane; (2) stage-parallel: steps of all points, multipliers, ratios
// ---------------------------------------------------------------------------------------
template <int GP>
LM_SWEEP void colloc_forward(const Params& P, const Mesh& M, const Options& O, const Coll& C, const Nws& W, int src,
                             const Scal& c0, double mu, double tau, double dtf, bool ls, TermStep& ts, StepInfo& si) {
  const int N = M.N, m = W.L.m, n6 = W.L.n6;
  const Lay& L = W.L;
  const double dw = W.dw;
  const double cw = ls ? 0.0 : 1.0;
  if (W.g == 0) {
    double x[6] = {0, 0, 0, 0, 0, 0};
    for (int k = 1; k <= N; ++k) {
      const double* kk = W.K(k);
      double du = kk[7] + kk[6] * dtf;
      for (int j = 0; j < 6; ++j) du += kk[j] * x[j];
      double* d = W.D(k);
      for (int j = 0; j < 6; ++j) d[L.d_xp + j] = x[j];
      d[L.d_du] = du;
      const double* Psi = W.Mo(src, k) + (6 * (m - 1)) * 9;
      double xn[6];
      for (int r = 0; r < 6; ++r) {
        double s = Psi[r * 9 + 6] * du + Psi[r * 9 + 7] * dtf + Psi[r * 9 + 8];
        for (int j = 0; j < 6; ++j) s += Psi[r * 9 + j] * x[j];
        xn[r] = s;
      }
      for (int r = 0; r < 6; ++r) x[r] = xn[r];
    }
  }
  Grp<GP>::sync(W.mask);
  double dphi = 0.0, dxmax = 0.0, pimax = 0.0;
  RatioMax rp, rz;
  rp.init(); rz.init();
  for (int k = 1 + W.g; k <= N; k += GP) {
    const double* x = W.X(src, k);
    double* d = W.D(k);
    const double* mrec = W.Mo(src, k);
    const double* Phi = mrec;
    const double* Hp = mrec + L.m_hp;
    const double* sc = mrec + L.m_sc;
    const double du = d[L.d_du];
    // steps of all collocation points
    for (int i = 0; i < n6; ++i) {
      const double* row = Phi + i * 9;
      double s = row[6] * du + row[7] * dtf + row[8];
      for (int j = 0; j < 6; ++j) s += row[j] * d[L.d_xp + j];
      d[i] = s;
      dxmax = dmax(dxmax, fabs(s));
    }
    dxmax = dmax(dxmax, fabs(du));
    // bounds: the angle of every point, the control of the step
    const double u = x[L.x_u];
    for (int j = 0; j < m; ++j) {
      const double a = x[6 * j + 4], da = d[6 * j + 4];
      const double dLa = a, dUa = P.a_ub - a;
      const double zla = x[L.x_zla + j], zua = x[L.x_zua + j];
      rp.push(-da, dLa); rp.push(da, dUa);
      const double rLa = 1.0 / dLa, rUa = 1.0 / dUa;
      rz.push(-((mu - zla * da) * rLa - zla), zla);
      rz.push(-((mu + zua * da) * rUa - zua), zua);
      dphi += mu * (rUa - rLa) * da;
    }
    {
      const double dLu = u + P.u_ub, dUu = P.u_ub - u;
      const double zlu = x[L.x_zlu], zuu = x[L.x_zuu];
      rp.push(-du, dLu); rp.push(du, dUu);
      const double rLu = 1.0 / dLu, rUu = 1.0 / dUu;
      rz.push(-((mu - zlu * du) * rLu - zlu), zlu);
      rz.push(-((mu + zuu * du) * rUu - zuu), zuu);
      dphi += mu * (rUu - rLu) * du;
    }
    // new row multipliers: E^T pi = e_m (x) sigma_{k+1} - (H d + g),  sigma_{k+1} = -(grad of the node's value function)
    double rhs[MAXN6];
    for (int j = 0; j < m; ++j) {
      const double* h = Hp + H_N * j;
      const double* dz = d + 6 * j;
      const double dd = h[H_D] + dw;
      rhs[6 * j + 0] = -((h[H_00] + dw) * dz[0] + h[H_02] * dz[2] + h[H_04] * dz[4] + h[H_T0 + 0] * dtf);
      rhs[6 * j + 1] = -(dd * dz[1] + h[H_T0 + 1] * dtf);
      rhs[6 * j + 2] = -(h[H_02] * dz[0] + (h[H_22] + dw) * dz[2] + h[H_24] * dz[4] + h[H_T0 + 2] * dtf);
      rhs[6 * j + 3] = -(dd * dz[3] + h[H_T0 + 3] * dtf);
      rhs[6 * j + 4] = -(h[H_04] * dz[0] + h[H_24] * dz[2] + (h[H_44] + dw) * dz[4] + h[H_T0 + 4] * dtf + h[H_G4A] + mu * h[H_G4B]);
      rhs[6 * j + 5] = -(dd * dz[5] + h[H_T0 + 5] * dtf);
    }
    {
      const double* V = W.Pn(k);             // value function of node k on (x_k, dtf, 1)
      const double* xk = d + 6 * (m - 1);
      for (int r = 0; r < 6; ++r) {
        double s = V[r * 8 + 6] * dtf + V[r * 8 + 7];
        for (int j = 0; j < 6; ++j) s += V[r * 8 + j] * xk[j];
        rhs[6 * (m - 1) + r] -= s;
      }
    }
    lu_solve_t(mrec + L.m_lu, mrec + L.m_piv, n6, rhs);
    for (int i = 0; i < n6; ++i) { d[L.d_pi + i] = rhs[i]; if (ls) pimax = dmax(pimax, fabs(rhs[i])); }
    (void)sc;
  }
  dphi = Grp<GP>::sum(W.mask, dphi);
  dxmax = dmax(Grp<GP>::max(W.mask, dxmax), fabs(dtf));
  pimax = Grp<GP>::max(W.mask, pimax);
  Grp<GP>::ratio_max(W.mask, rp);
  Grp<GP>::ratio_max(W.mask, rz);
  Grp<GP>::sync(W.mask);
  // terminal slacks and multipliers (every lane)
  {
    const double* zm = W.X(src, N) + 6 * (m - 1);
    const double* ds = W.D(N) + 6 * (m - 1);
    const double tf = c0.tf;
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
  W.pimax = pimax;
}

// ---------------------------------------------------------------------------------------
// evaluation pass, stage-parallel: trial point, merit and KKT-error terms, and the condensed model of the
// trial point (M records of buffer dst)
// ---------------------------------------------------------------------------------------
template <int GP>
LM_SWEEP void colloc_eval(const Params& P, const Mesh& M, const Options& O, const Coll& C, const Nws& W, int src, int dst,
                          const Scal& c0, const TermStep& ts, double mu, double alpha, double alpha_z, double alpha_lam,
                          Scal& t) {
  const int N = M.N, m = W.L.m, n6 = W.L.n6;
  const Lay& L = W.L;
  const double tf0 = c0.tf, dtf = ts.dtf;
  const double tf = tf0 + alpha * dtf;
  t.tf = tf;
  t.sg1 = c0.sg1 + alpha * ts.dsg1;
  t.sg2 = c0.sg2 + alpha * ts.dsg2;
  t.nu3 = c0.nu3 + alpha_lam * ts.dnu3;
  t.zs1 = c0.zs1 + alpha_z * ts.dzs1;
  t.zs2 = c0.zs2 + alpha_z * ts.dzs2;
  t.zLt = c0.zLt + alpha_z * ts.dzLt;
  t.zUt = c0.zUt + alpha_z * ts.dzUt;
  bool bad0 = false;
  double sumlog0, cmin0, cmax0, sz0, slam0, gtf0;
  {
    const double dLt = tf, dUt = P.tf_ub - tf;
    if (!(t.sg1 > 0 && t.sg2 > 0 && dLt > 0 && dUt > 0)) bad0 = true;
    t.zs1 = clip_mult(t.zs1, t.sg1, mu);
    t.zs2 = clip_mult(t.zs2, t.sg2, mu);
    t.zLt = clip_mult(t.zLt, dLt, mu);
    t.zUt = clip_mult(t.zUt, dUt, mu);
    sumlog0 = log((t.sg1 * t.sg2) * (dLt * dUt));
    const double q1 = t.sg1 * t.zs1, q2 = t.sg2 * t.zs2, q3 = dLt * t.zLt, q4 = dUt * t.zUt;
    cmin0 = dmin(dmin(q1, q2), dmin(q3, q4));
    cmax0 = dmax(dmax(q1, q2), dmax(q3, q4));
    sz0 = t.zs1 + t.zs2 + t.zLt + t.zUt;
    slam0 = t.zs1 + t.zs2 + fabs(t.nu3);
    gtf0 = O.obj_scale - t.zLt + t.zUt;
  }
  double theta = 0, prim = 0, dual = 0, sumlog = 0, cmin = 1e300, cmax = 0, slam = 0, sz = 0, gtf = 0;
  int bad = 0;
  // pass 1: the trial iterate of every step (the defects of step k need the trial mesh node k-1, the dual residual
  // the trial multipliers of step k+1)
  for (int k = 1 + W.g; k <= N; k += GP) {
    const double* xo = W.X(src, k);
    const double* d = W.D(k);
    double* xn = W.X(dst, k);
    for (int i = 0; i < n6; ++i) xn[i] = fma(alpha, d[i], xo[i]);
    const double u_old = xo[L.x_u], du = d[L.d_du];
    const double u = fma(alpha, du, u_old);
    xn[L.x_u] = u;
    for (int i = 0; i < n6; ++i) xn[L.x_lam + i] = fma(alpha_lam, d[L.d_pi + i] - xo[L.x_lam + i], xo[L.x_lam + i]);
    double slack = 1.0;
    for (int j = 0; j < m; ++j) {
      const double ao = xo[6 * j + 4], da = d[6 * j + 4];
      double zla = xo[L.x_zla + j], zua = xo[L.x_zua + j];
      zla += alpha_z * ((mu - zla * da) / ao - zla);
      zua += alpha_z * ((mu + zua * da) / (P.a_ub - ao) - zua);
      const double a = xn[6 * j + 4];
      const double dLa = a, dUa = P.a_ub - a;
      if (!(dLa > 0 && dUa > 0)) bad = 1;
      zla = clip_mult(zla, dLa, mu); zua = clip_mult(zua, dUa, mu);
      xn[L.x_zla + j] = zla; xn[L.x_zua + j] = zua;
      slack *= dLa * dUa;
      const double c1 = dLa * zla, c2 = dUa * zua;
      cmin = dmin(cmin, dmin(c1, c2)); cmax = dmax(cmax, dmax(c1, c2));
      sz += zla + zua;
    }
    {
      double zlu = xo[L.x_zlu], zuu = xo[L.x_zuu];
      zlu += alpha_z * ((mu - zlu * du) / (u_old + P.u_ub) - zlu);
      zuu += alpha_z * ((mu + zuu * du) / (P.u_ub - u_old) - zuu);
      const double dLu = u + P.u_ub, dUu = P.u_ub - u;
      if (!(dLu > 0 && dUu > 0)) bad = 1;
      zlu = clip_mult(zlu, dLu, mu); zuu = clip_mult(zuu, dUu, mu);
      xn[L.x_zlu] = zlu; xn[L.x_zuu] = zuu;
      slack *= dLu * dUu;
      const double c3 = dLu * zlu, c4 = dUu * zuu;
      cmin = dmin(cmin, dmin(c3, c4)); cmax = dmax(cmax, dmax(c3, c4));
      sz += zlu + zuu;
    }
    sumlog += log(slack);
  }
  Grp<GP>::sync(W.mask);
  // pass 2: condensed model of the trial point, defects, Lagrangian gradient
  for (int k = 1 + W.g; k <= N; k += GP) {
    const double* xn = W.X(dst, k);
    double* mrec = W.Mo(dst, k);
    double z0[6];
    const double* xp = W.X(dst, k - 1) + 6 * (m - 1);
    for (int r = 0; r < 6; ++r) z0[r] = k > 1 ? xp[r] : 0.0;
    const double hk = M.h[k], kap = hk * P.T, al = kap * tf;
    const double u = xn[L.x_u];
    // the Lagrangian gradient needs E^T lam at the trial point: evaluate it from the model functions directly
    // (E itself is overwritten by its LU factors inside build_step)
    double res[MAXN6];
    for (int i = 0; i < n6; ++i) res[i] = xn[L.x_lam + i];                      // identity part of E^T lam
    double gu = 0.0, gt = 0.0;
    double cdef[MAXN6], Fpt[MAXN6];
    build_step(P, C, L, hk, M.tau[k - 1], tf, false, xn, z0, mrec, cdef, Fpt);
    for (int j = 0; j < m; ++j) {
      const double* z = xn + 6 * j;
      const double tj = M.tau[k - 1] + C.tau[j] * hk;
      const double taum = P.mT * tj;
      Accel1 f;
      accel_first(P, z[0], z[2], z[4], taum * tf, f);
      double lamt[6] = {0, 0, 0, 0, 0, 0};
      for (int i = 0; i < m; ++i)
        for (int r = 0; r < 6; ++r) lamt[r] += C.N[i][j] * xn[L.x_lam + 6 * i + r];
      // - al * F_z(z_j)^T lamt_j
      res[6 * j + 0] -= al * (f.ay_y * lamt[1] + f.ax_y * lamt[3]);
      res[6 * j + 1] -= al * lamt[0];
      res[6 * j + 2] -= al * (f.ay_x * lamt[1] + f.ax_x * lamt[3]);
      res[6 * j + 3] -= al * lamt[2];
      res[6 * j + 4] -= al * (f.ay_a * lamt[1] + f.ax_a * lamt[3]);
      res[6 * j + 5] -= al * lamt[4];
      res[6 * j + 4] += xn[L.x_zua + j] - xn[L.x_zla + j];
      gu -= al * P.asc * lamt[5];
      gt -= kap * (lamt[0] * z[1] + lamt[1] * (f.ay + tf * f.ay_m * taum) + lamt[2] * z[3] + lamt[3] * (f.ax + tf * f.ax_m * taum) +
                   lamt[4] * z[5] + lamt[5] * P.asc * u);
    }
    gu += xn[L.x_zuu] - xn[L.x_zlu];
    for (int i = 0; i < n6; ++i) {
      const double ac = fabs(cdef[i]);
      theta += ac; prim = dmax(prim, ac);
      slam += fabs(xn[L.x_lam + i]);
    }
    if (k == N) {
      const double* z = xn + 6 * (m - 1);
      Terminal T;
      terminal_eval(P, z[0], z[1], z[2], z[3], T);
      const double c1 = T.g1 - t.sg1, c2 = T.g2 - t.sg2, c3 = T.g3;
      theta += fabs(c1) + fabs(c2) + fabs(c3);
      prim = dmax(prim, dmax(fabs(c1), dmax(fabs(c2), fabs(c3))));
      const double rinv = 1.0 / T.rT;
      double* rl = res + 6 * (m - 1);
      rl[0] += -t.zs1 * T.Yb * rinv + t.nu3 * z[1];
      rl[2] += -t.zs1 * z[2] * rinv + t.nu3 * z[3];
      rl[1] += -t.zs2 * 2.0 * z[1] + t.nu3 * T.Yb;
      rl[3] += -t.zs2 * 2.0 * z[3] + t.nu3 * z[2];
    } else {
      const double* xq = W.X(dst, k + 1);
      double* rl = res + 6 * (m - 1);
      for (int i = 0; i < m; ++i)
        for (int r = 0; r < 6; ++r) rl[r] -= xq[L.x_lam + 6 * i + r];            // sigma_{k+1}
    }
    for (int i = 0; i < n6; ++i) dual = dmax(dual, fabs(res[i]));
    dual = dmax(dual, fabs(gu));
    gtf += gt;
  }
  theta = Grp<GP>::sum(W.mask, theta);
  sumlog = Grp<GP>::sum(W.mask, sumlog) + sumlog0;
  slam = Grp<GP>::sum(W.mask, slam) + slam0;
  sz = Grp<GP>::sum(W.mask, sz) + sz0;
  gtf = Grp<GP>::sum(W.mask, gtf) + gtf0;
  prim = Grp<GP>::max(W.mask, prim);
  dual = dmax(Grp<GP>::max(W.mask, dual), fabs(gtf));
  cmin = dmin(Grp<GP>::min(W.mask, cmin), cmin0);
  cmax = dmax(Grp<GP>::max(W.mask, cmax), cmax0);
  const bool anybad = Grp<GP>::any(W.mask, bad) != 0 || bad0;
  t.theta = theta;
  t.fobj = O.obj_scale * tf;
  t.sumlog = anybad ? -1e300 : sumlog;
  t.prim_inf = prim; t.dual_inf = dual; t.cmin = cmin; t.cmax = cmax; t.sum_lam = slam; t.sum_z = sz;
  if (anybad || !(theta == theta)) t.theta = 1e300;
  Grp<GP>::sync(W.mask);
}

// ---------------------------------------------------------------------------------------
// start point: the bang-bang pitch-acceleration profile of start_rollout() (ascent_ipm.cuh) rolled out WITH THE
// COLLOCATION RULE ITSELF: every step is first predicted by Euler sub-steps from point to point and then
// corrected by three Newton iterations on its own collocation rows (the condensation's affine column is
// exactly -E^-1 c), so the start is dynamically feasible and only the terminal rows and the interior push of the
// angle are violated -- as for NODES = 2.  (With the Euler prediction alone, coarse high-order meshes start at
// theta ~ 10 and 4 % of the dispersions never recovered: there is no restoration phase to fall back on.)
// The control of a step is the profile's value at the step's mid time.  One lane; the others wait.
// ---------------------------------------------------------------------------------------
template <int GP>
LM_NOINLINE void colloc_init_guess(const Params& P, const Mesh& M, const Options& O, const Coll& C, const Nws& W, Scal& s,
                                   int variant) {
  const int N = M.N, m = W.L.m, n6 = W.L.n6;
  const Lay& L = W.L;
  // Start-point ladder (a problem that fails from one start is restarted from the next; this solver has no
  // restoration phase).  Measured on 300 six-parameter dispersions at NODES = 4, nt = 24 (host build), failures
  // per start: burn time guess + 0.06 with the Euler roll-out 2, guess itself 12, + Newton correction 30 / 34;
  // no problem fails from all of them.  A longer burn is the better guess: the terminal rows start less violated.
  //   0: tf_guess + 0.06, Euler roll-out     1: tf_guess, Euler roll-out
  //   2: tf_guess + 0.06, Newton-corrected   3: tf_guess, Newton-corrected
  const double tfg = (variant & 1) ? O.tf_guess : dmin(O.tf_guess + 0.06, 0.97);
  const double tf0 = dmin(dmax(tfg, 1e-2 * P.tf_ub), 0.99 * P.tf_ub);
  const bool newton = variant >= 2;
  if (W.g == 0) {
    const GuessProfile gp = guess_profile(P);
    const double a_lo = 1e-2 * P.a_ub, a_hi = 0.99 * P.a_ub;
    for (int b = 0; b < 2; ++b) for (int i = 0; i < L.XR; ++i) W.X(b, 0)[i] = 0.0;
    for (int i = 0; i < L.DR; ++i) W.D(0)[i] = 0.0;
    double z0[6] = {0, 0, 0, 0, 0, 0};
    for (int k = 1; k <= N; ++k) {
      const double tmid = (M.tau[k - 1] + 0.5 * M.h[k]) * tf0 * P.T;
      const double u = tmid < gp.t1 ? gp.ulev : (tmid < gp.t1 + gp.t2 ? -gp.ulev : 0.0);
      double* xr = W.X(0, k);
      for (int i = 0; i < L.XR; ++i) xr[i] = 0.0;
      // Euler prediction from point to point
      double y = z0[0], vy = z0[1], x = z0[2], vx = z0[3], a = z0[4], w = z0[5];
      double t_prev = M.tau[k - 1] * tf0 * P.T;
      for (int j = 0; j < m; ++j) {
        const double t = (M.tau[k - 1] + C.tau[j] * M.h[k]) * tf0 * P.T;
        const double dt = t - t_prev;
        w += dt * P.asc * u;
        a += dt * w;
        const double ac = dmin(dmax(a, a_lo), a_hi);
        double yn = y + dt * vy, xn = x + dt * vx, vyn = vy, vxn = vx;
        for (int itr = 0; itr < 3; ++itr) {                     // implicit Euler sub-step, as in start_rollout()
          double ay, ax;
          accel_value(P, yn, xn, ac, P.mflow * t, ay, ax);
          vyn = vy + dt * ay; vxn = vx + dt * ax;
          yn = y + dt * vyn;  xn = x + dt * vxn;
        }
        y = yn; vy = vyn; x = xn; vx = vxn;
        t_prev = t;
        double* z = xr + 6 * j;
        z[0] = y; z[1] = vy; z[2] = x; z[3] = vx; z[4] = newton ? a : ac; z[5] = w;
      }
      xr[L.x_u] = u;
      // Newton correction on the step's collocation rows (z_0 and u fixed)
      for (int itn = 0; itn < (newton ? 3 : 0); ++itn) {
        build_step(P, C, L, M.h[k], M.tau[k - 1], tf0, false, xr, z0, W.Mo(0, k), nullptr, nullptr);
        const double* Phi = W.Mo(0, k);
        for (int i = 0; i < n6; ++i) xr[i] += Phi[i * 9 + 8];
      }
      for (int r = 0; r < 6; ++r) z0[r] = xr[6 * (m - 1) + r];
      for (int j = 0; j < m; ++j) {
        xr[6 * j + 4] = dmin(dmax(xr[6 * j + 4], a_lo), a_hi);          // interior push of the angle (IPOPT's bound_push)
        xr[L.x_zla + j] = 1.0; xr[L.x_zua + j] = 1.0;
      }
      xr[L.x_zlu] = 1.0; xr[L.x_zuu] = 1.0;
      for (int i = 0; i < L.DR; ++i) W.D(k)[i] = 0.0;
    }
  }
  start_scalars(s, tf0);
  Grp<GP>::sync(W.mask);
}

}  // namespace colloc

// Sweeps policy of the higher-order collocation path for the IPM driver (ipm_iterate_t).
template <int GP>
struct SweepsColloc {
  enum : int { LANES_PER_PROBLEM = GP, MOVE_TERM = 0, STORES_REF = 0 };
  LM_HD static int n_eq(const colloc::Nws& W, int N) { return 6 * W.L.m * N + 3; }
  LM_HD static int n_bd(const colloc::Nws& W, int N) { return (2 * W.L.m + 2) * N + 4; }
  LM_HD static bool backward(const Params& P, const Mesh& M, const Options& O, const colloc::Nws& W, int src, const Scal& c0,
                             double mu, double dw, bool ls, double* dtf) {
    if (ls) colloc::colloc_build<GP>(P, M, *W.C, W, src, c0.tf, true);
    return colloc::colloc_backward<GP>(P, M, O, W, src, c0, mu, dw, ls, dtf);
  }
  LM_HD static void forward(const Params& P, const Mesh& M, const Options& O, const colloc::Nws& W, int src, const Scal& c0,
                            double mu, double tau, double dtf, bool ls, TermStep& ts, StepInfo& si) {
    colloc::colloc_forward<GP>(P, M, O, *W.C, W, src, c0, mu, tau, dtf, ls, ts, si);
  }
  LM_HD static void eval(const Params& P, const Mesh& M, const Options& O, const colloc::Nws& W, int src, int dst,
                         const Scal& c0, const TermStep& ts, double mu, double /*dw*/, double alpha, double alpha_z,
                         double alpha_lam, int /*mode*/, Scal& t, double* pimax) {
    colloc::colloc_eval<GP>(P, M, O, *W.C, W, src, dst, c0, ts, mu, alpha, alpha_z, alpha_lam, t);
    if (pimax) *pimax = W.pimax;
  }
  // the start points of the ladder, tried in turn by ipm_start / ipm_restart below (this solver has no restoration phase)
  enum : int { N_STARTS = 4 };
  LM_HD static void guess_variant(const Params& P, const Mesh& M, const Options& O, const colloc::Nws& W, Scal& s, int variant) {
    colloc::colloc_init_guess<GP>(P, M, O, *W.C, W, s, variant);
  }
  // node k of iterate `cur`: x = the six states and the control.  The multipliers of the collocation rows do not map
  // onto one row per node, and the C ABI rejects sensitivities for NODES >= 3, so lam (if not null) is set to NaN.
  LM_HD static void node(const colloc::Nws& W, int cur, int k, double* x, double* lam) {
    const double* xr = W.X(cur, k);
    if (x) {
      for (int i = 0; i < 6; ++i) x[i] = xr[6 * (W.L.m - 1) + i];     // the mesh node is the last collocation point of its step
      x[6] = xr[W.L.x_u];
    }
    if (lam) lam[0] = lam[1] = lam[2] = NAN;
  }
  LM_HD static void node_duals(const colloc::Nws&, int, int, double* d) {
    for (int i = 0; i < 9; ++i) d[i] = NAN;
  }
  LM_HD static void remerit(const Mesh&, const Options&, const colloc::Nws&, int, double, Scal&) {}
};

// Start of one problem on the collocation workspace: the first rung of the start ladder (colloc_init_guess).  The
// caller's start point and the batch reference are not read: the C ABI rejects a start point for NODES >= 3 and never
// sets a reference for them.
template <class SW>
LM_HD void ipm_start(const Params& P, const Mesh& M, const Options& O, const colloc::Nws& W, const GuessSrc&, const double*,
                     IpmState& S) {
  ipm_begin(O, S);
  S.start = 0;
  SW::guess_variant(P, M, O, W, S.cur, 0);
}

// A problem that failed from one rung of the ladder is restarted from the next, unless it stopped at MAX_ITER or no
// rung is left.  The iteration count carries on, so that MAX_ITER (LO:28) bounds the whole ladder and the reported
// iterations include the abandoned starts.  Returns true if it restarted.
template <class SW>
LM_HD bool ipm_restart(const Params& P, const Mesh& M, const Options& O, const colloc::Nws& W, IpmState& S) {
  if (S.ctl.status == ST_CONVERGED || S.ctl.status == ST_MAX_ITER || S.start + 1 >= (int)SW::N_STARTS) return false;
  const int it_used = S.ctl.iter;
  ipm_begin(O, S);
  S.ctl.iter = it_used; S.ctl.iter_best = it_used;
  SW::guess_variant(P, M, O, W, S.cur, ++S.start);
  return true;
}

}  // namespace lmato
