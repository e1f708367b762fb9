// Batched primal-dual interior-point method for the ascent NLP, one problem per thread.
//
// Replaces, for this one model family, what the reference reaches through
// m.solve() (LO:177): APMonitor's collocation transcription + AD + IPOPT/MA27.
//   subsystem (1) transcription ......... stage defects below (backward Euler == GEKKO NODES=2, LO:25)
//   subsystem (2) residual/Jacobian/Hessian  ascent_model.cuh + the Q assembly in riccati_backward()
//   subsystem (3) KKT factorisation ...... riccati_backward() / riccati_forward(): stage-wise
//                 block-tridiagonal LDL^T (Riccati recursion) with inertia read from the pivots
//   subsystem (4) barrier / fraction-to-boundary / filter line search: ipm_iterate_t()
//
// IPM = Waechter & Biegler, Math. Prog. 106 (2006) (the algorithm behind SOLVER=3, LO:26).
//
// Data layout (HBM): ws[stage][warp][field][lane] -- for one warp and one stage the N_FIELDS
// fields are N_FIELDS consecutive 256-byte rows, so every field access is the stage pointer plus
// a compile-time offset (no address arithmetic per access) and every warp access is one fully
// coalesced, 256-byte-aligned transaction.  All sweeps stream stage by stage through HBM; the rows a
// stage reads are staged one stage ahead in shared memory with cp.async (tl_* below).
#pragma once
#include "ascent_model.cuh"

namespace lmato {

// ---------------------------------------------------------------------------------------
// options / status
// ---------------------------------------------------------------------------------------
struct Options {
  double tol;            // scaled KKT error (IPOPT `tol`)
  double mu_init;        // 0.1
  double obj_scale;      // objective = obj_scale * tf
  double kappa_eps;      // sub-problem tolerance kappa_eps * mu (IPOPT: 10; default here 30)
  double kappa_mu;       // 0.2
  double theta_mu;       // barrier decrease mu <- min(kappa_mu mu, mu^theta_mu): IPOPT's 1.5 from the cold start,
  double theta_mu_warm;  // 2 from the batch warm start (measured: cold 30.0 vs 30.7 iterations, warm 24.6 vs 23.2)
  double tau_min;        // 0.99
  double delta_c;        // dual regularisation of the terminal equality row
  double tf_guess;       // initial tf (scaled, 0..1)
  double mu_min_factor;  // smallest barrier parameter = mu_min_factor * tol (IPOPT: 0.1)
  double w_dcost;        // weight of the move-suppression term (LO:99) relative to obj_scale*tf; 0 = off
  int max_iter;          // LO:28 MAX_ITER
  int max_ls;            // max backtracking steps
  int n_polish;          // extra Newton iterations after the tolerance is first met
};

enum Status : int {
  ST_CONVERGED = 0,
  ST_MAX_ITER = 1,
  ST_LINESEARCH_FAIL = 2,
  ST_INERTIA_FAIL = 3,
  ST_NUMERICAL = 4,
  ST_STALLED = 5,
  ST_RUNNING = -1,
};

// ---------------------------------------------------------------------------------------
// workspace fields (row index inside one [stage][warp] block; a row = 32 lanes)
// ---------------------------------------------------------------------------------------
enum : int {
  // iterate, two ping-pong copies at rows [0,17) and [17,34)
  F_Z = 0,          // 6: y, vy, x, vx, angle, angledot
  F_U = 6,          // 1
  F_LAM = 7,        // 6: defect multipliers
  F_ZLA = 13, F_ZUA = 14, F_ZLU = 15, F_ZUU = 16,
  N_ITER = 17,
  // step, rows [34,47)
  R_STEP = 2 * N_ITER,
  F_DS = R_STEP + 0,   // 6
  F_DU = R_STEP + 6,
  F_PI = R_STEP + 7,   // 6: new defect multipliers
  N_STEP = 13,
  // factor, rows [47,55): only the feedback law leaves the SM (the cost-to-go P, p stays in
  // registers during the backward sweep; multipliers are recovered by an adjoint recursion)
  R_FACT = R_STEP + N_STEP,
  F_K = R_FACT + 0,    // 7 feedback gains
  F_KFF = R_FACT + 7,
  N_FACT = 8,
  N_FIELDS = 2 * N_ITER + N_STEP + N_FACT   // 55 doubles per stage per problem
};
constexpr int LANES = 32;

struct Mesh {
  int N;                 // number of steps (nt-1)
  const double* h;       // h[k]  = time[k]-time[k-1], k=1..N (index 0 unused)   LO:21
  const double* tau;     // tau[k] = time[k]
};

// Staging tiles in shared memory (below): the handle is a shared-space byte address on the device and a
// plain pointer in the host build of these headers (tools/hostsim).
constexpr int TILE_DATA = 36;                       // largest set of workspace rows a stage of any sweep reads
constexpr int TL_H = TILE_DATA, TL_TAU = TILE_DATA + 1;   // + the mesh step h[k] and the node time tau[k]
constexpr int TILE_ROWS = TILE_DATA + 2;
#if defined(__CUDA_ARCH__)
typedef unsigned TileRef;
#else
typedef double* TileRef;
#endif

// Hides how a workspace pointer was computed from the optimiser.  Without it the loop-strength
// reduction turns every row address of a stage loop into its own 64-bit induction variable (two
// integer adds per row and stage, and a register pair each); with it a stage has one base pointer and
// the rows are immediate offsets.
template <class T>
LM_HD T* ws_opaque(T* q) {
#if defined(__CUDA_ARCH__)
  asm("" : "+l"(q));
#endif
  return q;
}

// View of one thread's column of the workspace.
struct Ws {
  double* p;             // base + (warp * N_FIELDS) * 32 + lane
  long SS;               // stage stride in doubles = n_warps * N_FIELDS * 32
  TileRef tl;            // this lane's column of the warp's two staging tiles
  mutable int ls_flag;   // 1 while the least-squares multiplier estimate runs: the sweeps re-read it from
                         // shared memory every stage (as a register it was spilled to local memory)
  LM_HD double* stage(int k) const { return ws_opaque(p + (long)k * SS); }
};
#define WS_AT(sp, row) (sp)[(row) * LANES]

// Staging of workspace rows in shared memory.  With 255 registers per thread only 8 warps are
// resident per SM, far too few to hide a memory round trip per stage, and eight warps' stage
// footprints thrash L1 (a software prefetch into L1 ended with a 1 % hit rate).  Instead every lane
// copies the rows of its own column that the NEXT stage reads into a per-warp double buffer with
// cp.async (LDGSTS: no registers, and no warp-level synchronisation, because a lane only ever reads
// what it copied itself), commits one group per stage and waits for all but the newest group before
// it consumes a tile.  The loads of the stage body are then shared-memory loads.
// Tile of stage k lives in buffer k & 1.
LM_HD TileRef tl_buf(const Ws& W, int k) {
#if defined(__CUDA_ARCH__)
  return W.tl + (unsigned)(k & 1) * (unsigned)(TILE_ROWS * LANES * 8);
#else
  return W.tl + (k & 1) * TILE_ROWS;
#endif
}
LM_HD void tl_copy(TileRef tb, int slot, const double* src) {
#if defined(__CUDA_ARCH__)
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(tb + (unsigned)(slot * LANES * 8)), "l"(src) : "memory");
#else
  tb[slot] = *src;
#endif
}
// rows [row0, row0 + NROWS) of the stage column sp -> slots [SLOT0, SLOT0 + NROWS)
template <int SLOT0, int NROWS>
LM_HD void tl_copy_rows(TileRef tb, const double* sp, int row0) {
#pragma unroll
  for (int r = 0; r < NROWS; ++r) tl_copy(tb, SLOT0 + r, sp + (row0 + r) * LANES);
}
// h[k], tau[k]: every lane stages its own copy (same address across the warp: one sector)
LM_HD void tl_copy_mesh(TileRef tb, const Mesh& M, int k) {
  tl_copy(tb, TL_H, M.h + k);
  tl_copy(tb, TL_TAU, M.tau + k);
}
LM_HD void tl_commit() {
#if defined(__CUDA_ARCH__)
  asm volatile("cp.async.commit_group;" ::: "memory");
#endif
}
// all groups but the newest have landed
LM_HD void tl_wait_prev() {
#if defined(__CUDA_ARCH__)
  asm volatile("cp.async.wait_group 1;" ::: "memory");
#endif
}
// start of a sweep: the rows about to be copied were written by this thread's own stores
LM_HD void tl_begin() {
#if defined(__CUDA_ARCH__)
  asm volatile("cp.async.wait_all;" ::: "memory");
  __threadfence_block();
#endif
}
LM_HD double tl_ld(TileRef tb, int slot) {
#if defined(__CUDA_ARCH__)
  double v;
  // volatile keeps it after the wait (volatile asms are not reordered among themselves)
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(tb + (unsigned)(slot * LANES * 8)));
  return v;
#else
  return tb[slot];
#endif
}

constexpr int NFILT = 12;
#ifndef LMATO_LS_NULL
#define LMATO_LS_NULL 12
#endif
#ifndef LMATO_WARM_STALL_WINDOW
#define LMATO_WARM_STALL_WINDOW 30
#endif

// Per-problem scalar state (registers / local memory).
struct Scal {
  double tf, zLt, zUt;            // global final time and its bound multipliers
  double sg1, sg2, zs1, zs2, nu3; // terminal slacks, their multipliers, equality multiplier
  double theta, fobj, sumlog;     // constraint violation (l1), objective, sum of log slacks
  double dual_inf, prim_inf, cmin, cmax, sum_lam, sum_z;
};

struct Ctl {
  double mu, tau;
  double theta_max, theta_min;
  double dw_last;
  double ft[NFILT], fp[NFILT];
  int nf;
  int iter;
  int status;
  // stall guard (this solver has no restoration phase): consecutive accepted steps shorter than 1e-6, and the
  // iteration at which the KKT error last improved
  int tiny_steps;
  int null_steps;      // line searches of this solve that ended as a null step (see LMATO_LS_NULL)
  int iter_best;
  double err_best;
};

// ---------------------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------------------
LM_HD constexpr int pidx(int i, int j) {  // packed lower-triangular index, i >= j
  return i * (i + 1) / 2 + j;
}
LM_HD double dmax(double a, double b) { return a > b ? a : b; }
LM_HD double dmin(double a, double b) { return a < b ? a : b; }

// 1/a, 1/b, 1/c, 1/d with a single division (all arguments are positive slacks in (0, ~2)).
LM_HD void recip4(double a, double b, double c, double d, double& ia, double& ib, double& ic, double& id) {
  const double ab = a * b, cd = c * d;
  const double ip = lm_rcp(ab * cd);
  const double iab = ip * cd, icd = ip * ab;
  ia = iab * b; ib = iab * a; ic = icd * d; id = icd * c;
}

// kappa_Sigma safeguard (IPOPT eq. 16) written on the complementarity product so that the common
// path has no division:  z in [mu/(kS d), kS mu/d]  <=>  z d in [mu/kS, kS mu].
LM_HD double clip_mult(double z, double d, double mu) {
  const double kS = 1e10;
  const double c = z * d;
  if (c > kS * mu) return kS * mu / d;
  if (c < mu / kS) return mu / (kS * d);
  return z;
}

// Stage Jacobian data: everything needed to apply E^{-1} and E^{-T}.
//   E = d defect_k / d s_k  for s = (y, vy, x, vx, a, w, tf); d defect_k / d s_{k-1} = -I;
//   d defect_k / d u_k = -beta e_5.
struct StageJac {
  double al;                  // alpha = h*T*tf
  double ala, alb, alc, ald;  // alpha * (ay_y, ay_x, ax_y, ax_x)
  double m11, m13, m31, m33;  // inverse of the 2x2 velocity block (only after stagejac_invert)
  double ga1, ga3;            // alpha * (ay_a, ax_a)
  double e0, e1, e2, e3, e4, e5;  // tf column (negated entries of E)
  double beta;                // alpha * asc
};

LM_HD void stagejac_build(const Params& P, double kap, double tf, double taum /* d mass/d tf */,
                          const Accel1& f, double vy, double vx, double w, double u, StageJac& J) {
  const double al = kap * tf;
  J.al = al;
  J.ala = al * f.ay_y; J.alb = al * f.ay_x; J.alc = al * f.ax_y; J.ald = al * f.ax_x;
  J.ga1 = al * f.ay_a; J.ga3 = al * f.ax_a;
  const double alt = al * taum;
  J.e0 = kap * vy;
  J.e1 = fma(kap, f.ay, alt * f.ay_m);
  J.e2 = kap * vx;
  J.e3 = fma(kap, f.ax, alt * f.ax_m);
  J.e4 = kap * w;
  J.e5 = kap * P.asc * u;
  J.beta = al * P.asc;
}

LM_HD void stagejac_invert(StageJac& J) {
  const double al = J.al;
  const double a2a = al * J.ala, a2b = al * J.alb, a2c = al * J.alc, a2d = al * J.ald;
  const double d11 = 1.0 - a2a, d33 = 1.0 - a2d;
  const double Dinv = lm_rcp(d11 * d33 - a2b * a2c);
  J.m11 = d33 * Dinv; J.m13 = a2b * Dinv; J.m31 = a2c * Dinv; J.m33 = d11 * Dinv;
}

// v <- E^{-1} v
LM_HD void solveE(const StageJac& J, double* v) {
  const double v6 = v[6];
  const double v5 = fma(J.e5, v6, v[5]);
  const double v4 = v[4] + J.al * v5 + J.e4 * v6;
  const double r0 = fma(J.e0, v6, v[0]);
  const double r2 = fma(J.e2, v6, v[2]);
  const double r1 = v[1] + J.ga1 * v4 + J.e1 * v6;
  const double r3 = v[3] + J.ga3 * v4 + J.e3 * v6;
  const double t1 = r1 + J.ala * r0 + J.alb * r2;
  const double t3 = r3 + J.alc * r0 + J.ald * r2;
  const double v1 = J.m11 * t1 + J.m13 * t3;
  const double v3 = J.m31 * t1 + J.m33 * t3;
  v[0] = fma(J.al, v1, r0);
  v[1] = v1;
  v[2] = fma(J.al, v3, r2);
  v[3] = v3;
  v[4] = v4;
  v[5] = v5;
}

// w <- A11^T w, A11 = inverse of the (y, vy, x, vx) block of E
LM_HD void applyA11T(const StageJac& J, double& w0, double& w1, double& w2, double& w3) {
  const double t0 = w0 + J.ala * w1 + J.alc * w3;
  const double t2 = w2 + J.alb * w1 + J.ald * w3;
  const double n0 = J.m11 * t0 + J.m31 * t2;
  const double n2 = J.m13 * t0 + J.m33 * t2;
  w1 = fma(J.al, n0, w1);
  w3 = fma(J.al, n2, w3);
  w0 = n0; w2 = n2;
}

// g <- E^{-T} g
LM_HD void solveET(const StageJac& J, double* g) {
  double w0 = g[0], w1 = g[1], w2 = g[2], w3 = g[3];
  applyA11T(J, w0, w1, w2, w3);
  const double gaw = J.ga1 * w1 + J.ga3 * w3;
  const double gew = J.e0 * w0 + J.e1 * w1 + J.e2 * w2 + J.e3 * w3;
  const double w4 = g[4] + gaw;
  const double w5 = g[5] + J.al * w4;
  const double w6 = g[6] + gew + J.e4 * w4 + J.e5 * w5;
  g[0] = w0; g[1] = w1; g[2] = w2; g[3] = w3; g[4] = w4; g[5] = w5; g[6] = w6;
}

// E^T lam restricted to the six real states (lam[6] multiplies the trivial tf row).
LM_HD void applyET6(const StageJac& J, const double* l, double* out) {
  out[0] = l[0] - J.ala * l[1] - J.alc * l[3];
  out[1] = l[1] - J.al * l[0];
  out[2] = l[2] - J.alb * l[1] - J.ald * l[3];
  out[3] = l[3] - J.al * l[2];
  out[4] = l[4] - J.ga1 * l[1] - J.ga3 * l[3];
  out[5] = l[5] - J.al * l[4];
}

// ---------------------------------------------------------------------------------------
// initial guess (restated independently in oracle/ascent_nlp.py: initial_guess)
// ---------------------------------------------------------------------------------------
// Start point: a dynamically consistent roll-out of a bang-bang pitch-acceleration profile
// (u = +0.9 until t1, -0.9 until t1+t2, then 0), i.e. the shape of the known optimum
// (Angle_vs_Time.png).  Only the three terminal rows and the interior push of `angle`
// are infeasible at the start.
struct GuessProfile { double t1, t2, ulev; };

LM_HD GuessProfile guess_profile(const Params& P) {
  GuessProfile g;
  const double a_tgt = dmin(0.40, 0.8 * P.a_ub);   // ~69 deg of physical pitch
  const double w_rem = 3.5e-4;                      // residual pitch rate [rad/s of `angle`]
  g.ulev = 0.9 * P.u_ub;
  const double ueff = g.ulev * P.asc;
  g.t1 = sqrt(a_tgt / ueff);
  g.t2 = dmax(g.t1 - w_rem / ueff, 0.0);
  return g;
}

// Caller-supplied start point (SURVEY 8f.4): trajectories in the OUTPUT layout of the solver,
// [variable][node][problem] with the ten variables in the reference's order (LO:83-100), and tf.
struct GuessSrc {
  const double* traj;    // [10][nt][B]
  const double* tf;      // [B]
  long B, b;
  enum : int { V_Y = 0, V_YDOT = 1, V_X = 3, V_XDOT = 4, V_ANGLE = 6, V_ANGLEDOT = 7, V_U = 9 };
  LM_HD double at(int v, int k, int nt) const { return traj[((long)v * nt + k) * B + b]; }
};

// ---------------------------------------------------------------------------------------
// Warm start: every problem of a batch may start from one reference central-path point (the
// batch-mean problem solved down to mu_ref ~ 1e-3) instead of the generic roll-out.  That skips
// the globalisation phase (about 7 of 27 iterations); at smaller mu_ref the iterate sits too close
// to the reference's active bounds and the method jams, so 1e-3 it is.  The reference column is
// REF_ROWS x (N+1) doubles, ref[row * (N+1) + k]: the 17 rows of the 7-state iterate (row7() below) followed by one
// row of scalars (node 0..).  Lengths are stored divided by the reference's distance scale S_ref = r_periapsis
// (LO:107), so a problem rescales them to its own.
// ---------------------------------------------------------------------------------------
enum : int { REF_ROWS = N_ITER + 1, REF_OK = 0, REF_MU = 1, REF_S = 2, REF_TF = 3, REF_ZLT = 4, REF_ZUT = 5,
             REF_SG1 = 6, REF_SG2 = 7, REF_ZS1 = 8, REF_ZS2 = 9, REF_NU3 = 10, REF_NSCAL = 11 };

// ---------------------------------------------------------------------------------------
// Start points of every NODES = 2 workspace layout.  The values of a node come from start_node() (roll-out, caller's
// start point) or ref_node() (batch reference); a layout -- the Sweeps policies Sweeps7, Sweeps8 and SweepsCoop --
// only says where they go (SW::store_node), how node 0 is zeroed (SW::zero_node0), whether it carries the move slack
// pair (SW::MOVE_TERM) and how many lanes share a problem (SW::LANES_PER_PROBLEM = G; the thread layouts: G = 1).
// ---------------------------------------------------------------------------------------
namespace coop { template <int G> struct Grp; }     // the lanes of one problem (ascent_coop.cuh)
// this lane's index among them and their mask (the cooperative workspace: ascent_coop.cuh)
LM_HD int grp_lane(const Ws&) { return 0; }
LM_HD unsigned grp_mask(const Ws&) { return 1u; }

// One node of a start point in the row order of the 8-state iterate (ascent_ipm_dc.cuh: dc::F_*; the cooperative X
// record).  The 7-state iterate and the reference column hold the first NODE_N7 fields without lam_6.
enum : int { NODE_Z = 0, NODE_U = 6, NODE_LAM = 7 /* 7 */, NODE_ZLA = 14, NODE_ZUA = 15, NODE_ZLU = 16, NODE_ZUU = 17,
             NODE_PP = 18, NODE_PN = 19, NODE_ZPP = 20, NODE_ZPN = 21, NODE_N = 22, NODE_N7 = NODE_PP };
// row of the 7-state iterate (and of the reference column) that holds node field f < NODE_N7, f != NODE_LAM + 6
LM_HD constexpr int row7(int f) { return f < NODE_LAM + 6 ? f : f - 1; }
static_assert(row7(NODE_U) == F_U && row7(NODE_LAM) == F_LAM && row7(NODE_ZLA) == F_ZLA && row7(NODE_ZUU) == F_ZUU &&
              row7(NODE_ZUU) + 1 == N_ITER, "7-state rows");

// Node k >= 1 of a cold or caller start: primal values as given, defect multipliers 0, bound multipliers 1 (an
// unbounded control -- circular model, coup5 = 0 -- starts exactly on the central path of its vacuous bounds), and
// with the move term the slack pair on its central path for mu_init with lam_6 = 0 (z_p = z_n = w, p + n = t(v),
// p - n = v, v = u - u_prev).
LM_HD void start_node(const Params& P, const Options& O, const double* z6, double u, double u_prev, bool move, double* x) {
#pragma unroll
  for (int i = 0; i < 6; ++i) x[NODE_Z + i] = z6[i];
  x[NODE_U] = u;
#pragma unroll
  for (int i = 0; i < 7; ++i) x[NODE_LAM + i] = 0.0;
  x[NODE_ZLA] = 1.0; x[NODE_ZUA] = 1.0;
  x[NODE_ZLU] = P.coup5 != 0.0 ? 1.0 : O.mu_init / (u + P.u_ub);
  x[NODE_ZUU] = P.coup5 != 0.0 ? 1.0 : O.mu_init / (P.u_ub - u);
  if (move) {
    const double wd = O.w_dcost, v = u - u_prev;
    const double tt = (O.mu_init + sqrt(O.mu_init * O.mu_init + wd * wd * v * v)) / wd;
    x[NODE_PP] = 0.5 * (tt + v); x[NODE_PN] = 0.5 * (tt - v); x[NODE_ZPP] = wd; x[NODE_ZPN] = wd;
  } else {
    x[NODE_PP] = 1.0; x[NODE_PN] = 1.0; x[NODE_ZPP] = 0.0; x[NODE_ZPN] = 0.0;
  }
}

// Node k >= 1 from the reference column: lengths rescaled by r = S_ref / S and the multipliers of their rows by
// ri = S / S_ref.  The reference is a solve without the move term (at mu_ref ~ 1e-3 >> w the two central paths
// practically coincide): with the move term the slack pair is put exactly on its own central path for mu_ref and the
// reference's moves (z_p + z_n = 2w, p z_p = n z_n = mu) and lam_6 = w - z_p follows from dual feasibility.
LM_HD void ref_node(const double* ref, int N1, int k, double r, double ri, double mu, double w, bool move, double* x) {
#pragma unroll
  for (int f = 0; f < NODE_N7; ++f)
    if (f != NODE_LAM + 6) x[f] = ref[row7(f) * N1 + k];
#pragma unroll
  for (int i = 0; i < 4; ++i) { x[NODE_Z + i] *= r; x[NODE_LAM + i] *= ri; }    // y, vy, x, vx and their rows
  if (move) {
    const double v = x[NODE_U] - (k > 1 ? ref[row7(NODE_U) * N1 + k - 1] : 0.0);
    const double tt = (mu + sqrt(mu * mu + w * w * v * v)) / w;
    const double pp = 0.5 * (tt + v), pn = 0.5 * (tt - v);
    x[NODE_PP] = pp; x[NODE_PN] = pn; x[NODE_ZPP] = mu / pp; x[NODE_ZPN] = mu / pn;
    x[NODE_LAM + 6] = w - mu / pp;
  } else {
    x[NODE_PP] = 1.0; x[NODE_PN] = 1.0; x[NODE_ZPP] = 0.0; x[NODE_ZPN] = 0.0;
    x[NODE_LAM + 6] = 0.0;
  }
}

// node k of a converged reference solve into the reference column
LM_HD void ref_put_node(double* ref, int N1, int k, const double* x) {
#pragma unroll
  for (int f = 0; f < NODE_N7; ++f)
    if (f != NODE_LAM + 6) ref[row7(f) * N1 + k] = x[f];
}

LM_HD void ref_put_scalars(double* ref, int N1, const Params& P, const Scal& c, double mu, bool ok) {
  double* sc = ref + N_ITER * N1;
  sc[REF_OK] = ok ? 1.0 : 0.0; sc[REF_MU] = mu; sc[REF_S] = P.S; sc[REF_TF] = c.tf;
  sc[REF_ZLT] = c.zLt; sc[REF_ZUT] = c.zUt; sc[REF_SG1] = c.sg1; sc[REF_SG2] = c.sg2;
  sc[REF_ZS1] = c.zs1; sc[REF_ZS2] = c.zs2; sc[REF_NU3] = c.nu3;
}

// The start scalars, the barrier parameter mu and the length ratios r, ri of a start from the reference column, or
// false if the column holds no reference.
LM_HD bool ref_scalars(const Params& P, const double* ref, int N1, Scal& s, double& mu, double& r, double& ri) {
  const double* sc = ref + N_ITER * N1;
  if (!(sc[REF_OK] > 0.5)) return false;
  r = sc[REF_S] * P.Sinv; ri = P.S / sc[REF_S];
  mu = sc[REF_MU];
  s.tf = dmin(sc[REF_TF], 0.99 * P.tf_ub);
  s.zLt = sc[REF_ZLT]; s.zUt = sc[REF_ZUT];
  s.sg1 = sc[REF_SG1]; s.sg2 = sc[REF_SG2]; s.zs1 = sc[REF_ZS1]; s.zs2 = sc[REF_ZS2]; s.nu3 = sc[REF_NU3];
  return true;
}

LM_HD void start_scalars(Scal& s, double tf0) {
  s.tf = tf0;
  s.zLt = 1.0; s.zUt = 1.0;
  s.sg1 = 1e-2; s.sg2 = 1e-2; s.zs1 = 1.0; s.zs2 = 1.0; s.nu3 = 0.0;
}

// The built-in start point: the roll-out of guess_profile(), a sequential integration carried by each of the G lanes
// of the problem (lane g stores the nodes k with (k - 1) % G == g).
template <class SW, class WS>
LM_NOINLINE void start_rollout(const Params& P, const Mesh& M, const Options& O, const WS& W, Scal& s) {
  constexpr int G = SW::LANES_PER_PROBLEM;
  const int N = M.N, g = grp_lane(W);
  const double tf0 = dmin(dmax(O.tf_guess, 1e-2 * P.tf_ub), 0.99 * P.tf_ub);
  const GuessProfile gp = guess_profile(P);
  double y = 0, vy = 0, x = 0, vx = 0, a = 0, w = 0, t_prev = 0, u_prev = 0;
  const double a_lo = 1e-2 * P.a_ub, a_hi = 0.99 * P.a_ub;
  if (g == 0) SW::zero_node0(W);
  for (int k = 1; k <= N; ++k) {
    const double t = M.tau[k] * tf0 * P.T;
    const double dt = t - t_prev;
    const double tm = 0.5 * (t + t_prev);
    double u = tm < gp.t1 ? gp.ulev : (tm < gp.t1 + gp.t2 ? -gp.ulev : 0.0);
    if (P.coup5 != 0.0) {
      w += dt * P.asc * u;
      a += dt * w;
    } else {
      // circular model: pitch ramps linearly from ~34 deg (PDF p.21 Fig 9); angledot and u follow
      const double a_new = 0.2 + 0.45 * M.tau[k];
      if (mv_is_angle(P) != 0.0) { w = 0.0; u = dmin(dmax(a_new, a_lo), a_hi); }    // the MV is the pitch angle
      else { w = (a_new - a) / dt; u = w / (dt * P.asc); }
      a = a_new;
    }
    const double ac = dmin(dmax(a, a_lo), a_hi);
    const double m = P.mflow * P.T * M.tau[k] * tf0;
    // backward-Euler step for (y, vy, x, vx): three fixed-point sweeps
    double yn = y + dt * vy, xn = x + dt * vx, vyn = vy, vxn = vx;
    for (int itr = 0; itr < 3; ++itr) {
      double ay, ax;
      accel_value(P, yn, xn, ac, m, ay, ax);
      vyn = vy + dt * ay; vxn = vx + dt * ax;
      yn = y + dt * vyn;  xn = x + dt * vxn;
    }
    y = yn; vy = vyn; x = xn; vx = vxn;
    if (((k - 1) % G) == g) {
      const double z6[6] = {y, vy, x, vx, ac, w};
      double xk[NODE_N];
      start_node(P, O, z6, u, u_prev, SW::MOVE_TERM != 0, xk);
      SW::store_node(W, k, xk);
    }
    u_prev = u;
    t_prev = t;
  }
  start_scalars(s, tf0);
  coop::Grp<G>::sync(grp_mask(W));
}

// Caller-supplied start point, stage-parallel over the G lanes.  The primal values are taken as given and only pushed
// into the interior of their bounds (IPOPT's bound_push); multipliers and slacks start as in the roll-out, so
// iteration 0 is again the least-squares multiplier estimate.  Node 0 is pinned whatever the guess says (LO:145-151).
template <class SW, class WS>
LM_NOINLINE void start_from_guess(const Params& P, const Mesh& M, const Options& O, const WS& W, const GuessSrc& Gs,
                                  Scal& s) {
  constexpr int G = SW::LANES_PER_PROBLEM;
  const int N = M.N, nt = N + 1, g = grp_lane(W);
  const double tf0 = dmin(dmax(Gs.tf[Gs.b], 1e-2 * P.tf_ub), 0.99 * P.tf_ub);
  const double a_lo = 1e-2 * P.a_ub, a_hi = 0.99 * P.a_ub, u_hi = 0.99 * P.u_ub;
  if (g == 0) SW::zero_node0(W);
  const bool mva = mv_is_angle(P) != 0.0;       // the MV is the pitch angle: its slot follows the angle row
  for (int k = 1 + g; k <= N; k += G) {
    const double ak = dmin(dmax(Gs.at(GuessSrc::V_ANGLE, k, nt), a_lo), a_hi);
    const double u = mva ? ak : dmin(dmax(Gs.at(GuessSrc::V_U, k, nt), -u_hi), u_hi);
    const double up = k > 1 ? (mva ? dmin(dmax(Gs.at(GuessSrc::V_ANGLE, k - 1, nt), a_lo), a_hi)
                                   : dmin(dmax(Gs.at(GuessSrc::V_U, k - 1, nt), -u_hi), u_hi)) : 0.0;
    const double z6[6] = {Gs.at(GuessSrc::V_Y, k, nt), Gs.at(GuessSrc::V_YDOT, k, nt), Gs.at(GuessSrc::V_X, k, nt),
                          Gs.at(GuessSrc::V_XDOT, k, nt), ak, mva ? 0.0 : Gs.at(GuessSrc::V_ANGLEDOT, k, nt)};
    double xk[NODE_N];
    start_node(P, O, z6, u, up, SW::MOVE_TERM != 0, xk);
    SW::store_node(W, k, xk);
  }
  start_scalars(s, tf0);
  coop::Grp<G>::sync(grp_mask(W));
}

// Start from the reference column, stage-parallel over the G lanes; false (nothing written) if it holds none.
template <class SW, class WS>
LM_NOINLINE bool start_from_ref(const Params& P, const Mesh& M, const Options& O, const WS& W, const double* ref,
                                Scal& s, double* mu_out) {
  constexpr int G = SW::LANES_PER_PROBLEM;
  const int N1 = M.N + 1, g = grp_lane(W);
  double mu, r, ri;
  if (!ref_scalars(P, ref, N1, s, mu, r, ri)) return false;
  if (g == 0) SW::zero_node0(W);
  for (int k = 1 + g; k <= M.N; k += G) {
    double xk[NODE_N];
    ref_node(ref, N1, k, r, ri, mu, O.w_dcost, SW::MOVE_TERM != 0, xk);
    SW::store_node(W, k, xk);
  }
  *mu_out = mu;
  coop::Grp<G>::sync(grp_mask(W));
  return true;
}

// ---------------------------------------------------------------------------------------
// shared building blocks of the Newton system (used by the factorisation AND by the adjoint
// recursion, so that both see exactly the same Hessian)
// ---------------------------------------------------------------------------------------
struct TermStep { double dtf, dsg1, dsg2, dzs1, dzs2, dnu3, dzLt, dzUt; };

// Terminal rows condensed onto the last node (LO:161, 169, 173): Hessian block on (y,vy,x,vx)
// [lower triangle], gradient, and the tf entries (objective + tf bound barrier).
struct TermQP { double H[4][4]; double g[4]; double g6, H66; };

LM_HD void terminal_qp(const Params& P, const Options& O, const Scal& c0, const double* zn, double mu,
                       double dw, bool ls, TermQP& q) {
  Terminal T;
  terminal_eval(P, zn[0], zn[1], zn[2], zn[3], T);
  const double rinv = 1.0 / T.rT;
  const double g1y = T.Yb * rinv, g1x = zn[2] * rinv;
  const double i1 = 1.0 / c0.sg1, i2 = 1.0 / c0.sg2;
  const double w1 = ls ? 1.0 : c0.zs1 * i1, w2 = ls ? 1.0 : c0.zs2 * i2, w3 = 1.0 / O.delta_c;
  const double c1 = T.g1 - c0.sg1, c2 = T.g2 - c0.sg2;
  // gradient terms: grad g_i * (w_i c_i - mu/sg_i), grad g3 * (nu3 + g3/delta_c)
  const double q1 = ls ? -c0.zs1 : w1 * c1 - mu * i1;
  const double q2 = ls ? -c0.zs2 : w2 * c2 - mu * i2;
  const double q3 = ls ? 0.0 : c0.nu3 + T.g3 * w3;
  const double hz1 = ls ? 0.0 : c0.zs1, hz2 = ls ? 0.0 : c0.zs2, hn3 = ls ? 0.0 : c0.nu3;
  const double G2y = 2.0 * zn[1], G2x = 2.0 * zn[3];
  const double G3[4] = {zn[1], T.Yb, zn[3], zn[2]};     // grad g3 wrt (y, vy, x, vx)
  q.g[0] = g1y * q1 + G3[0] * q3;
  q.g[1] = G2y * q2 + G3[1] * q3;
  q.g[2] = g1x * q1 + G3[2] * q3;
  q.g[3] = G2x * q2 + G3[3] * q3;
  // Hessian: w_i grad grad^T + multipliers * second derivatives (mult of g1,g2 = -zs)
  const double r3 = rinv * rinv * rinv;
  const double h1yy = zn[2] * zn[2] * r3, h1xx = T.Yb * T.Yb * r3, h1yx = -T.Yb * zn[2] * r3;
  q.H[0][0] = w1 * g1y * g1y - hz1 * h1yy + w3 * G3[0] * G3[0];
  q.H[2][0] = w1 * g1x * g1y - hz1 * h1yx + w3 * G3[2] * G3[0];
  q.H[2][2] = w1 * g1x * g1x - hz1 * h1xx + w3 * G3[2] * G3[2];
  q.H[1][1] = w2 * G2y * G2y - 2.0 * hz2 + w3 * G3[1] * G3[1];
  q.H[3][1] = w2 * G2x * G2y + w3 * G3[3] * G3[1];
  q.H[3][3] = w2 * G2x * G2x - 2.0 * hz2 + w3 * G3[3] * G3[3];
  q.H[1][0] = w3 * G3[1] * G3[0] + hn3;
  q.H[3][0] = w3 * G3[3] * G3[0];
  q.H[2][1] = w3 * G3[2] * G3[1];
  q.H[3][2] = w3 * G3[3] * G3[2] + hn3;
  q.H[0][1] = q.H[1][0]; q.H[0][2] = q.H[2][0]; q.H[0][3] = q.H[3][0];
  q.H[1][2] = q.H[2][1]; q.H[1][3] = q.H[3][1]; q.H[2][3] = q.H[3][2];
  const double tf = c0.tf;
  const double dLt = tf, dUt = P.tf_ub - tf;
  q.g6 = ls ? O.obj_scale - c0.zLt + c0.zUt : O.obj_scale - mu / dLt + mu / dUt;
  q.H66 = ls ? 1.0 : c0.zLt / dLt + c0.zUt / dUt + dw;
}

// Stage Hessian of the barrier Lagrangian on s = (y,vy,x,vx,a,w,tf) and u (sparse).
struct StageQ {
  double q00, q02, q22, q04, q24, q44;        // (y,x,a) block (includes delta_w and Sigma_a)
  double q06, q16, q26, q36, q46, q56, q66;   // tf column
  double d;                                   // diagonal of the (vy, vx, w) entries (= delta_w or 1)
  double q4;                                  // gradient entry of `angle`
  double R, r, sig;                           // control: Hessian, gradient, u-tf cross term
};

LM_HD void stage_hessian(const Params& P, const Accel1& f, const StageJac& J, double kap, double taum,
                         const double* lam, double a, double u, double zla, double zua, double zlu,
                         double zuu, double mu, double dw, bool ls, StageQ& q) {
  if (!ls) {
    double rLa, rUa, rLu, rUu;
    recip4(a, P.a_ub - a, u + P.u_ub, P.u_ub - u, rLa, rUa, rLu, rUu);
    Accel2 h2;
    accel_second(P, f, lam[1], lam[3], h2);
    const double al = J.al, alt = al * taum;
    q.q00 = -al * h2.yy + dw;
    q.q02 = -al * h2.yx;
    q.q22 = -al * h2.xx + dw;
    q.q04 = -al * h2.ya;
    q.q24 = -al * h2.xa;
    q.q44 = -al * h2.aa + zla * rLa + zua * rUa + dw;
    q.d = dw;
    const double Phy = lam[1] * f.ay_y + lam[3] * f.ax_y;
    const double Phx = lam[1] * f.ay_x + lam[3] * f.ax_x;
    const double Pha = lam[1] * f.ay_a + lam[3] * f.ax_a;
    const double Phm = lam[1] * f.ay_m + lam[3] * f.ax_m;
    q.q06 = -kap * Phy - alt * h2.ym;
    q.q26 = -kap * Phx - alt * h2.xm;
    q.q46 = -kap * Pha - alt * h2.am;
    q.q16 = -kap * lam[0];
    q.q36 = -kap * lam[2];
    q.q56 = -kap * lam[4];
    q.q66 = -2.0 * kap * Phm * taum - alt * h2.mm * taum;
    q.q4 = mu * (rUa - rLa);
    q.R = zlu * rLu + zuu * rUu + dw;
    q.r = mu * (rUu - rLu);
    q.sig = -kap * lam[5] * P.asc;   // u-tf cross term
  } else {
    q.q00 = 1.0; q.q02 = 0.0; q.q22 = 1.0; q.q04 = 0.0; q.q24 = 0.0; q.q44 = 1.0; q.d = 1.0;
    q.q06 = q.q16 = q.q26 = q.q36 = q.q46 = q.q56 = q.q66 = 0.0;
    q.q4 = -zla + zua;
    q.R = 1.0; q.r = -zlu + zuu; q.sig = 0.0;
  }
}

// ---------------------------------------------------------------------------------------
// evaluation pass: trial point  x + alpha*dx  (alpha=0: the current point), swept from the
// last node to the first.  Writes the trial iterate into buffer `dst` and returns its merit /
// KKT-error ingredients.
//
// mode EV_READ_PI : the new defect multipliers pi_k are read from the workspace;
// mode EV_NEWTON  : they are first computed by the adjoint recursion of the Newton system,
//                     E_k^T pi_k = pi_{k+1} - (Q_k ds_k + q_k)      (old point, old multipliers)
//                   and stored (a later back-tracking trial reads them).  This is what lets the
//                   factorisation keep only the feedback gains: the 33 doubles of P_{k-1}, p_{k-1}
//                   per stage never travel through HBM.
// mode EV_LSQ     : same recursion for the least-squares multiplier estimate (Q = I).
// ---------------------------------------------------------------------------------------
// Staging tiles of the 7-state sweeps (tl_* above): "CUR" = rows F_U .. N_ITER-1 of the source iterate at
// stage k (control, multipliers), "PZ"/"PDS" = state and its step at stage k-1.
enum : int {
  N_CUR = N_ITER - F_U,                            // 11
  EV_CUR = 0, EV_DU = EV_CUR + N_CUR, EV_PI = EV_DU + 1, EV_PZ = EV_PI + 6, EV_PDS = EV_PZ + 6, EV_ROWS = EV_PDS + 6,
  BK_CUR = 0, BK_PZ = BK_CUR + N_CUR, BK_ROWS = BK_PZ + 6,
  FW_Z = 0, FW_ZB = FW_Z + 7, FW_K = FW_ZB + (N_ITER - F_ZLA), FW_ROWS = FW_K + N_FACT
};
static_assert(EV_ROWS <= TILE_DATA && BK_ROWS <= TILE_DATA && FW_ROWS <= TILE_DATA, "tile too small");
#define TL7_CUR(tb, base, f) tl_ld(tb, (base) + (f) - F_U)      // row f (>= F_U) of the source iterate

LM_HD void ev7_stage_copy(const Mesh& M, const Ws& W, int k, int so, bool read_pi) {
  const TileRef tb = tl_buf(W, k);
  tl_copy_mesh(tb, M, k);
  const double* sp = W.stage(k);
  const double* sm = ws_opaque(sp - W.SS);
  const double* spo = ws_opaque(sp + so * LANES);
  const double* smo = ws_opaque(sm + so * LANES);
  tl_copy_rows<EV_CUR, N_CUR>(tb, spo, F_U);
  tl_copy(tb, EV_DU, sp + F_DU * LANES);
  if (read_pi) tl_copy_rows<EV_PI, 6>(tb, sp, F_PI);
  tl_copy_rows<EV_PZ, 6>(tb, smo, F_Z);
  tl_copy_rows<EV_PDS, 6>(tb, sm, F_DS);
  tl_commit();
}
LM_HD void bk7_stage_copy(const Mesh& M, const Ws& W, int k, int so) {
  const TileRef tb = tl_buf(W, k);
  tl_copy_mesh(tb, M, k);
  const double* spo = ws_opaque(W.stage(k) + so * LANES);
  tl_copy_rows<BK_CUR, N_CUR>(tb, spo, F_U);
  tl_copy_rows<BK_PZ, 6>(tb, ws_opaque(spo - W.SS), F_Z);
  tl_commit();
}
LM_HD void fw7_stage_copy(const Mesh& M, const Ws& W, int k, int so) {
  const TileRef tb = tl_buf(W, k);
  tl_copy_mesh(tb, M, k);
  const double* sp = W.stage(k);
  const double* spo = ws_opaque(sp + so * LANES);
  tl_copy_rows<FW_Z, 7>(tb, spo, F_Z);
  tl_copy_rows<FW_ZB, N_ITER - F_ZLA>(tb, spo, F_ZLA);
  tl_copy_rows<FW_K, N_FACT>(tb, sp, F_K);
  tl_commit();
}
// Inside the stage loops the same copies are issued in two halves, each its own commit group -- (a) at the top of the
// stage body, (b) in the middle of it -- so that a stage's LDGSTS do not reach the load/store unit in one burst (see
// ascent_ipm_dc.cuh for the measurement).  The wait is unchanged: before stage k is consumed everything but the newest
// group, part (a) of the next stage, has landed.
LM_HD void ev7_stage_copy_a(const Mesh& M, const Ws& W, int k, int so, bool read_pi) {
  const TileRef tb = tl_buf(W, k);
  tl_copy_mesh(tb, M, k);
  const double* sp = W.stage(k);
  tl_copy_rows<EV_CUR, N_CUR>(tb, ws_opaque(sp + so * LANES), F_U);
  tl_copy(tb, EV_DU, sp + F_DU * LANES);
  if (read_pi) tl_copy_rows<EV_PI, 6>(tb, sp, F_PI);
  tl_commit();
}
LM_HD void ev7_stage_copy_b(const Ws& W, int k, int so) {
  const TileRef tb = tl_buf(W, k);
  const double* sm = ws_opaque(W.stage(k) - W.SS);
  tl_copy_rows<EV_PZ, 6>(tb, ws_opaque(sm + so * LANES), F_Z);
  tl_copy_rows<EV_PDS, 6>(tb, sm, F_DS);
  tl_commit();
}
LM_HD void bk7_stage_copy_a(const Mesh& M, const Ws& W, int k, int so) {
  const TileRef tb = tl_buf(W, k);
  tl_copy_mesh(tb, M, k);
  tl_copy_rows<BK_CUR, N_CUR>(tb, ws_opaque(W.stage(k) + so * LANES), F_U);
  tl_commit();
}
LM_HD void bk7_stage_copy_b(const Ws& W, int k, int so) {
  const TileRef tb = tl_buf(W, k);
  tl_copy_rows<BK_PZ, 6>(tb, ws_opaque(W.stage(k) + so * LANES - W.SS), F_Z);
  tl_commit();
}
LM_HD void fw7_stage_copy_a(const Mesh& M, const Ws& W, int k, int so) {
  const TileRef tb = tl_buf(W, k);
  tl_copy_mesh(tb, M, k);
  const double* spo = ws_opaque(W.stage(k) + so * LANES);
  tl_copy_rows<FW_Z, 7>(tb, spo, F_Z);
  tl_copy_rows<FW_ZB, N_ITER - F_ZLA>(tb, spo, F_ZLA);
  tl_commit();
}
LM_HD void fw7_stage_copy_b(const Ws& W, int k) {
  const TileRef tb = tl_buf(W, k);
  tl_copy_rows<FW_K, N_FACT>(tb, W.stage(k), F_K);
  tl_commit();
}

enum : int { EV_READ_PI = 0, EV_NEWTON = 1, EV_LSQ = 2 };

LM_SWEEP void eval_pass(const Params& P, const Mesh& M, const Options& O, const Ws& W, int src, int dst,
                           const Scal& c0, const TermStep& ts, double mu, double dw, double alpha,
                           double alpha_z, double alpha_lam, int mode, Scal& t, double* pimax_out) {
  const int N = M.N;
  const int so = src * N_ITER, dd = dst * N_ITER;
  tl_begin();
  ev7_stage_copy(M, W, N, so, mode == EV_READ_PI);
  const double tf0 = c0.tf, dtf = ts.dtf;
  t.tf = tf0 + alpha * dtf;
  const double tf = t.tf;
  const bool ls = (mode == EV_LSQ);
  double theta = 0, prim = 0, dual = 0, sumlog = 0, cmin = 1e300, cmax = 0, slam = 0, sz = 0;
  double gtf = 0;                          // d Lagrangian / d tf accumulated over stages
  double pimax = 0;
  bool bad = false;
  // ---- terminal scalars of the trial point ----
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
  // state of node k at the old point and its step (carried in registers: node k-1 is read while
  // node k is processed, because the defect of node k needs the trial state of node k-1)
  double zo[6], ds[6];
  {
    const double* sp = W.stage(N);
#pragma unroll
    for (int i = 0; i < 6; ++i) { zo[i] = WS_AT(sp, so + F_Z + i); ds[i] = WS_AT(sp, F_DS + i); }
  }
  double lam_next[6] = {0, 0, 0, 0, 0, 0};   // trial multipliers of node k+1
  double pi_next[6] = {0, 0, 0, 0, 0, 0};    // adjoint of node k+1
  for (int k = N; k >= 1; --k) {
    double* sp = W.stage(k);
    // stage the rows of the next stage, then wait for this stage's tile
    if (k > 1) ev7_stage_copy_a(M, W, k - 1, so, mode == EV_READ_PI); else tl_commit();
    tl_wait_prev();
    const TileRef tb = tl_buf(W, k);
    double z[6], zpo[6], dsp[6], zp[6], lam[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) z[i] = fma(alpha, ds[i], zo[i]);
#pragma unroll
    for (int i = 0; i < 6; ++i) {                 // node k-1 (node 0 rows are zeros)
      zpo[i] = tl_ld(tb, EV_PZ + i); dsp[i] = tl_ld(tb, EV_PDS + i);
      zp[i] = fma(alpha, dsp[i], zpo[i]);
    }
    const double u_old = TL7_CUR(tb, EV_CUR, F_U);
    const double du = tl_ld(tb, EV_DU);
    const double u = fma(alpha, du, u_old);
    double lam_old[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) lam_old[i] = TL7_CUR(tb, EV_CUR, F_LAM + i);
    double zla = TL7_CUR(tb, EV_CUR, F_ZLA), zua = TL7_CUR(tb, EV_CUR, F_ZUA);
    double zlu = TL7_CUR(tb, EV_CUR, F_ZLU), zuu = TL7_CUR(tb, EV_CUR, F_ZUU);
    const double kap = tl_ld(tb, TL_H) * P.T;
    const double taum = P.mT * tl_ld(tb, TL_TAU);
    // ---- new multipliers pi_k ----
    double pi[6];
    if (mode != EV_READ_PI) {
      Accel1 f0;
      accel_first(P, zo[0], zo[2], zo[4], taum * tf0, f0);
      StageJac J0;
      stagejac_build(P, kap, tf0, taum, f0, zo[1], zo[3], zo[5], u_old, J0);
      stagejac_invert(J0);
      StageQ q;
      stage_hessian(P, f0, J0, kap, taum, lam_old, zo[4], u_old, zla, zua, zlu, zuu, mu, dw, ls, q);
      double g[7];
      g[0] = pi_next[0] - (q.q00 * ds[0] + q.q02 * ds[2] + q.q04 * ds[4] + q.q06 * dtf);
      g[1] = pi_next[1] - (q.d * ds[1] + q.q16 * dtf);
      g[2] = pi_next[2] - (q.q02 * ds[0] + q.q22 * ds[2] + q.q24 * ds[4] + q.q26 * dtf);
      g[3] = pi_next[3] - (q.d * ds[3] + q.q36 * dtf);
      g[4] = pi_next[4] - (q.q04 * ds[0] + q.q24 * ds[2] + q.q44 * ds[4] + q.q46 * dtf + q.q4);
      g[5] = P.coup5 * pi_next[5] - (q.d * ds[5] + q.q56 * dtf);
      g[6] = 0.0;
      if (k == N) {
        TermQP tq;
        terminal_qp(P, O, c0, zo, mu, dw, ls, tq);
#pragma unroll
        for (int i = 0; i < 4; ++i)
          g[i] -= tq.H[i][0] * ds[0] + tq.H[i][1] * ds[1] + tq.H[i][2] * ds[2] + tq.H[i][3] * ds[3] + tq.g[i];
      }
      solveET(J0, g);
#pragma unroll
      for (int i = 0; i < 6; ++i) { pi[i] = g[i]; WS_AT(sp, F_PI + i) = g[i]; pimax = dmax(pimax, fabs(g[i])); }
    } else {
#pragma unroll
      for (int i = 0; i < 6; ++i) pi[i] = tl_ld(tb, EV_PI + i);
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) lam[i] = fma(alpha_lam, pi[i] - lam_old[i], lam_old[i]);
    if (k > 1) ev7_stage_copy_b(W, k - 1, so); else tl_commit();     // second half of the next stage's tile
    // ---- bound multipliers: dz = (mu - z dx)/d - z  (old d, old z), then the kappa_Sigma clip ----
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
      // kappa_Sigma safeguard: one (rarely taken) branch for the four multipliers of the node
      const double c1 = dLa * zla, c2 = dUa * zua, c3 = dLu * zlu, c4 = dUu * zuu;
      const double hi = 1e10 * mu, lo = 1e-10 * mu;
      if (dmax(dmax(c1, c2), dmax(c3, c4)) > hi || dmin(dmin(c1, c2), dmin(c3, c4)) < lo) {
        zla = clip_mult(zla, dLa, mu); zua = clip_mult(zua, dUa, mu);
        zlu = clip_mult(zlu, dLu, mu); zuu = clip_mult(zuu, dUu, mu);
      }
    }
    sumlog += lm_log_pos((dLa * dUa) * (dLu * dUu));
    {
      const double c1 = dLa * zla, c2 = dUa * zua, c3 = dLu * zlu, c4 = dUu * zuu;
      cmin = dmin(cmin, dmin(dmin(c1, c2), dmin(c3, c4)));
      cmax = dmax(cmax, dmax(dmax(c1, c2), dmax(c3, c4)));
    }
    sz += (zla + zua) + (zlu + zuu);
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
    c[5] = z[5] - P.coup5 * zp[5] - J.beta * u;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      const double ac = fabs(c[i]);
      theta += ac;
      prim = dmax(prim, ac);
      slam += fabs(lam[i]);
    }
    // ---- Lagrangian gradient wrt s_k: E_k^T lam_k - lam_{k+1} + bound / terminal terms ----
    double res[6];
    applyET6(J, lam, res);
    res[4] += zua - zla;
    if (k == N) {
      Terminal T;
      terminal_eval(P, z[0], z[1], z[2], z[3], T);
      const double c1 = T.g1 - t.sg1, c2 = T.g2 - t.sg2, c3 = T.g3;
      theta += fabs(c1) + fabs(c2) + fabs(c3);
      prim = dmax(prim, dmax(fabs(c1), dmax(fabs(c2), fabs(c3))));
      // multipliers of g1, g2 are -zs1, -zs2 (slack stationarity)
      const double rinv = 1.0 / T.rT;
      res[0] += -t.zs1 * T.Yb * rinv + t.nu3 * z[1];
      res[2] += -t.zs1 * z[2] * rinv + t.nu3 * z[3];
      res[1] += -t.zs2 * 2.0 * z[1] + t.nu3 * T.Yb;
      res[3] += -t.zs2 * 2.0 * z[3] + t.nu3 * z[2];
    } else {
#pragma unroll
      for (int i = 0; i < 5; ++i) res[i] -= lam_next[i];
      res[5] -= P.coup5 * lam_next[5];
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) dual = dmax(dual, fabs(res[i]));
    dual = dmax(dual, fabs(-J.beta * lam[5] - zlu + zuu));     // d L / d u_k
    gtf -= J.e0 * lam[0] + J.e1 * lam[1] + J.e2 * lam[2] + J.e3 * lam[3] + J.e4 * lam[4] + J.e5 * lam[5];
    // ---- write the trial iterate, shift the pipeline ----
double* spd = ws_opaque(sp + dd * LANES);
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      WS_AT(spd, F_Z + i) = z[i]; WS_AT(spd, F_LAM + i) = lam[i];
      lam_next[i] = lam[i]; pi_next[i] = pi[i]; zo[i] = zpo[i]; ds[i] = dsp[i];
    }
    WS_AT(spd, F_U) = u;
    WS_AT(spd, F_ZLA) = zla; WS_AT(spd, F_ZUA) = zua;
    WS_AT(spd, F_ZLU) = zlu; WS_AT(spd, F_ZUU) = zuu;
  }
  dual = dmax(dual, fabs(gtf));
  t.theta = theta;
  t.fobj = O.obj_scale * tf;
  t.sumlog = bad ? -1e300 : sumlog;
  t.prim_inf = prim; t.dual_inf = dual; t.cmin = cmin; t.cmax = cmax; t.sum_lam = slam; t.sum_z = sz;
  if (bad || !(theta == theta)) t.theta = 1e300;
  if (pimax_out) *pimax_out = pimax;
}

// ---------------------------------------------------------------------------------------
// backward Riccati sweep = block LDL^T of the KKT matrix in stage order.
// Returns false if a pivot shows wrong inertia (caller increases delta_w and retries).
//
// Per stage:  W = Q_k + P_k,  Wt = Abar^T W Abar  with  Abar = E_k^{-1} = T1 T2 T3,
//   T1 = diag(A11, I)   A11 = inverse of the (y,vy,x,vx) block of E          (4x4, applied as an operator)
//   T2 = [I C; 0 I]     C = [ga | 0 | e]  couples (angle, tf) into the velocity rows
//   T3 = diag(I, A22)   A22 = [[1, al, e4+al*e5], [0, 1, e5], [0, 0, 1]]      (angle, angledot, tf chain)
// then the control is condensed (it enters through the angledot row only).  Only the feedback
// gains K_k, k_k leave the SM; the cost-to-go P, p lives in registers.
// ---------------------------------------------------------------------------------------
LM_SWEEP bool riccati_backward(const Params& P, const Mesh& M, const Options& O, const Ws& W, int src,
                                  const Scal& c0, double mu, double dw, bool ls_arg, double* dtf_out) {
  const bool ls = ls_arg;
  // ls == true: least-squares multiplier estimate (IPOPT section 3.6): Hessian := I, defects := 0,
  // gradient := grad f - zL + zU.
  const int N = M.N;
  const double tf = c0.tf;
  const int so = src * N_ITER;
  tl_begin();
  bk7_stage_copy(M, W, N, so);
  // cost-to-go Hessian in blocks: A = (p,p) 4x4 symmetric (full storage), B = (p,q) 4x3,
  // Cq = (q,q) 3x3 symmetric (upper triangle used); p = (y,vy,x,vx), q = (angle, angledot, tf)
  double A[4][4], Bm[4][3], C00, C01, C02, C11, C12, C22;
  double pv[7];
  double zn[6];    // state at node k
  {
    const double* sp = W.stage(N);
#pragma unroll
    for (int i = 0; i < 6; ++i) zn[i] = WS_AT(sp, so + F_Z + i);
  }
  {
    TermQP tq;
    terminal_qp(P, O, c0, zn, mu, dw, ls, tq);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int j = 0; j < 4; ++j) A[i][j] = tq.H[i][j];
#pragma unroll
      for (int j = 0; j < 3; ++j) Bm[i][j] = 0.0;
      pv[i] = tq.g[i];
    }
    C00 = C01 = C02 = C11 = C12 = 0.0;
    C22 = tq.H66;
    pv[4] = 0.0; pv[5] = 0.0; pv[6] = tq.g6;
  }
  bool ok = true;
  for (int k = N; k >= 1; --k) {
    double* sp = W.stage(k);
    if (k > 1) bk7_stage_copy_a(M, W, k - 1, so); else tl_commit();
    tl_wait_prev();
    const TileRef tb = tl_buf(W, k);
    const bool ls = W.ls_flag != 0;      // shadows the argument: a shared-memory load per stage
    double lam[6], zm[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) lam[i] = TL7_CUR(tb, BK_CUR, F_LAM + i);
#pragma unroll
    for (int i = 0; i < 6; ++i) zm[i] = tl_ld(tb, BK_PZ + i);       // node k-1 (node 0 rows are zeros)
    const double u = TL7_CUR(tb, BK_CUR, F_U);
    const double zla = TL7_CUR(tb, BK_CUR, F_ZLA), zua = TL7_CUR(tb, BK_CUR, F_ZUA);
    const double zlu = TL7_CUR(tb, BK_CUR, F_ZLU), zuu = TL7_CUR(tb, BK_CUR, F_ZUU);
    const double kap = tl_ld(tb, TL_H) * P.T;
    const double taum = P.mT * tl_ld(tb, TL_TAU);
    Accel1 f;
    accel_first(P, zn[0], zn[2], zn[4], taum * tf, f);
    StageJac J;
    stagejac_build(P, kap, tf, taum, f, zn[1], zn[3], zn[5], u, J);
    stagejac_invert(J);
    const double al = J.al;
    // ---- W = Q_k + P_k (in place), g = q_k + p_k ----
    StageQ q;
    stage_hessian(P, f, J, kap, taum, lam, zn[4], u, zla, zua, zlu, zuu, mu, dw, ls, q);
    A[0][0] += q.q00;
    A[2][0] += q.q02; A[0][2] += q.q02;
    A[2][2] += q.q22;
    A[1][1] += q.d; A[3][3] += q.d;
    Bm[0][0] += q.q04; Bm[2][0] += q.q24;
    C00 += q.q44; C11 += q.d;
    Bm[0][2] += q.q06; Bm[1][2] += q.q16; Bm[2][2] += q.q26; Bm[3][2] += q.q36;
    C02 += q.q46; C12 += q.q56; C22 += q.q66;
    pv[4] += q.q4;
    // ---- defect ----
    double c[6];
    if (!ls) {
      c[0] = zn[0] - zm[0] - al * zn[1];
      c[1] = zn[1] - zm[1] - al * f.ay;
      c[2] = zn[2] - zm[2] - al * zn[3];
      c[3] = zn[3] - zm[3] - al * f.ax;
      c[4] = zn[4] - zm[4] - al * zn[5];
      c[5] = zn[5] - P.coup5 * zm[5] - J.beta * u;
    } else {
#pragma unroll
      for (int i = 0; i < 6; ++i) c[i] = 0.0;
    }
    // ---- T1: A <- A11^T A A11,  B <- A11^T B ----
#pragma unroll
    for (int j = 0; j < 4; ++j) applyA11T(J, A[0][j], A[1][j], A[2][j], A[3][j]);
#pragma unroll
    for (int i = 0; i < 4; ++i) applyA11T(J, A[i][0], A[i][1], A[i][2], A[i][3]);
#pragma unroll
    for (int j = 0; j < 3; ++j) applyA11T(J, Bm[0][j], Bm[1][j], Bm[2][j], Bm[3][j]);
    if (k > 1) bk7_stage_copy_b(W, k - 1, so); else tl_commit();     // second half of the next stage's tile
    // ---- T2: couple (angle, tf) into the velocity rows ----
    {
      double AC0[4], AC2[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        AC0[i] = A[i][1] * J.ga1 + A[i][3] * J.ga3;
        AC2[i] = A[i][0] * J.e0 + A[i][1] * J.e1 + A[i][2] * J.e2 + A[i][3] * J.e3;
      }
      double CtB0[3], CtB2[3];
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        CtB0[j] = J.ga1 * Bm[1][j] + J.ga3 * Bm[3][j];
        CtB2[j] = J.e0 * Bm[0][j] + J.e1 * Bm[1][j] + J.e2 * Bm[2][j] + J.e3 * Bm[3][j];
      }
      const double CtAC00 = J.ga1 * AC0[1] + J.ga3 * AC0[3];
      const double CtAC02 = J.ga1 * AC2[1] + J.ga3 * AC2[3];
      const double CtAC22 = J.e0 * AC2[0] + J.e1 * AC2[1] + J.e2 * AC2[2] + J.e3 * AC2[3];
      C00 += 2.0 * CtB0[0] + CtAC00;
      C01 += CtB0[1];
      C02 += CtB0[2] + CtB2[0] + CtAC02;
      C12 += CtB2[1];
      C22 += 2.0 * CtB2[2] + CtAC22;
#pragma unroll
      for (int i = 0; i < 4; ++i) { Bm[i][0] += AC0[i]; Bm[i][2] += AC2[i]; }
    }
    // ---- T3: (angle, angledot, tf) chain ----
    {
      const double s = J.e4 + al * J.e5, e5 = J.e5;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const double b0 = Bm[i][0], b1 = Bm[i][1];
        Bm[i][2] += s * b0 + e5 * b1;
        Bm[i][1] = fma(al, b0, b1);
      }
      // X = Cq A22 (rows), then A22^T X
      const double x00 = C00, x01 = al * C00 + C01, x02 = s * C00 + e5 * C01 + C02;
      const double x11 = al * C01 + C11, x12 = s * C01 + e5 * C11 + C12;   // row 1 of X: [C01, x11, x12]
      const double x22 = s * C02 + e5 * C12 + C22;                          // row 2 of X: [C02,  . , x22]
      C00 = x00; C01 = x01; C02 = x02;
      C11 = al * x01 + x11;
      C12 = al * x02 + x12;
      C22 = s * x02 + e5 * x12 + x22;
    }
    solveET(J, pv);                      // g~ = E^{-T} (q + p)
    // ---- condense the control (enters through the angledot row: q-index 1) ----
    const double beta = J.beta;
    const double Ruu = q.R + beta * beta * C11;
    double Rux[7];
#pragma unroll
    for (int i = 0; i < 4; ++i) Rux[i] = beta * Bm[i][1];
    Rux[4] = beta * C01; Rux[5] = beta * C11; Rux[6] = beta * C12 + q.sig;
    double rx[7];
#pragma unroll
    for (int i = 0; i < 4; ++i)
      rx[i] = pv[i] - (A[i][0] * c[0] + A[i][1] * c[1] + A[i][2] * c[2] + A[i][3] * c[3] + Bm[i][0] * c[4] + Bm[i][1] * c[5]);
    rx[4] = pv[4] - (Bm[0][0] * c[0] + Bm[1][0] * c[1] + Bm[2][0] * c[2] + Bm[3][0] * c[3] + C00 * c[4] + C01 * c[5]);
    rx[5] = pv[5] - (Bm[0][1] * c[0] + Bm[1][1] * c[1] + Bm[2][1] * c[2] + Bm[3][1] * c[3] + C01 * c[4] + C11 * c[5]);
    rx[6] = pv[6] - (Bm[0][2] * c[0] + Bm[1][2] * c[1] + Bm[2][2] * c[2] + Bm[3][2] * c[3] + C02 * c[4] + C12 * c[5]);
    const double ru = q.r + beta * rx[5];
    // d defect_k / d s_{k-1} = -D with D = diag(1,1,1,1,1,coup5,1): the previous node sees the
    // angledot column scaled by coup5 (0 in the circular model)
    const double cp = P.coup5;
    Rux[5] *= cp; rx[5] *= cp;
#pragma unroll
    for (int i = 0; i < 4; ++i) Bm[i][1] *= cp;
    C01 *= cp; C11 *= cp * cp; C12 *= cp;
    if (!(Ruu > 0.0) || !(Ruu < 1e300)) ok = false;
    const double Rinv = lm_rcp(Ruu);
    double RuxS[7];
#pragma unroll
    for (int i = 0; i < 7; ++i) { RuxS[i] = Rux[i] * Rinv; WS_AT(sp, F_K + i) = -RuxS[i]; }
    WS_AT(sp, F_KFF) = -ru * Rinv;
    // P_{k-1} = Wt - Rux Rux^T / Ruu   (symmetrised)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int j = 0; j <= i; ++j) {
        const double v = 0.5 * (A[i][j] + A[j][i]) - Rux[i] * RuxS[j];
        A[i][j] = v; A[j][i] = v;
      }
#pragma unroll
      for (int j = 0; j < 3; ++j) Bm[i][j] -= Rux[i] * RuxS[4 + j];
    }
    C00 -= Rux[4] * RuxS[4]; C01 -= Rux[4] * RuxS[5]; C02 -= Rux[4] * RuxS[6];
    C11 -= Rux[5] * RuxS[5]; C12 -= Rux[5] * RuxS[6]; C22 -= Rux[6] * RuxS[6];
#pragma unroll
    for (int i = 0; i < 7; ++i) pv[i] = rx[i] - RuxS[i] * ru;
#pragma unroll
    for (int i = 0; i < 6; ++i) zn[i] = zm[i];
    if (!ok) return false;
  }
  // free initial tf: minimise 0.5 P66 dtf^2 + p6 dtf
  if (!(C22 > 0.0)) return false;
  *dtf_out = -pv[6] / C22;
  return true;
}

// ---------------------------------------------------------------------------------------
// forward sweep: recover the primal Newton step, fraction-to-boundary limits and d(phi)/d(alpha)
// ---------------------------------------------------------------------------------------
struct StepInfo { double a_max, a_z, dphi, dxmax; };

// running maximum of num/den (den > 0) without dividing: keeps the pair
struct RatioMax {
  double n, d;
  LM_HD void init() { n = 0.0; d = 1.0; }
  LM_HD void push(double num, double den) { if (num * d > n * den) { n = num; d = den; } }
};

LM_SWEEP void riccati_forward(const Params& P, const Mesh& M, const Options& O, const Ws& W, int src,
                                 const Scal& c0, double mu, double tau, double dtf, bool ls_arg, TermStep& ts,
                                 StepInfo& si) {
  const bool ls = ls_arg;
  const int N = M.N;
  const double tf = c0.tf;
  const int so = src * N_ITER;
  tl_begin();
  fw7_stage_copy(M, W, 1, so);
  double ds[7] = {0, 0, 0, 0, 0, 0, dtf};
  double zm[6] = {0, 0, 0, 0, 0, 0};
  double dphi = 0.0, dxmax = fabs(dtf);
  RatioMax rp, rz;      // max of (-dx/slack) over primal bounds, (-dz/z) over bound multipliers
  rp.init(); rz.init();
  const double cw = ls ? 0.0 : 1.0;   // defects are dropped in the least-squares mode
  for (int k = 1; k <= N; ++k) {
    double* sp = W.stage(k);
    if (k < N) fw7_stage_copy_a(M, W, k + 1, so); else tl_commit();
    tl_wait_prev();
    const TileRef tb = tl_buf(W, k);
    const bool ls = W.ls_flag != 0;      // shadows the argument: a shared-memory load per stage
    double zn[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) zn[i] = tl_ld(tb, FW_Z + i);
    const double u = tl_ld(tb, FW_Z + 6);
    const double kap = tl_ld(tb, TL_H) * P.T;
    const double taum = P.mT * tl_ld(tb, TL_TAU);
    Accel1 f;
    accel_first(P, zn[0], zn[2], zn[4], taum * tf, f);
    StageJac J;
    stagejac_build(P, kap, tf, taum, f, zn[1], zn[3], zn[5], u, J);
    stagejac_invert(J);
    const double al = J.al;
    double du = tl_ld(tb, FW_K + 7);
#pragma unroll
    for (int i = 0; i < 7; ++i) du = fma(tl_ld(tb, FW_K + i), ds[i], du);
    double xi[7];
    xi[0] = ds[0] - cw * (zn[0] - zm[0] - al * zn[1]);
    xi[1] = ds[1] - cw * (zn[1] - zm[1] - al * f.ay);
    xi[2] = ds[2] - cw * (zn[2] - zm[2] - al * zn[3]);
    xi[3] = ds[3] - cw * (zn[3] - zm[3] - al * f.ax);
    xi[4] = ds[4] - cw * (zn[4] - zm[4] - al * zn[5]);
    xi[5] = P.coup5 * ds[5] - cw * (zn[5] - P.coup5 * zm[5] - J.beta * u) + J.beta * du;
    xi[6] = dtf;
    solveE(J, xi);
    if (k < N) fw7_stage_copy_b(W, k + 1); else tl_commit();         // second half of the next stage's tile
#pragma unroll
    for (int i = 0; i < 6; ++i) { ds[i] = xi[i]; WS_AT(sp, F_DS + i) = xi[i]; zm[i] = zn[i]; dxmax = dmax(dxmax, fabs(xi[i])); }
    WS_AT(sp, F_DU) = du;
    dxmax = dmax(dxmax, fabs(du));
    // fraction to the boundary (IPOPT eq. 15) for angle and control, and their multipliers
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
  // terminal slacks and multipliers
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
  // alpha_max = min(1, tau / max ratio)
  si.a_max = (rp.n > tau * rp.d) ? tau * rp.d / rp.n : 1.0;
  si.a_z = (rz.n > tau * rz.d) ? tau * rz.d / rz.n : 1.0;
  si.dphi = dphi; si.dxmax = dxmax;
}

// ---------------------------------------------------------------------------------------
// IPM driver pieces
// ---------------------------------------------------------------------------------------
LM_HD double kkt_error(const Scal& s, double mu, int n_eq, int n_bd) {
  const double smax = 100.0;
  const double sd = dmax(smax, (s.sum_lam + s.sum_z) / (double)(n_eq + n_bd)) / smax;
  const double sc = dmax(smax, s.sum_z / (double)n_bd) / smax;
  const double comp = dmax(fabs(s.cmax - mu), fabs(s.cmin - mu));
  return dmax(dmax(s.dual_inf / sd, s.prim_inf), comp / sc);
}

// IPOPT's Compare_le: a <= b up to 10 machine epsilons of a reference magnitude.
LM_HD bool cmp_le(double a, double b, double ref) { return a - b <= 2.2204460492503131e-15 * fabs(ref); }

LM_HD bool filter_ok(const Ctl& c, double th, double ph) {
  for (int i = 0; i < c.nf; ++i)
    if (!cmp_le(th, c.ft[i], c.ft[i]) && !cmp_le(ph, c.fp[i], c.fp[i])) return false;
  return true;
}

LM_HD void filter_add(Ctl& c, double th, double ph) {
  // drop dominated entries, then append (overwrite the weakest if full)
  int n = 0;
  for (int i = 0; i < c.nf; ++i)
    if (!(c.ft[i] >= th && c.fp[i] >= ph)) { c.ft[n] = c.ft[i]; c.fp[n] = c.fp[i]; ++n; }
  if (n == NFILT) {   // merge: keep the envelope conservative by replacing the largest-theta entry
    int w = 0;
    for (int i = 1; i < n; ++i) if (c.ft[i] > c.ft[w]) w = i;
    c.ft[w] = th; c.fp[w] = ph;
  } else { c.ft[n] = th; c.fp[n] = ph; ++n; }
  c.nf = n;
}

// ---------------------------------------------------------------------------------------
// Resumable per-problem driver.  ipm_begin() after the start point is in buffer 0;
// ipm_iterate() performs one iteration (iteration 0 = least-squares multiplier estimate, IPOPT
// section 3.6, which runs through the very same three sweeps) and returns true once the problem
// is finished.  The CUDA kernel calls it in a loop with a block barrier in between so that all
// warps of an SM run the same sweep at the same time (instruction-cache locality).
// ---------------------------------------------------------------------------------------
enum : int { PH_LSQ = 0, PH_NEWTON = 1 };

struct IpmState {
  bool warm;        // start point carries its own multipliers (skip the least-squares estimate)
  bool from_guess;  // start point supplied by the caller (lmato_set_initial_guess)
  unsigned char start;   // rung of the collocation start ladder (ascent_colloc.cuh), set by its ipm_start only; one
                         // byte, so that it fills padding and IpmState keeps its size on every other kernel's stack
  int iters_prior;  // iterations of an abandoned warm / caller-supplied start of the same problem (reported with the rest)
  Scal cur;
  Ctl ctl;
  TermStep ts;
  double err0;
  int src;
  int phase;
  int polish_left;
  bool polishing;
};

struct SolveOut { double tf; int status; int iters; double kkt; double mu; int cur; };

LM_HD void ipm_begin(const Options& O, IpmState& S) {
  S.ts.dtf = S.ts.dsg1 = S.ts.dsg2 = S.ts.dzs1 = S.ts.dzs2 = S.ts.dnu3 = S.ts.dzLt = S.ts.dzUt = 0.0;
  S.ctl.mu = O.mu_init;
  S.ctl.tau = dmax(O.tau_min, 1.0 - S.ctl.mu);
  S.ctl.nf = 0; S.ctl.dw_last = 0.0; S.ctl.iter = 0; S.ctl.status = ST_RUNNING;
  S.ctl.tiny_steps = 0; S.ctl.null_steps = 0; S.ctl.iter_best = 0; S.ctl.err_best = 1e300;
  S.ctl.theta_max = 1e300; S.ctl.theta_min = 0.0;
  S.err0 = 1e300;
  S.src = 0;
  S.phase = PH_LSQ;
  S.polish_left = -1;
  S.polishing = false;
  S.warm = false;
  S.from_guess = false;
  S.iters_prior = 0;
}

// Start of one problem on the sweeps SW: the caller's start point if G has one (lmato_set_initial_guess), else the
// batch reference if `ref` holds one (it then also gives the barrier parameter), else the built-in roll-out.
template <class SW, class WS>
LM_HD void ipm_start(const Params& P, const Mesh& M, const Options& O, const WS& W, const GuessSrc& G, const double* ref,
                     IpmState& S) {
  ipm_begin(O, S);
  double mu0 = 0.0;
  if (G.traj) {
    start_from_guess<SW>(P, M, O, W, G, S.cur);
    S.from_guess = true;
  } else if (ref && start_from_ref<SW>(P, M, O, W, ref, S.cur, &mu0)) {
    S.warm = true;
    S.ctl.mu = mu0;
    S.ctl.tau = dmax(O.tau_min, 1.0 - mu0);
  } else {
    start_rollout<SW>(P, M, O, W, S.cur);
  }
}

// After ipm_iterate_t has finished a problem: a warm start, or a caller's start point, that did not converge is
// restarted from the built-in roll-out, with the iterations spent so far reported with the rest.  (IPOPT would enter
// its feasibility restoration phase from such a point, e.g. from the reference's all-zero start values LO:39, 83-96;
// this solver's substitute is a start point that is dynamically feasible by construction.)  Returns true if it
// restarted.
template <class SW, class WS>
LM_HD bool ipm_restart(const Params& P, const Mesh& M, const Options& O, const WS& W, IpmState& S) {
  if (!(S.warm || S.from_guess) || S.ctl.status == ST_CONVERGED) return false;
  const int prior = S.iters_prior + S.ctl.iter;
  ipm_begin(O, S);
  S.iters_prior = prior;
  start_rollout<SW>(P, M, O, W, S.cur);
  return true;
}

// Node k of iterate `cur` in a thread's workspace column with the iterate rows of SW (Sweeps7 / Sweeps8): x = the six
// states and the control, lam = the multipliers of the ydot, xdot and angledot rows; either may be null.
template <class SW>
LM_HD void ws_node(const Ws& W, int cur, int k, double* x, double* lam) {
  const double* sp = W.stage(k);
  if (x) {
    for (int i = 0; i < 6; ++i) x[i] = WS_AT(sp, cur * SW::NITER + SW::FZ + i);
    x[6] = WS_AT(sp, cur * SW::NITER + SW::FU);
  }
  if (!lam) return;
  lam[0] = WS_AT(sp, cur * SW::NITER + SW::FLAM + 1);
  lam[1] = WS_AT(sp, cur * SW::NITER + SW::FLAM + 3);
  lam[2] = WS_AT(sp, cur * SW::NITER + SW::FLAM + 5);
}

// The multipliers of node k of iterate `cur` (same layouts as ws_node): d[0..5] those of the six defect rows, d[6] that
// of the angle's upper bound, d[7], d[8] those of the control's lower and upper bound.
template <class SW>
LM_HD void ws_node_duals(const Ws& W, int cur, int k, double* d) {
  const double* sp = W.stage(k);
  for (int i = 0; i < 6; ++i) d[i] = WS_AT(sp, cur * SW::NITER + SW::FLAM + i);
  for (int i = 0; i < 3; ++i) d[6 + i] = WS_AT(sp, cur * SW::NITER + SW::FZLA + 1 + i);
}

// Sweeps policy of the 7-state formulation (dcost = 0); ascent_ipm_dc.cuh provides the 8-state one.
struct Sweeps7 {
  enum : int { NFIELDS = N_FIELDS, NITER = N_ITER, FZ = F_Z, FU = F_U, FLAM = F_LAM, FZLA = F_ZLA, REFROWS = REF_ROWS,
               MOVE_TERM = 0, LANES_PER_PROBLEM = 1, STORES_REF = 0 };
  LM_HD static int n_eq(const Ws&, int N) { return 6 * N + 3; }
  LM_HD static int n_bd(const Ws&, int N) { return 4 * N + 4; }
  LM_HD static bool backward(const Params& P, const Mesh& M, const Options& O, const Ws& W, int src, const Scal& c0,
                             double mu, double dw, bool ls, double* dtf) {
    return riccati_backward(P, M, O, W, src, c0, mu, dw, ls, dtf);
  }
  LM_HD static void forward(const Params& P, const Mesh& M, const Options& O, const Ws& W, int src, const Scal& c0,
                            double mu, double tau, double dtf, bool ls, TermStep& ts, StepInfo& si) {
    riccati_forward(P, M, O, W, src, c0, mu, tau, dtf, ls, ts, si);
  }
  LM_HD static void eval(const Params& P, const Mesh& M, const Options& O, const Ws& W, int src, int dst,
                         const Scal& c0, const TermStep& ts, double mu, double dw, double alpha, double alpha_z,
                         double alpha_lam, int mode, Scal& t, double* pimax) {
    eval_pass(P, M, O, W, src, dst, c0, ts, mu, dw, alpha, alpha_z, alpha_lam, mode, t, pimax);
  }
  // start points (start_rollout, start_from_guess, start_from_ref): node k into this layout's rows, node 0 pinned at
  // zero (LO:145-151: its state and step rows are literal zeros, so that the sweeps read "node k-1" without a special
  // case at k = 1)
  LM_HD static void store_node(const Ws& W, int k, const double* x) {
    double* sp = W.stage(k);
#pragma unroll
    for (int f = 0; f < NODE_N7; ++f)
      if (f != NODE_LAM + 6) WS_AT(sp, row7(f)) = x[f];
#pragma unroll
    for (int i = 0; i < N_STEP; ++i) WS_AT(sp, R_STEP + i) = 0.0;
  }
  LM_HD static void zero_node0(const Ws& W) {
    double* s0 = W.stage(0);
#pragma unroll
    for (int i = 0; i < 6; ++i) { WS_AT(s0, F_Z + i) = 0.0; WS_AT(s0, N_ITER + F_Z + i) = 0.0; WS_AT(s0, F_DS + i) = 0.0; }
  }
  LM_HD static void node(const Ws& W, int cur, int k, double* x, double* lam) { ws_node<Sweeps7>(W, cur, k, x, lam); }
  LM_HD static void node_duals(const Ws& W, int cur, int k, double* d) { ws_node_duals<Sweeps7>(W, cur, k, d); }
  LM_HD static void remerit(const Mesh&, const Options&, const Ws&, int, double, Scal&) {}
};

template <class SW, class WS>
LM_HD bool ipm_iterate_t(const Params& P, const Mesh& M, const Options& O, const WS& W, IpmState& S) {
  Ctl& ctl = S.ctl;
  Scal& cur = S.cur;
  const int N = M.N;
  const int n_eq = SW::n_eq(W, N);
  const int n_bd = SW::n_bd(W, N);
  const bool ls = (S.phase == PH_LSQ);
  W.ls_flag = ls ? 1 : 0;
  if (!ls) {
    S.err0 = kkt_error(cur, 0.0, n_eq, n_bd);
    // barrier parameter update (IPOPT eq. 7)
    const double mu_min = O.tol * O.mu_min_factor;
    // (the sub-problem tolerance kappa_eps*mu is floored at tol: below that it would ask for more
    //  than the final test does, and more than FP64 can deliver for the dual residual)
    bool mu_changed = false;
    while (kkt_error(cur, ctl.mu, n_eq, n_bd) <= dmax(O.kappa_eps * ctl.mu, O.tol) && ctl.mu > mu_min * (1.0 + 1e-12)) {
      ctl.mu = dmax(mu_min, dmin(O.kappa_mu * ctl.mu, pow(ctl.mu, S.warm ? O.theta_mu_warm : O.theta_mu)));
      ctl.tau = dmax(O.tau_min, 1.0 - ctl.mu);
      ctl.nf = 0;
      mu_changed = true;
    }
    if (mu_changed) SW::remerit(M, O, W, S.src, ctl.mu, cur);
    // Converged = scaled KKT error <= tol with the barrier parameter at its floor.  Requiring the
    // floor pins the final point on the central path: the control on the singular arc is a nearly
    // flat direction of this NLP and moves like O(mu / sigma_min) (DESIGN.md "Tolerance").
    if (S.err0 <= O.tol && ctl.mu <= mu_min * (1.0 + 1e-12)) {
      // Newton converges quadratically here; `n_polish` more iterations take the point from
      // "residual <= tol" to the FP64 floor, which is what makes two implementations agree on the
      // weakly determined control.  A polish step that fails leaves the converged point in place.
      if (S.polish_left < 0) S.polish_left = O.n_polish;
      if (S.polish_left == 0) { ctl.status = ST_CONVERGED; return true; }
      --S.polish_left;
      S.polishing = true;
    } else {
      S.polishing = false;
    }
    if (ctl.iter >= O.max_iter) { ctl.status = S.polishing ? ST_CONVERGED : ST_MAX_ITER; return true; }
    // Stall guard.  An infeasible problem (e.g. too little pitch authority to reach the orbit with tf <= 1)
    // ends up pressed against a bound, where the fraction-to-boundary rule allows only steps of ~1e-9 that the
    // filter keeps accepting; IPOPT would switch to its restoration phase and report infeasibility.  Here the
    // problem is stopped -- in a batch one such lane would otherwise hold its whole SM for MAX_ITER iterations.
    if (S.err0 < 0.9 * ctl.err_best) { ctl.err_best = S.err0; ctl.iter_best = ctl.iter; }
    // (a batch warm start or a caller's start point that makes no progress is given up much earlier: the lane then
    //  restarts from the built-in roll-out, and every iteration it spends here holds its whole warp)
    const int stall_window = (S.warm || S.from_guess) ? LMATO_WARM_STALL_WINDOW : 100;
    if (!S.polishing && (ctl.tiny_steps >= 10 || ctl.iter - ctl.iter_best >= stall_window)) { ctl.status = ST_STALLED; return true; }
  }
  const bool polishing = S.polishing;
  // factorisation with inertia correction (IPOPT Algorithm IC)
  double dw = 0.0, dtf = 0.0;
  bool fact_ok = false;
  for (int attempt = 0; attempt < 40; ++attempt) {
    if (ls && S.warm) break;
    if (SW::backward(P, M, O, W, S.src, cur, ctl.mu, dw, ls, &dtf)) { fact_ok = true; break; }
    if (ls) break;
    if (dw == 0.0) dw = (ctl.dw_last == 0.0) ? 1e-4 : dmax(1e-20, ctl.dw_last / 3.0);
    else dw *= (ctl.dw_last == 0.0) ? 100.0 : 8.0;
    if (dw > 1e40) break;
  }
  // The three sweeps are inlined into the kernel, so each has exactly one call site: the
  // least-squares multiplier estimate ("iteration 0") runs through the same forward sweep and the
  // same trial loop as a Newton iteration, with its own modes.
  if (!ls && !fact_ok) { ctl.status = polishing ? ST_CONVERGED : ST_INERTIA_FAIL; return true; }
  if (dw > 0.0) ctl.dw_last = dw;
  StepInfo si;
  si.a_max = 0.0; si.a_z = 0.0; si.dphi = 0.0; si.dxmax = 0.0;
  if (fact_ok) SW::forward(P, M, O, W, S.src, cur, ctl.mu, ctl.tau, dtf, ls, S.ts, si);
  if (!ls && (!(si.dphi == si.dphi) || !(si.dxmax < 1e300))) { ctl.status = polishing ? ST_CONVERGED : ST_NUMERICAL; return true; }
  // filter line search (IPOPT section 2.3)
  const double theta = cur.theta;
  const double phi = cur.fobj - ctl.mu * cur.sumlog;
  const double dphi = si.dphi;
  const double g_th = 1e-5, g_ph = 1e-8, s_th = 1.1, s_ph = 2.3, eta = 1e-8, delta = 1.0;
  bool accepted = false, ftype = false, null_step = false;
  // switching condition (IPOPT eq. 19): alpha * (-dphi)^s_ph > delta * theta^s_th.  The two powers
  // do not depend on alpha, so they are evaluated once per iteration.
  const bool sw_possible = !ls && (theta <= ctl.theta_min) && (dphi < 0.0);
  const double sw_lhs = sw_possible ? pow(-dphi, s_ph) : 0.0;
  const double sw_rhs = sw_possible ? delta * pow(theta, s_th) : 0.0;
  // trial parameters.  Least-squares phase: the point does not move; the first pass takes the
  // least-squares multipliers of the defect rows (alpha_lam = 1), and if the solve failed or they
  // are huge a second pass (alpha_lam = 0) keeps the old ones.
  Scal trial;
  double alpha = ls ? 0.0 : si.a_max;
  const double a_z = ls ? 0.0 : si.a_z;
  const double dw_eval = ls ? 0.0 : dw;
  double a_lam = ls ? (fact_ok ? 1.0 : 0.0) : alpha;
  int mode = ls ? (fact_ok ? EV_LSQ : EV_READ_PI) : EV_NEWTON;
  for (int lsi = 0; lsi < O.max_ls; ++lsi) {
    double pimax = 0.0;
    SW::eval(P, M, O, W, S.src, 1 - S.src, cur, S.ts, ctl.mu, dw_eval, alpha, a_z, a_lam, mode, trial, &pimax);
    if (ls) {
      if (mode == EV_LSQ) {
        const bool have = pimax <= 1e3 * dmax(1.0, O.obj_scale) && fabs(S.ts.dnu3) <= 1e3 * dmax(1.0, O.obj_scale);
#if defined(LMATO_TRACE) && !defined(__CUDA_ARCH__)
        printf("LS multipliers: pimax %.3e dnu3 %.3e dtf %.3e -> %s\n", pimax, S.ts.dnu3, dtf, have ? "used" : "discarded");
#endif
        if (!have) { mode = EV_READ_PI; a_lam = 0.0; continue; }
      }
      accepted = true;
      break;
    }
    const double th_t = trial.theta;
    const double ph_t = trial.fobj - ctl.mu * trial.sumlog;
    bool ok = (th_t <= ctl.theta_max) && (ph_t == ph_t) && (ph_t < 1e299) && filter_ok(ctl, th_t, ph_t);
    if (ok) {
      ftype = sw_possible && (alpha * sw_lhs > sw_rhs);
      if (ftype) ok = cmp_le(ph_t - phi, eta * alpha * dphi, phi);
      else ok = cmp_le(th_t, (1.0 - g_th) * theta, theta) || cmp_le(ph_t - phi, -g_ph * theta, phi);
    }
    // Terminal phase (analogue of IPOPT's tiny-step rule): once the violation is below tol before
    // and after the step and the merit changes by less than tol (relative), both filter measures
    // are rounding noise and cannot rank points any more; the Newton step is taken as is.
    if (!ok && lsi == 0 && theta <= O.tol && th_t <= O.tol && (ph_t == ph_t) &&
        fabs(ph_t - phi) <= O.tol * dmax(1.0, fabs(phi))) { ok = true; ftype = true; }
    // A step the filter still rejects after LMATO_LS_NULL halvings (alpha < 2.5e-4 of the fraction-to-boundary step)
    // is not searched further.  Where the search used to go on it either failed after max_ls trials or ended 28-30
    // halvings deep at alpha ~ 1e-9, on the filter's rounding margins: one sweep over all stages per trial, with the
    // lane's whole warp and, at the per-iteration barrier, its CTA in tow -- single such problems cost a
    // 65 536-problem batch 8-25 % of its time (82 -> 90-105 ms).  The trial is taken as it is, a null step, twice
    // per solve; the third time the line search has failed (IPOPT would enter its restoration phase).
    if (!ok && !ls && lsi + 1 >= LMATO_LS_NULL) {
      if (ctl.null_steps < 2 && th_t < 1e299 && (ph_t == ph_t)) { ok = true; ftype = true; null_step = true; }
      else break;
    }
    if (ok) { accepted = true; break; }
    alpha *= 0.5;
    a_lam = alpha;
    mode = EV_READ_PI;
  }
  if (ls) {
    cur = trial; S.src = 1 - S.src;
    ctl.theta_max = 1e4 * dmax(1.0, cur.theta);
    ctl.theta_min = 1e-4 * dmax(1.0, cur.theta);
    S.phase = PH_NEWTON;
    return false;
  }
#if defined(LMATO_TRACE) && !defined(__CUDA_ARCH__)
  if (!accepted) printf("LS FAIL theta %.3e phi %.6e dphi %.3e amax %.3e dx %.2e th_t %.3e ph_t %.6e\n", theta, phi, dphi, si.a_max, si.dxmax, trial.theta, trial.fobj - ctl.mu * trial.sumlog);
#endif
  if (!accepted) { ctl.status = polishing ? ST_CONVERGED : ST_LINESEARCH_FAIL; return true; }
  if (!ftype) filter_add(ctl, (1.0 - g_th) * theta, phi - g_ph * theta);
  cur = trial; S.src = 1 - S.src;
  ++ctl.iter;
  ctl.tiny_steps = (alpha < 1e-6) ? ctl.tiny_steps + 1 : 0;
  if (null_step) ++ctl.null_steps;
#if defined(LMATO_TRACE) && !defined(__CUDA_ARCH__)
  printf("%3d tf %.8f th %.3e err %.3e mu %.1e a %.3e az %.3e dw %.1e dphi %.2e dx %.2e nf %d %s\n", ctl.iter, cur.tf,
         cur.theta, S.err0, ctl.mu, alpha, si.a_z, dw, dphi, si.dxmax, ctl.nf, ftype ? "f" : "h");
#endif
  return false;
}

LM_HD void ipm_result(const IpmState& S, SolveOut& out) {
  out.tf = S.cur.tf; out.status = S.ctl.status; out.iters = S.iters_prior + S.ctl.iter; out.kkt = S.err0; out.mu = S.ctl.mu;
  out.cur = S.src;
}

}  // namespace lmato
