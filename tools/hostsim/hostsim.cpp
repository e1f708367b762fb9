// DEVELOPER TOOL -- NOT PART OF THE PRODUCT.
//
// Compiles the device solver core (csrc/ascent_ipm.cuh) with g++ so that the IPM control
// logic can be stepped through on a box without a GPU.  It is not built by
// __graft_entry__.build(), not loaded by the Python package, not used by any test as the
// thing under test, and bench.py never calls it.  The product path is the CUDA library
// only and fails loudly without it.
//
//   g++ -O2 -std=c++17 -I lunar_module_ascent_trajectory_optimiser_b200/csrc tools/hostsim/hostsim.cpp -o /tmp/hostsim
//   /tmp/hostsim [nt] [seed dispersions...]
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <vector>
#include <random>
#include <array>
#include "ascent_colloc.cuh"
#include "ascent_fly.cuh"
#include "ascent_plan.h"
#include "ascent_result.cuh"

using namespace lmato;

// Raw parameter column (include/lmato_b200.h) of the nominal problem with six of its values replaced.
static std::array<double, LMATO_NPARAM> make_params(double Ft, double M0, double Mdot, double addm, double rp, double ra) {
  std::array<double, LMATO_NPARAM> r;
  r[LMATO_P_G] = 6.674e-11; r[LMATO_P_M] = 7.346e22; r[LMATO_P_R0] = 1738100.0; r[LMATO_P_FT] = Ft; r[LMATO_P_M0] = M0;
  r[LMATO_P_M_DOT] = Mdot; r[LMATO_P_FUEL_MASS] = 2376.0; r[LMATO_P_ANGLE_DOUBLEDOT_MAX] = addm;
  r[LMATO_P_R_PERIAPSIS] = rp; r[LMATO_P_R_APOAPSIS] = ra; r[LMATO_P_FINAL_TIME] = 470.0;
  r[LMATO_P_MASS_SCALAR] = 2376.0; r[LMATO_P_ANGLE_UB] = M_PI / 3.0; r[LMATO_P_U_BOUND] = 1.0;
  return r;
}

// The options every entry point starts from: the library's solve_options on its defaults, with the solve running to
// exactly `tol` (no OTOL / RTOL) and MAX_ITER 500; each entry point then applies its own environment overrides.  Three
// departures from the library are kept on purpose, so that host results stay comparable with earlier ones:
//   - w_dcost is the raw move weight `wdc` (WDC), not obj_scale * dcost / objective_nodes;
//   - n_polish is the caller's (4 unless NPOL is set, 2 in hostsim_warm_batch), where the library's automatic value
//     is 2 with the move term and 4 without;
//   - theta_mu_warm is 2.0 with and without the move term (the library: 1.5 without).
static Options make_options(int nt, double tol, double obj_scale, double mu_min_factor, int n_polish, double wdc) {
  lmato_options o = default_options();
  o.tol = tol; o.otol = 0.0; o.rtol = 0.0; o.obj_scale = obj_scale; o.mu_min_factor = mu_min_factor; o.max_iter = 500;
  o.n_polish = n_polish;
  Options O = solve_options(o, nt, wdc > 0);
  O.w_dcost = wdc;
  O.theta_mu_warm = 2.0;
  return O;
}

// the model the CIRCULAR environment variable selects
static int model_from_env() { return getenv("CIRCULAR") ? LMATO_MODEL_CIRCULAR : LMATO_MODEL_ELLIPTICAL; }

// Start point of the next hostsim_solve / hostsim_solve_coop calls (B = 1, b = 0): a caller's start point
// (guess_traj [10][nt] in the output layout, guess_tf), the counterpart of lmato_set_initial_guess, and a reference
// column ([REF_ROWS][nt], as hostsim_reference writes it), the counterpart of the handle's warm-start reference.  Any
// of them may be NULL; with neither a guess nor a reference holding REF_OK the solve starts from the roll-out.
static const double* g_guess_traj = nullptr;
static const double* g_guess_tf = nullptr;
static const double* g_ref = nullptr;
extern "C" void hostsim_set_start(const double* guess_traj, const double* guess_tf, const double* ref) {
  g_guess_traj = guess_traj; g_guess_tf = guess_tf; g_ref = ref;
}

// One problem on the sweeps SW, started and restarted as the kernels do (ipm_start / ipm_restart), with the results
// written as the kernels write them (B = 1, b = 0).
template <class SW, class WS>
static void solve_one(const ResultOut& R, const Params& P, const Mesh& M, const Options& O, int model, const WS& W) {
  IpmState S;
  ipm_start<SW>(P, M, O, W, GuessSrc{g_guess_traj, g_guess_tf, 1, 0}, g_ref, S);
  do {
    while (!ipm_iterate_t<SW>(P, M, O, W, S)) {}
  } while (ipm_restart<SW>(P, M, O, W, S));
  write_results<SW, 1>(R, P, M, O.obj_scale, model, W, 0, 1u, S, 0);
}

int main(int argc, char** argv) {
  int nt = argc > 1 ? atoi(argv[1]) : 200;
  int nprob = argc > 2 ? atoi(argv[2]) : 1;
  int verbose = argc > 3 ? atoi(argv[3]) : 0;
  int only = argc > 4 ? atoi(argv[4]) : -1;
  const int N = nt - 1;
  std::vector<double> h(N + 1), tau(N + 1);
  for (int k = 0; k <= N; ++k) { tau[k] = (double)k / N; h[k] = k ? tau[k] - tau[k - 1] : 0.0; }
  Mesh M{N, h.data(), tau.data()};
  Options O = make_options(nt, 1e-10, 10.0, 1e-3, 4, getenv("WDC") ? atof(getenv("WDC")) : 0.0);
  if (getenv("MMF")) O.mu_min_factor = atof(getenv("MMF"));
  if (getenv("NPOL")) O.n_polish = atoi(getenv("NPOL"));
  if (getenv("THMU")) O.theta_mu = atof(getenv("THMU"));
  if (getenv("KMU")) O.kappa_mu = atof(getenv("KMU"));
  if (getenv("KEPS")) O.kappa_eps = atof(getenv("KEPS"));
  if (getenv("OBJ")) O.obj_scale = atof(getenv("OBJ"));
  if (getenv("MU0")) O.mu_init = atof(getenv("MU0"));
  if (getenv("TOL")) O.tol = atof(getenv("TOL"));
  if (getenv("TF0")) O.tf_guess = atof(getenv("TF0"));
  if (getenv("DC")) O.delta_c = atof(getenv("DC"));
  const int nfields = O.w_dcost > 0 ? (int)dc::N_FIELDS : (int)N_FIELDS;
  std::vector<double> ws((size_t)nfields * LANES * (N + 1), 0.0);   // one warp block, lane 0 used
  std::vector<double> tile(2 * TILE_ROWS, 0.0);
  Ws W{ws.data(), (long)nfields * LANES, tile.data()};
  std::vector<double> traj((size_t)LMATO_NVAR * nt);
  std::mt19937_64 rng(11);
  std::uniform_real_distribution<double> U(0.0, 1.0);
  int nfail = 0, itsum = 0, itmax = 0;
  for (int p = 0; p < nprob; ++p) {
    double u[6];
    for (int i = 0; i < 6; ++i) u[i] = (p == 0) ? 0.5 : U(rng);
    const double Ft = 15346.0 * (1 + 0.02 * (2 * u[0] - 1));
    const double Isp = 309.7 * (1 + 0.01 * (2 * u[1] - 1));
    const double Mdot = (p == 0) ? 5.053 : Ft / (Isp * 9.807);
    const double M0 = 4821.0 * (1 + 0.02 * (2 * u[2] - 1));
    const double addm = 5e-4 * std::pow(2.0, 2 * u[3] - 1);
    const double rp = 17703.0 * (1 + 0.10 * (2 * u[4] - 1));
    const double ra = 88615.0 * (1 + 0.10 * (2 * u[5] - 1));
    if (only >= 0 && p != only) continue;
    Params P = derive_params(make_params(Ft, M0, Mdot, addm, rp, ra).data(), 1, 0, LMATO_MODEL_ELLIPTICAL);
    std::fill(ws.begin(), ws.end(), 0.0);
    int status, iters;
    double tf, kkt, fmass;
    const ResultOut R{traj.data(), &tf, &fmass, &status, &iters, &kkt, nullptr, 1};
    if (O.w_dcost > 0) solve_one<Sweeps8>(R, P, M, O, LMATO_MODEL_ELLIPTICAL, W);
    else solve_one<Sweeps7>(R, P, M, O, LMATO_MODEL_ELLIPTICAL, W);
    itsum += iters; if (iters > itmax) itmax = iters;
    if (status != 0) ++nfail;
    if (verbose || nprob <= 20 || status != 0)
      printf("p %4d status %d iters %3d kkt %.2e tf %.10f tf_s %.8f  (Ft %.1f M0 %.1f Mdot %.4f addm %.2e rp %.0f ra %.0f)\n",
             p, status, iters, kkt, tf, tf * P.T, Ft, M0, Mdot, addm, rp, ra);
    if (p == 0 && nprob == 1) {
      printf("final y %.9f x %.9f vy %.9f vx %.9f\n", traj[LMATO_V_Y * nt + N] * P.S, traj[LMATO_V_X * nt + N] * P.S,
             traj[LMATO_V_YDOT * nt + N] * P.S, traj[LMATO_V_XDOT * nt + N] * P.S);
      printf("final mass %.9f\n", fmass);
    }
  }
  printf("solved %d problems: %d failures, mean iters %.1f, max %d\n", nprob, nfail, (double)itsum / nprob, itmax);
  return 0;
}

// d tf / d parameter (include/lmato_b200.h, lmato_sens_t: 4 values) of the next hostsim_solve / hostsim_solve_coop
// calls, or NULL: the counterpart of lmato_set_sensitivity_output.
static double* g_dtf = nullptr;
extern "C" void hostsim_set_sensitivity_output(double* dtf) { g_dtf = dtf; }

// d tf / d params[p] for every row p (LMATO_NPARAM values) of the next hostsim_solve / hostsim_solve_coop calls, or
// NULL: the counterpart of lmato_set_param_sensitivity_output.
static double* g_dtf_all = nullptr;
extern "C" void hostsim_set_param_sensitivity_output(double* dtf_all) { g_dtf_all = dtf_all; }

// ctypes entry for developer-side comparisons against tests/golden (NOT the product path).
extern "C" int hostsim_solve(const double* raw14, int nt, const double* time, double tol, double obj_scale,
                             double mu_min_factor, double* traj /* [10][nt] */, double* tf_out, int* iters, double* kkt) {
  const int N = nt - 1;
  std::vector<double> h(N + 1), tau(N + 1);
  for (int k = 0; k <= N; ++k) { tau[k] = time ? time[k] : (double)k / N; h[k] = k ? tau[k] - tau[k - 1] : 0.0; }
  Mesh M{N, h.data(), tau.data()};
  const Options O = make_options(nt, tol, obj_scale, mu_min_factor, getenv("NPOL") ? atoi(getenv("NPOL")) : 4,
                                 getenv("WDC") ? atof(getenv("WDC")) : 0.0);
  const int model = model_from_env();
  const Params P = derive_params(raw14, 1, 0, model);      // as the thread kernel: no circular move formulation
  const bool DC = O.w_dcost > 0;
  const int nfields = DC ? (int)dc::N_FIELDS : (int)N_FIELDS;
  std::vector<double> ws((size_t)nfields * LANES * (N + 1), 0.0);
  std::vector<double> tile(2 * TILE_ROWS, 0.0);
  Ws W{ws.data(), (long)nfields * LANES, tile.data()};
  int status;
  double fmass;
  const ResultOut R{traj, tf_out, &fmass, &status, iters, kkt, g_dtf, 1, g_dtf_all, raw14};
  if (DC) solve_one<Sweeps8>(R, P, M, O, model, W);
  else solve_one<Sweeps7>(R, P, M, O, model, W);
  return status;
}

// Finite-difference check of the hand-derived model derivatives (ascent_model.cuh) at one point:
// returns the largest relative error of accel_first's eight first derivatives and of the
// second-derivative contraction used by the Hessian (accel_second) against central differences.
extern "C" double hostsim_check_derivatives(const double* raw14, double y, double x, double a, double m) {
  const Params P = derive_params(raw14, 1, 0, LMATO_MODEL_ELLIPTICAL);
  Accel1 f;
  accel_first(P, y, x, a, m, f);
  const double v[4] = {y, x, a, m};
  const double an1[2][4] = {{f.ay_y, f.ay_x, f.ay_a, f.ay_m}, {f.ax_y, f.ax_x, f.ax_a, f.ax_m}};
  double worst = 0.0;
  Accel1 fp[4], fm[4];
  double hs[4];
  for (int j = 0; j < 4; ++j) {
    double p[4] = {v[0], v[1], v[2], v[3]}, q[4] = {v[0], v[1], v[2], v[3]};
    hs[j] = 1e-6 * std::fmax(1.0, std::fabs(v[j]));
    p[j] += hs[j]; q[j] -= hs[j];
    accel_first(P, p[0], p[1], p[2], p[3], fp[j]);
    accel_first(P, q[0], q[1], q[2], q[3], fm[j]);
    const double fd[2] = {(fp[j].ay - fm[j].ay) / (2 * hs[j]), (fp[j].ax - fm[j].ax) / (2 * hs[j])};
    for (int i = 0; i < 2; ++i)
      worst = std::fmax(worst, std::fabs(fd[i] - an1[i][j]) / std::fmax(1e-12, std::fabs(an1[i][j])));
  }
  // second derivatives: H = wy * d2 ay + wx * d2 ax over (y, x, a, m), against differences of the first ones
  const double wy = 0.7, wx = -1.3;
  Accel2 h2;
  accel_second(P, f, wy, wx, h2);
  const double an2[4][4] = {{h2.yy, h2.yx, h2.ya, h2.ym}, {h2.yx, h2.xx, h2.xa, h2.xm},
                            {h2.ya, h2.xa, h2.aa, h2.am}, {h2.ym, h2.xm, h2.am, h2.mm}};
  for (int j = 0; j < 4; ++j) {
    const double gp[4] = {wy * fp[j].ay_y + wx * fp[j].ax_y, wy * fp[j].ay_x + wx * fp[j].ax_x,
                          wy * fp[j].ay_a + wx * fp[j].ax_a, wy * fp[j].ay_m + wx * fp[j].ax_m};
    const double gm[4] = {wy * fm[j].ay_y + wx * fm[j].ax_y, wy * fm[j].ay_x + wx * fm[j].ax_x,
                          wy * fm[j].ay_a + wx * fm[j].ax_a, wy * fm[j].ay_m + wx * fm[j].ax_m};
    for (int i = 0; i < 4; ++i) {
      const double fd = (gp[i] - gm[i]) / (2 * hs[j]);
      double scale = 0.0;
      for (int a2 = 0; a2 < 4; ++a2) scale = std::fmax(scale, std::fabs(an2[i][a2]));
      worst = std::fmax(worst, std::fabs(fd - an2[i][j]) / std::fmax(1e-12, scale));
    }
  }
  return worst;
}

// The cooperative sweeps (csrc/ascent_coop.cuh) run by one lane (G = 1): same entry as hostsim_solve.
extern "C" int hostsim_solve_coop(const double* raw14, int nt, const double* time, double tol, double obj_scale,
                                  double mu_min_factor, double* traj /* [10][nt] */, double* tf_out, int* iters, double* kkt) {
  const int N = nt - 1;
  std::vector<double> h(N + 1), tau(N + 1);
  for (int k = 0; k <= N; ++k) { tau[k] = time ? time[k] : (double)k / N; h[k] = k ? tau[k] - tau[k - 1] : 0.0; }
  Mesh M{N, h.data(), tau.data()};
  const Options O = make_options(nt, tol, obj_scale, mu_min_factor, getenv("NPOL") ? atoi(getenv("NPOL")) : 4,
                                 getenv("WDC") ? atof(getenv("WDC")) : 0.0);
  const int model = model_from_env();
  const bool DC = O.w_dcost > 0;
  const Params P = derive_params(raw14, 1, 0, model, DC);   // the circular model with its move term: MV slot = pitch angle
  std::vector<double> ws((size_t)coop::coop_doubles_per_problem(nt), 0.0);
  std::vector<double> scr(coop::SCR_DOUBLES, 0.0);
  coop::Cws W{ws.data(), nt, scr.data(), 0, 1u, 1u, 0.0, 0.0, 0, 0u};
  int status;
  double fmass;
  const ResultOut R{traj, tf_out, &fmass, &status, iters, kkt, g_dtf, 1, g_dtf_all, raw14};
  const bool vrec = getenv("VREC") != nullptr;     // the variant that keeps W_k, g_k instead of running the adjoint recursion
  if (DC && model == LMATO_MODEL_CIRCULAR) solve_one<SweepsCoop<1, 1, 2, false>>(R, P, M, O, model, W);
  else if (DC && vrec) solve_one<SweepsCoop<1, 1, true, true>>(R, P, M, O, model, W);
  else if (DC)         solve_one<SweepsCoop<1, 1, true, false>>(R, P, M, O, model, W);
  else if (vrec)       solve_one<SweepsCoop<1, 1, false, true>>(R, P, M, O, model, W);
  else                 solve_one<SweepsCoop<1, 1, false, false>>(R, P, M, O, model, W);
  return status;
}

// Higher-order collocation (csrc/ascent_colloc.cuh), GP = 1, with the kernel's start ladder.  Ncol: row-major m x m,
// tauc: m points.  TF0 sets tf_guess.
extern "C" int hostsim_solve_colloc(const double* raw14, int nt, const double* time, int nodes, const double* Ncol,
                                    const double* tauc, double tol, double obj_scale, double mu_min_factor,
                                    double* traj /* [10][nt] */, double* tf_out, int* iters, double* kkt) {
  const int N = nt - 1, m = nodes - 1;
  std::vector<double> h(N + 1), tau(N + 1);
  for (int k = 0; k <= N; ++k) { tau[k] = time ? time[k] : (double)k / N; h[k] = k ? tau[k] - tau[k - 1] : 0.0; }
  Mesh M{N, h.data(), tau.data()};
  Options O = make_options(nt, tol, obj_scale, mu_min_factor, getenv("NPOL") ? atoi(getenv("NPOL")) : 4, 0.0);
  if (getenv("TF0")) O.tf_guess = atof(getenv("TF0"));
  const Params P = derive_params(raw14, 1, 0, LMATO_MODEL_ELLIPTICAL);   // NODES >= 3: the elliptical model only
  colloc::Coll C;
  C.m = m;
  for (int i = 0; i < m; ++i) { C.tau[i] = tauc[i]; for (int j = 0; j < m; ++j) C.N[i][j] = Ncol[i * m + j]; }
  std::vector<double> ws((size_t)colloc::colloc_doubles_per_problem(nt, m), 0.0);
  colloc::Nws W;
  W.base = ws.data(); W.N1 = nt; W.L.init(m); W.C = &C; W.g = 0; W.mask = 1u; W.dw = 0.0; W.pimax = 0.0; W.ls_flag = 0;
  int status;
  double fmass;
  const ResultOut R{traj, tf_out, &fmass, &status, iters, kkt, nullptr, 1};
  solve_one<SweepsColloc<1>>(R, P, M, O, LMATO_MODEL_ELLIPTICAL, W);
  return status;
}

// The reference solve of the batch warm start (lmato_solve_batch's ref_mode 1 launch) for the problem raw14 on a
// uniform mesh of nt nodes: the cooperative sweeps without the move term, solved down to mu_ref (tol = 10 mu_ref,
// mu_min_factor 0.1, no polish), started from the reference already in ref_out if it holds one, then stored there
// ([REF_ROWS][nt]).  Returns the solve's status.
extern "C" int hostsim_reference(const double* raw14, int nt, double mu_ref, double* ref_out) {
  const int N = nt - 1;
  std::vector<double> h(N + 1), tau(N + 1);
  for (int k = 0; k <= N; ++k) { tau[k] = (double)k / N; h[k] = k ? tau[k] - tau[k - 1] : 0.0; }
  Mesh M{N, h.data(), tau.data()};
  Options O = reference_options(make_options(nt, 1e-10, 10.0, 1e-3, 4, 0.0), mu_ref);
  if (getenv("KEPS")) O.kappa_eps = atof(getenv("KEPS"));
  if (getenv("KMU")) O.kappa_mu = atof(getenv("KMU"));
  const Params P = derive_params(raw14, 1, 0, model_from_env());
  std::vector<double> ws((size_t)coop::coop_doubles_per_problem(nt), 0.0), scr(coop::SCR_DOUBLES, 0.0);
  coop::Cws W{ws.data(), nt, scr.data(), 0, 1u, 1u, 0.0, 0.0, 0, 0u};
  using SW = SweepsCoop<1, 1, false, false>;
  IpmState S;
  ipm_start<SW>(P, M, O, W, GuessSrc{nullptr, nullptr, 1, 0}, ref_out, S);
  do {
    while (!ipm_iterate_t<SW>(P, M, O, W, S)) {}
  } while (ipm_restart<SW>(P, M, O, W, S));
  SW::store_ref(P, M, W, S.src, S.cur, S.ctl.mu, S.ctl.status == ST_CONVERGED, ref_out);
  return S.ctl.status;
}

// Batch warm start on the host (what lmato_solve_batch does on the device): the batch-mean problem is solved to
// mu_ref by hostsim_reference, and every dispersed problem then starts from that reference on the cooperative sweeps
// (with the move term if wdc > 0).  It leaves no start point set (hostsim_set_start).  Returns the mean iteration
// count; used to study barrier-update strategies on the CPU.
//   hostsim_warm_batch(nprob, nt, wdc, mu_ref, out_iters[nprob], out_status[nprob], out_tf[nprob])
extern "C" double hostsim_warm_batch(int nprob, int nt, double wdc, double mu_ref, int* out_iters, int* out_status, double* out_tf) {
  const int N = nt - 1;
  std::vector<double> h(N + 1), tau(N + 1);
  for (int k = 0; k <= N; ++k) { tau[k] = (double)k / N; h[k] = k ? tau[k] - tau[k - 1] : 0.0; }
  Mesh M{N, h.data(), tau.data()};
  Options O = make_options(nt, 1e-10, 10.0, 1e-3, 2, wdc);
  if (getenv("THMUW")) O.theta_mu_warm = atof(getenv("THMUW"));
  if (getenv("KEPS")) O.kappa_eps = atof(getenv("KEPS"));
  if (getenv("KMU")) O.kappa_mu = atof(getenv("KMU"));
  if (getenv("NPOL")) O.n_polish = atoi(getenv("NPOL"));
  if (getenv("MMF")) O.mu_min_factor = atof(getenv("MMF"));
  std::mt19937_64 rng(11);
  std::uniform_real_distribution<double> U(0.0, 1.0);
  std::vector<Params> Ps;
  double mean[6] = {0, 0, 0, 0, 0, 0};
  for (int p = 0; p < nprob; ++p) {
    double u[6];
    for (int i = 0; i < 6; ++i) u[i] = (p == 0) ? 0.5 : U(rng);
    const double Ft = 15346.0 * (1 + 0.02 * (2 * u[0] - 1));
    const double Isp = 309.7 * (1 + 0.01 * (2 * u[1] - 1));
    const double Mdot = (p == 0) ? 5.053 : Ft / (Isp * 9.807);
    const double M0 = 4821.0 * (1 + 0.02 * (2 * u[2] - 1));
    const double addm = 5e-4 * std::pow(2.0, 2 * u[3] - 1);
    const double rp = 17703.0 * (1 + 0.10 * (2 * u[4] - 1));
    const double ra = 88615.0 * (1 + 0.10 * (2 * u[5] - 1));
    Ps.push_back(derive_params(make_params(Ft, M0, Mdot, addm, rp, ra).data(), 1, 0, LMATO_MODEL_ELLIPTICAL));
    const double v[6] = {Ft, M0, Mdot, addm, rp, ra};
    for (int i = 0; i < 6; ++i) mean[i] += v[i] / nprob;
  }
  std::vector<double> ref((size_t)dc::REF_ROWS * nt, 0.0);
  hostsim_reference(make_params(mean[0], mean[1], mean[2], mean[3], mean[4], mean[5]).data(), nt, mu_ref, ref.data());
  std::vector<double> ws((size_t)coop::coop_doubles_per_problem(nt), 0.0), scr(coop::SCR_DOUBLES, 0.0);
  coop::Cws W{ws.data(), nt, scr.data(), 0, 1u, 1u, 0.0, 0.0, 0, 0u};
  hostsim_set_start(nullptr, nullptr, ref.data());
  double itsum = 0, fmass;
  for (int p = 0; p < nprob; ++p) {
    const ResultOut R{nullptr, out_tf + p, &fmass, out_status + p, out_iters + p, nullptr, nullptr, 1};
    if (wdc > 0) solve_one<SweepsCoop<1, 1, true, false>>(R, Ps[p], M, O, LMATO_MODEL_ELLIPTICAL, W);
    else solve_one<SweepsCoop<1, 1, false, false>>(R, Ps[p], M, O, LMATO_MODEL_ELLIPTICAL, W);
    itsum += out_iters[p];
  }
  hostsim_set_start(nullptr, nullptr, nullptr);
  return itsum / nprob;
}

// plan_solve (csrc/ascent_plan.h) for a handle with the default options but for kernel, coop_lanes, dcost and
// warm_start: out = {kind, lanes, ctas_per_sm, move, grid, slots, ws_bytes, alloc_bytes, warm, use_dc}.
extern "C" void hostsim_plan(int sm_count, int nt, int nodes, int model, int kernel, int coop_lanes, double dcost,
                             int warm_start, int64_t B, int has_guess, int64_t warm_batch, int64_t* out) {
  lmato_options o = default_options();
  o.kernel = kernel; o.coop_lanes = coop_lanes; o.dcost = dcost; o.warm_start = warm_start;
  const LaunchPlan p = plan_solve(sm_count, nt, nodes, model, o, B, has_guess != 0, warm_batch);
  const int64_t v[10] = {p.kernel.kind, p.kernel.lanes, p.kernel.ctas_per_sm, p.kernel.move, p.grid, p.slots,
                         (int64_t)p.ws_bytes, (int64_t)p.alloc_bytes, p.warm, p.use_dc};
  for (int i = 0; i < 10; ++i) out[i] = v[i];
}

// The post-solve flight (csrc/ascent_fly.cuh) of one problem, as fly_control_kernel runs it: raw14 the parameter
// column, model lmato_model_t, time the mesh (NULL = uniform), traj [10][nt] a solve's output, fin [LMATO_NFLY], out
// [10][nt] or NULL.
extern "C" void hostsim_fly(const double* raw14, int model, int nt, const double* time, const double* traj, double tf,
                            int substeps, double* fin, double* out) {
  std::vector<double> tau(nt);
  for (int k = 0; k < nt; ++k) tau[k] = time ? time[k] : (double)k / (nt - 1);
  const Params P = derive_params(raw14, 1, 0, model);
  fly_one(P, model, tau.data(), nt, traj, tf, substeps, 1, 0, fin, out);
}
