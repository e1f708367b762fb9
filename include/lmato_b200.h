/* lmato_b200.h -- C ABI of the B200-native batched lunar-ascent trajectory optimiser.
 *
 * Drop-in boundary for ONE hot path of the reference: the GEKKO/IPOPT solve
 *     m.solve(disp=True)                      /root/reference/Launch_Optimiser.py:177
 * together with the model declaration that feeds it (LO:19-176) and the `.value`
 * read-back that follows it (LO:178-202).  The reference has no FFI of its own (the
 * boundary there is a Python object API over a process boundary to the `apm`
 * executable); INTEGRATION.md shows the ctypes binding a maintainer of the reference
 * would add.  Everything here is plain C: pointers, sizes, ints.  No exceptions cross
 * this boundary; every function returns an lmato_status_t and lmato_last_error() gives
 * the text of the last failure on the calling thread.
 *
 * Beyond the reference's solve there are post-solve checks: lmato_coast_orbit (the PDF's orbit coast) and
 * lmato_fly_control, which flies each solved control through the continuous dynamics and reports how far the vehicle
 * really ends up from the target orbit (the transcription error of the solve).
 *
 * Threading: a handle is bound to one CUDA device and must be used from one host thread
 * at a time.  Solves on one handle share its workspace: they are serialised on the device even when
 * issued on different streams (a solve on a new stream waits for the handle's previous solve).
 * Distinct handles are independent.  Ownership: the caller owns every
 * input/output buffer; the library owns only the workspace inside the handle.
 */
#ifndef LMATO_B200_H
#define LMATO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct lmato_handle lmato_handle;

typedef enum {
  LMATO_OK = 0,
  LMATO_ERR_INVALID = 1,     /* bad argument */
  LMATO_ERR_CUDA = 2,        /* CUDA runtime failure (text in lmato_last_error) */
  LMATO_ERR_NO_DEVICE = 3,   /* no usable CUDA device: there is NO CPU fallback */
  LMATO_ERR_UNSUPPORTED = 4  /* model / NODES combination not implemented */
} lmato_status_t;

/* Model variants.  ELLIPTICAL = Launch_Optimiser.py as shipped (LO:83-173);
 * CIRCULAR = the "original IB-document" model (reference PDF p.26-28). */
typedef enum { LMATO_MODEL_ELLIPTICAL = 0, LMATO_MODEL_CIRCULAR = 1 } lmato_model_t;

/* Per-problem parameter rows of the `params` array, shape [LMATO_NPARAM][B], row-major
 * (struct of arrays: row p, problem b at params[p*B + b]).  Names and defaults are the
 * reference's literals. */
enum {
  LMATO_P_G = 0,                 /* LO:50  6.674e-11 */
  LMATO_P_M = 1,                 /* LO:51  7.346e22  */
  LMATO_P_R0 = 2,                /* LO:52  1738100   */
  LMATO_P_FT = 3,                /* LO:61  15346     */
  LMATO_P_M0 = 4,                /* LO:62  4821      */
  LMATO_P_M_DOT = 5,             /* LO:63/65  5.053  */
  LMATO_P_FUEL_MASS = 6,         /* LO:64  2376      */
  LMATO_P_ANGLE_DOUBLEDOT_MAX = 7,  /* LO:66  5e-4   */
  LMATO_P_R_PERIAPSIS = 8,       /* LO:70  17703     */
  LMATO_P_R_APOAPSIS = 9,        /* LO:71  88615     */
  LMATO_P_FINAL_TIME = 10,       /* LO:38  470       */
  LMATO_P_MASS_SCALAR = 11,      /* LO:108 = fuel_mass (2576 in the PDF original) */
  LMATO_P_ANGLE_UB = 12,         /* LO:94  pi/3      */
  LMATO_P_U_BOUND = 13,          /* LO:96  1         */
  LMATO_NPARAM = 14
};

/* Rows of the output trajectory, shape [LMATO_NVAR][nt][B]; GEKKO declaration order
 * (LO:83-96).  Scaled units, exactly as the reference's `.value` lists (LO:188-202);
 * node 0 holds the pinned initial values (all zero). */
enum {
  LMATO_V_Y = 0, LMATO_V_YDOT = 1, LMATO_V_YDOUBLEDOT = 2,
  LMATO_V_X = 3, LMATO_V_XDOT = 4, LMATO_V_XDOUBLEDOT = 5,
  LMATO_V_ANGLE = 6, LMATO_V_ANGLEDOT = 7, LMATO_V_MASS = 8,
  LMATO_V_ANGLEDOUBLEDOT = 9,
  LMATO_NVAR = 10
};

/* Per-problem solve status (not an error of the call). */
enum {
  LMATO_ST_CONVERGED = 0,        /* scaled KKT error <= tol */
  LMATO_ST_MAX_ITER = 1,         /* MAX_ITER reached (LO:28) */
  LMATO_ST_LINESEARCH_FAIL = 2,  /* filter line search could not make progress: no acceptable step within max_ls
                                    halvings, or a third search of the solve that was still rejected after 12 (the
                                    first two are taken as null steps); IPOPT would enter its restoration phase */
  LMATO_ST_INERTIA_FAIL = 3,     /* KKT inertia could not be corrected */
  LMATO_ST_NUMERICAL = 4,        /* NaN/Inf encountered */
  LMATO_ST_STALLED = 5           /* no progress: ten consecutive steps shorter than 1e-6, or no improvement of the KKT
                                    error for 100 iterations (what IPOPT's restoration phase reports as infeasible) */
};

typedef struct {
  double tol;        /* scaled KKT tolerance (IPOPT `tol`); default 1e-10 (see DESIGN.md "Tolerance") */
  double mu_init;    /* initial barrier parameter; default 0.1 */
  double obj_scale;  /* objective = obj_scale * tf; default 10 */
  double tf_guess;   /* initial scaled final time; default 0.9 */
  double delta_c;    /* dual regularisation of the terminal equality row; default 1e-8 */
  double mu_min_factor; /* barrier floor = mu_min_factor * tol; default 1e-3 (IPOPT uses 0.1) */
  int32_t max_iter;  /* LO:28 MAX_ITER; default 20000 (the reference's value) */
  int32_t max_ls;    /* max backtracking steps per iteration; default 40 */
  int32_t n_polish;  /* Newton iterations taken after tol is first met; default -1 = automatic: 2 with the
                        DCOST term (it regularises the flat control directions), 4 without (DESIGN.md "Tolerance") */
  int32_t warm_start; /* 1 (default): batches of >= 512 problems (below that the serial reference solve costs more than it saves) first solve the batch-mean problem down to
                         mu_ref and start every problem from that central-path point; a problem that fails
                         from there is restarted from the generic cold start.  0: always cold start.  2: warm start for
                         every batch size.  The handle keeps its last reference and the next reference solve
                         starts from it. */
  double mu_ref;     /* barrier parameter at which the reference solve stops; default 1e-3 */
  double dcost;      /* LO:99 angledoubledot.DCOST: l1 move suppression dcost*sum|MV_k - MV_{k-1}|; default
                        1e-5 (the reference's value); 0 switches the term off (7-state fast path).  For
                        LMATO_MODEL_CIRCULAR the MV is the pitch angle (PDF p.27 src 69-73, DCOST = 1e-5 there too);
                        that model with the term runs on the cooperative kernel at every batch size */
  double kappa_eps;  /* barrier sub-problem tolerance factor (IPOPT barrier_tol_factor, default there 10): mu is
                        reduced once E_mu <= kappa_eps*mu; default 30 (2.4 fewer iterations, same answers) */
  int32_t objective_nodes; /* APMonitor sums the objective over the horizon: minimise objective_nodes*tf +
                        dcost*sum|dMV|; 0 (default) = nt-1.  Only the ratio dcost/objective_nodes matters. */
  int32_t kernel;    /* lmato_kernel_t: which kernel solves a batch; default LMATO_KERNEL_AUTO (by batch size) */
  int32_t coop_lanes; /* COOP kernel: lanes per problem in the stage-parallel phases, 8 or 32; 0 (default) = by batch size */
  int32_t reserved_;
  double otol;       /* LO:31 m.options.OTOL and */
  double rtol;       /* LO:32 m.options.RTOL (the reference sets both to 1e-3, the defaults here).  How APMonitor
                        maps them onto IPOPT's `tol` cannot be verified without GEKKO; the rule here is the
                        conservative one: a solve runs to min(tol, otol, rtol), so the reference's 1e-3 never
                        loosens the default 1e-10 and a tighter OTOL/RTOL tightens it.  0 = ignore. */
} lmato_options;

/* Kernel mapping (both solve the same NLP with the same IPM and agree to rounding; DESIGN.md section 3):
 *   THREAD  one problem per thread, one coalesced workspace row per warp and stage: least HBM traffic per
 *           problem, needs ~37 888 problems in flight to fill a B200;
 *   COOP    eight lanes of a warp per problem, stage-parallel model evaluation, cost-to-go distributed by rows:
 *           short critical path per problem, fills the GPU with ~4 700 problems;
 *   AUTO    COOP up to 6 144 problems per call, THREAD above; the circular model with its move term (dcost > 0) always
 *           runs on COOP.  COOP takes 32 lanes per problem up to 8 problems per SM and 8 lanes above that, and
 *           two CTAs per SM once one CTA per SM cannot hold the whole batch. */
typedef enum { LMATO_KERNEL_AUTO = 0, LMATO_KERNEL_THREAD = 1, LMATO_KERNEL_COOP = 2 } lmato_kernel_t;

/* Fill `o` with the defaults above. */
void lmato_default_options(lmato_options* o);

/* Create a solver for one device and one mesh.
 *   device  CUDA ordinal
 *   nt      number of mesh nodes (LO:20, 200)
 *   time    host pointer to nt normalised times in [0,1], strictly increasing, time[0]=0
 *           (LO:21); NULL = linspace(0,1,nt)
 *   nodes   collocation NODES (LO:25), 2..6.  2 (the reference's value, backward Euler) runs on the two tuned
 *           kernels; 3..6 (Lobatto collocation with NODES-1 points per step, MV held over the step) run on the
 *           general collocation kernel: elliptical model, no DCOST term, no warm start / guess / sensitivities
 *   model   lmato_model_t
 * Replaces: GEKKO() + m.time + m.options.* (LO:19-33). */
lmato_status_t lmato_create(lmato_handle** out, int32_t device, int32_t nt, const double* time,
                            int32_t nodes, int32_t model);
lmato_status_t lmato_destroy(lmato_handle* h);
lmato_status_t lmato_set_options(lmato_handle* h, const lmato_options* o);

/* Solve B independent ascent problems.  All pointers are DEVICE pointers on the handle's
 * device; `stream` is a cudaStream_t (NULL = default stream).  Asynchronous with respect
 * to the host: results are valid after the stream is synchronised.
 *   params        [LMATO_NPARAM][B]
 *   out_traj      [LMATO_NVAR][nt][B] or NULL
 *   out_tf        [B]   scaled final time in (0,1)  (tf.value[0], LO:178)
 *   out_final_mass[B]   kg:  M0 - fuel_mass * mass(nt-1)
 *   out_status    [B]   LMATO_ST_*
 *   out_iters     [B]   IPM iterations used, including those of an abandoned warm start / caller's start point
 *   out_kkt       [B]   final scaled KKT error, or NULL
 * Replaces: m.solve() (LO:177) and the read-back LO:178-202. */
lmato_status_t lmato_solve_batch(lmato_handle* h, const double* params, int64_t B,
                                 double* out_traj, double* out_tf, double* out_final_mass,
                                 int32_t* out_status, int32_t* out_iters, double* out_kkt,
                                 void* stream);

/* Same with HOST buffers: copies params to the device, solves, copies results back and
 * synchronises.  This is the end-to-end call the Python API makes for host tensors. */
lmato_status_t lmato_solve_batch_host(lmato_handle* h, const double* params, int64_t B,
                                      double* out_traj, double* out_tf, double* out_final_mass,
                                      int32_t* out_status, int32_t* out_iters, double* out_kkt);

/* Device list (SURVEY 8b/8e): one host process, several GPUs.  The batch is index-partitioned (problem i ->
 * devices[floor(i*ndev/B)], contiguous ranges whose sizes differ by at most one), every device solves its
 * shard concurrently with its own handle, and each writes its slice of the caller's HOST result arrays
 * (same shapes as lmato_solve_batch_host; pinned host memory makes the copies asynchronous).  The problems
 * are independent and the results land on the host, so no collective is involved; the one-process-per-GPU
 * path (torchrun) with its single NCCL allgather lives in the Python host layer (`sharded_solve`).
 * A device may be named more than once (each entry gets its own handle and workspace). */
typedef struct lmato_multi lmato_multi;
lmato_status_t lmato_multi_create(lmato_multi** out, const int32_t* devices, int32_t ndev, int32_t nt,
                                  const double* time, int32_t nodes, int32_t model);
lmato_status_t lmato_multi_destroy(lmato_multi* m);
lmato_status_t lmato_multi_set_options(lmato_multi* m, const lmato_options* o);
lmato_status_t lmato_multi_device_count(lmato_multi* m, int32_t* n);
lmato_status_t lmato_multi_solve_host(lmato_multi* m, const double* params, int64_t B,
                                      double* out_traj, double* out_tf, double* out_final_mass,
                                      int32_t* out_status, int32_t* out_iters, double* out_kkt);

/* Start point for the following solves on this handle (SURVEY 8f.4: accept a previous solution as the guess;
 * the reference's counterpart is the `value=` argument of m.Var / m.MV / m.FV, LO:39, 83-96):
 *   guess_traj [LMATO_NVAR][nt][B]  in the layout of out_traj (the rows of ydoubledot, xdoubledot and mass are
 *                                   ignored: the device formulation eliminates them),  guess_tf [B].
 * The primal values are taken as given and pushed into the interior of their bounds; node 0 stays pinned.
 * DEVICE pointers for lmato_solve_batch, HOST pointers for lmato_solve_batch_host; NULL, NULL (the default)
 * returns to the built-in start (roll-out / batch warm start).  The buffers must stay valid until the
 * solve that uses them has finished. */
lmato_status_t lmato_set_initial_guess(lmato_handle* h, const double* guess_traj, const double* guess_tf);

/* Parametric sensitivities of the optimal final time (SURVEY 8f.4; no counterpart in the reference).
 * Registers an extra output for the following solves on this handle: out_dtf [LMATO_NSENS][B] = d tf / d parameter
 * (tf in the reference's scaled units, parameter in the units of the params block) for the parameters of
 * lmato_sens_t, from the multipliers at the solution (envelope theorem; costs one pass over the converged
 * iterate).  A DEVICE pointer for lmato_solve_batch, a HOST pointer for lmato_solve_batch_host; NULL (the
 * default) switches the output off.  Entries of problems that did not converge are meaningless.  For
 * LMATO_MODEL_CIRCULAR the LMATO_S_ANGLE_DOUBLEDOT_MAX entry is NaN: that model has no pitch-acceleration limit
 * (its MV is the pitch angle itself, PDF p.27), so tf does not depend on that row of the params block; the other
 * three entries are computed as for the elliptical model. */
#define LMATO_NSENS 4
typedef enum lmato_sens {
  LMATO_S_FT = 0,                   /* thrust Ft (LO:61) */
  LMATO_S_M0 = 1,                   /* wet mass M0 (LO:62) */
  LMATO_S_M_DOT = 2,                /* propellant flow M_dot (LO:63) */
  LMATO_S_ANGLE_DOUBLEDOT_MAX = 3   /* pitch acceleration limit (LO:66) */
} lmato_sens_t;
lmato_status_t lmato_set_sensitivity_output(lmato_handle* h, double* out_dtf);

/* d tf / d params[p] for every row p of the params block:  out_dtf_dp [LMATO_NPARAM][B], row p = LMATO_P_*.
 * Registered, switched off (NULL), addressed and checked like lmato_set_sensitivity_output (a DEVICE
 * pointer for lmato_solve_batch, a HOST pointer for lmato_solve_batch_host; entries of problems that did not
 * converge are meaningless), and independent of it: either output, both or neither may be registered, and
 * registering this one changes no bit of any other output.  Its rows Ft, M0, M_dot and angle_doubledot_max are the
 * values of lmato_set_sensitivity_output, bit for bit.  Each entry is the partial derivative with respect to that
 * one row, the other rows held: tf in the reference's scaled units (0..1) per unit of the raw row, from the same
 * envelope-theorem pass over the converged iterate, i.e. the derivative of the whole objective (with the move term
 * when DCOST > 0) divided by obj_scale.  r_periapsis is both the target perilune and the distance scale of the
 * scaled dynamics; its row covers both roles.  For LMATO_MODEL_CIRCULAR the rows angle_doubledot_max and u_bound
 * are NaN: that model reads neither.  NODES >= 3: the solve answers LMATO_ERR_UNSUPPORTED while it is registered. */
lmato_status_t lmato_set_param_sensitivity_output(lmato_handle* h, double* out_dtf_dp);

/* The collocation rule used for NODES = 2..6 (host only, no GPU needed): tau[NODES-1] = the non-initial Lobatto
 * points on (0,1], N[(NODES-1)^2] row-major with  h N f_{1..} = z_{1..} - z_0  (SURVEY Appendix B.2). */
lmato_status_t lmato_collocation_rule(int32_t nodes, double* tau, double* N);

/* Introspection (for benchmarks and tests). */
lmato_status_t lmato_workspace_bytes(lmato_handle* h, int64_t B, int64_t* bytes);
lmato_status_t lmato_kernel_launches(lmato_handle* h, int64_t* n);  /* launches so far */
/* Device time of the last lmato_solve_batch IPM kernel in milliseconds (CUDA events on
 * the launching stream); synchronises that stream. */
lmato_status_t lmato_last_kernel_ms(lmato_handle* h, double* ms);
/* Measured FP64 FMA peak of the handle's device in GFLOP/s (dependent-chain-free DFMA
 * micro-benchmark; used as the roofline denominator, MEASURED_PEAKS.json has no FP64). */
lmato_status_t lmato_measure_fp64_peak(lmato_handle* h, double* gflops);

/* Post-solve orbit check (reference PDF p.28-29 src 185-237): coast each state around the Moon with the PDF's
 * explicit Euler scheme (a from the current position; position += old velocity*dt; velocity += a*dt).
 *   state [4][B]  x, y, vx, vy   SI, Moon-centred (device pointer)
 *   gm            Gs*m_2 (PDF src 186-188: 6.67e-11 * 7.346e22), dt (PDF: 0.001), nsteps (PDF: 6600/dt)
 *   out   [6][B]  r_min, r_max over the coast, then the final x, y, vx, vy (device pointer)
 * Asynchronous on `stream`. */
lmato_status_t lmato_coast_orbit(lmato_handle* h, const double* state, int64_t B, double gm, double dt,
                                 int64_t nsteps, double* out, void* stream);

/* Post-solve flight check (no counterpart in the reference): fly each solved control through the continuous ascent
 * dynamics (LO:114-136) and report where the vehicle really ends up.  A solve returns the optimum of the transcribed
 * problem (backward Euler for NODES = 2); flown, the NODES = 2 plan of the reference script (nt = 200) misses the
 * target radius by about 2 km and the target speed by about 10 m/s (DESIGN.md section 7).  Classical RK4 in
 * normalised time with `substeps` equal sub-steps per mesh step, the MV of node k held on (t_{k-1}, t_k] (MV_TYPE = 0,
 * LO:29, as both transcriptions hold it), from the pinned zeros of node 0 (LO:145-151).  The flight does not depend on
 * the handle's NODES; it uses the handle's mesh and model.  One thread per problem.
 *   params     [LMATO_NPARAM][B]
 *   traj       [LMATO_NVAR][nt][B]   a solve's out_traj; only the MV row is read (angledoubledot, or angle for
 *                                    LMATO_MODEL_CIRCULAR, PDF p.27)
 *   tf         [B]   the solved scaled final time
 *   out_final  [LMATO_NFLY][B]
 *   out_traj   [LMATO_NVAR][nt][B] or NULL: the flown states in the layout of a solve (node 0 zero, the acceleration
 *              rows evaluated at the flown nodes, the MV row copied from traj, rows the model lacks zero)
 * DEVICE pointers, asynchronous on `stream`.  The call neither uses nor waits for the handle's solve workspace: stream
 * order is the only ordering it needs with respect to solves.  Problems that did not converge are flown as given.
 * LMATO_ERR_INVALID for a NULL handle or buffer, B < 0 or substeps < 1; B = 0 does nothing. */
#define LMATO_NFLY 10   /* rows: y, ydot, x, xdot, angle, angledot, mass at tf (scaled, like out_traj),
                           radius miss [m], speed miss [m/s], flight-path angle [rad] */
lmato_status_t lmato_fly_control(lmato_handle* h, const double* params, int64_t B, const double* traj,
                                 const double* tf, int32_t substeps, double* out_final /* [LMATO_NFLY][B] */,
                                 double* out_traj /* [LMATO_NVAR][nt][B] or NULL */, void* stream);

/* Device self-test of the solver's branch-free FP64 math (rcp, rsqrt, log, sin, cos) against the
 * CUDA math library: max_err5 = {rel rcp, rel rsqrt, rel log, abs sin, abs cos}. */
lmato_status_t lmato_selftest_math(lmato_handle* h, double* max_err5);

const char* lmato_last_error(void);
const char* lmato_version(void);

#ifdef __cplusplus
}
#endif
#endif /* LMATO_B200_H */
