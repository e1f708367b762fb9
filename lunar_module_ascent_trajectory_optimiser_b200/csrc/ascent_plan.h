// Launch plan of one solve: which kernel a batch gets, its grid and workspace, the batch warm start, and the solver
// options the kernels receive.  Host code only, without the CUDA runtime: the library (ascent_cabi.cu) and the host
// simulator (tools/hostsim) compile the same rules.
#pragma once
#include <stddef.h>
#include <stdint.h>

#include "ascent_colloc.cuh"

namespace lmato {

// Thread kernel: one CTA of 256 threads (8 warps) per SM; 255 registers x 256 threads fills the register file.
constexpr int kBlock = 256;
constexpr int kBlocksPerSM = 1;
// Cooperative and collocation kernels: CTAs of 256 threads, G = 8 lanes in the sequential phases, and at most two
// CTAs per SM (128 registers per thread).
constexpr int kCoopBlock = 256;
constexpr int kCoopBlocksPerSM = 2;
constexpr int kCoopG = 8;
// Which kernel solves a batch of B problems.  One thread per problem needs ~1 wave (SMs x 256 problems) to fill
// the GPU and streams the least HBM traffic per problem; eight lanes per problem fill it with an eighth of that
// and shorten the critical path of every problem, at ~2.5x the traffic.  Measured cross-over on B200 at nt = 200:
// between 16 384 and 32 768 problems (profiles/README.md).
constexpr int64_t kCoopMaxBatch = 6144;
// Batch warm start: one reference solve of the batch-mean problem (cooperative kernel, one group) against ~6 saved
// iterations per problem.  Measured with the reference solve on the cooperative kernel (1.8 ms on the first call of a
// handle, 0.2 ms afterwards): 512 problems 7.2 ms cold, 7.3 ms warm on the first call, 5.5 ms on later calls; from
// 1 024 problems up the first call wins as well (tools/gpu_warm_threshold.py).
constexpr int64_t kWarmStartMinBatch = 512;

// The defaults of lmato_options (include/lmato_b200.h).
inline lmato_options default_options() {
  lmato_options o{};
  o.tol = 1e-10;
  o.mu_init = 0.1;
  o.obj_scale = 10.0;
  o.tf_guess = 0.9;
  o.delta_c = 1e-8;
  o.mu_min_factor = 1e-3;
  o.n_polish = -1;           // automatic: 2 with the DCOST term, 4 without (DESIGN.md "Tolerance")
  o.warm_start = 1;
  o.mu_ref = 1e-3;
  o.dcost = 1e-5;            // LO:99
  o.kappa_eps = 30.0;
  o.objective_nodes = 0;     // 0 = nt - 1
  o.kernel = LMATO_KERNEL_AUTO;
  o.coop_lanes = 0;
  o.otol = 1e-3;             // LO:31
  o.rtol = 1e-3;             // LO:32
  o.max_iter = 20000;        // LO:28
  o.max_ls = 40;
  return o;
}

enum KernelKind : int { kThreadKernel, kCoopKernel, kCollocKernel };

// One solve-kernel instantiation (the table in ascent_cabi.cu): its kind, lanes per problem (GP), CTAs per SM (BPS) and
// move term (0 none, 1 the move term of LO:99, 2 the circular model's, MV = angle).  The thread kernel has one lane,
// and move 1 selects its 8-state sweeps.
struct KernelKey {
  int kind, lanes, ctas_per_sm, move;
  bool operator==(const KernelKey& o) const {
    return kind == o.kind && lanes == o.lanes && ctas_per_sm == o.ctas_per_sm && move == o.move;
  }
};

struct LaunchPlan {
  KernelKey kernel;
  long grid;              // CTAs
  long slots;             // the thread kernel's problem slots (its grid x kBlock), passed to every kernel
  size_t ws_bytes;        // the kernel's workspace: what lmato_workspace_bytes reports
  size_t alloc_bytes;     // the workspace to allocate: also holds the warm start's reference solve
  bool warm;              // solve the batch-mean reference first and start every problem from it
  bool use_dc;            // the move-suppression term is in the objective
};

// CTAs for B problems in chunks of 32 / lanes per warp: one per chunk, at least one, at most cap.
inline long grid_for(int64_t B, int lanes, long cap) {
  const long per_chunk = 32 / lanes;
  const long chunks = (B + per_chunk - 1) / per_chunk;
  return chunks < cap ? (chunks > 0 ? chunks : 1) : cap;
}

// Workspace of a cooperative or collocation launch: one block of `per_problem` doubles per group.
inline size_t group_ws_bytes(long per_problem, long grid, int lanes) {
  return sizeof(double) * (size_t)per_problem * (size_t)(grid * (kCoopBlock / lanes));
}

// The launch of a batch of B problems on a device with sm_count SMs.  warm_batch is the size of the batch the B
// problems belong to (B itself, or the whole batch when they are one device's shard of it): the shards of one batch
// keep the batch warm start even when a shard alone is small.
inline LaunchPlan plan_solve(int sm_count, int nt, int nodes, int model, const lmato_options& o, int64_t B,
                             bool has_guess, int64_t warm_batch) {
  const bool hi_order = nodes > 2;            // NODES >= 3: the general collocation kernel
  // The move-suppression term: DCOST on the MV angledoubledot of the elliptical model (LO:99), on the MV angle of the
  // circular model (PDF p.27 src 69-73).  The circular model with the term is carried by the cooperative kernel only.
  const bool circular_move = model == LMATO_MODEL_CIRCULAR && o.dcost > 0.0;
  LaunchPlan p;
  p.use_dc = o.dcost > 0.0 && !hi_order;      // the l1 move term is carried by the NODES = 2 kernels only
  // one CTA per SM, but never more CTAs than 32-problem chunks
  p.slots = grid_for(B, 1, (long)sm_count * kBlocksPerSM) * kBlock;
  if (hi_order) {
    const int gp = B <= (int64_t)sm_count * 8 ? 32 : 8;
    p.kernel = KernelKey{kCollocKernel, gp, 1, 0};
    p.grid = grid_for(B, gp, sm_count);
    p.ws_bytes = group_ws_bytes(colloc::colloc_doubles_per_problem(nt, nodes - 1), p.grid, gp);
  } else if (circular_move || o.kernel == LMATO_KERNEL_COOP || (o.kernel != LMATO_KERNEL_THREAD && B <= kCoopMaxBatch)) {
    // lanes per problem in the stage-parallel phases: a whole warp per problem while that still gives every SM at
    // most ~8 warps (the latency regime), otherwise 8 lanes (four problems per warp)
    const int gp = (o.coop_lanes == 8 || o.coop_lanes == 32) ? o.coop_lanes : B <= (int64_t)sm_count * 8 ? 32 : 8;
    // CTAs per SM: one (255 registers per thread) while one CTA per SM holds the whole batch, else two
    const int bps = B <= (int64_t)sm_count * (kCoopBlock / gp) ? 1 : kCoopBlocksPerSM;
    p.kernel = KernelKey{kCoopKernel, gp, bps, !p.use_dc ? 0 : circular_move ? 2 : 1};
    p.grid = grid_for(B, gp, (long)sm_count * bps);
    p.ws_bytes = group_ws_bytes(coop::coop_doubles_per_problem(nt), p.grid, gp);
  } else {
    p.kernel = KernelKey{kThreadKernel, 1, kBlocksPerSM, p.use_dc ? 1 : 0};
    p.grid = p.slots / kBlock;
    p.ws_bytes = sizeof(double) * (size_t)(p.use_dc ? (int)dc::N_FIELDS : (int)N_FIELDS) * (size_t)nt * (size_t)p.slots;
  }
  // (a caller-supplied guess replaces the batch warm start; no batch warm start for the circular model with its move
  //  term either: the reference column of the 7-state solve carries a different MV)
  p.warm = !hi_order && !has_guess && !circular_move &&
           (o.warm_start == 2 || (o.warm_start == 1 && warm_batch >= kWarmStartMinBatch));
  p.alloc_bytes = p.ws_bytes;
  if (p.warm) {      // the reference solve: one warp of one CTA
    const size_t r = group_ws_bytes(coop::coop_doubles_per_problem(nt), 1, 32);
    if (r > p.alloc_bytes) p.alloc_bytes = r;
  }
  return p;
}

// The solver options of a batch on a mesh of nt nodes, with or without the move term.
inline Options solve_options(const lmato_options& o, int nt, bool use_dc) {
  Options O;
  // OTOL / RTOL (LO:31-32): how APMonitor maps them onto IPOPT's `tol` is not verifiable here, so the rule is
  // the conservative one: the solve runs to the tightest of tol, otol and rtol (defaults 1e-10, 1e-3, 1e-3).
  double tol = o.tol;
  if (o.otol > 0.0 && o.otol < tol) tol = o.otol;
  if (o.rtol > 0.0 && o.rtol < tol) tol = o.rtol;
  O.tol = tol; O.mu_init = o.mu_init; O.obj_scale = o.obj_scale;
  // barrier decrease exponent: IPOPT's 1.5 from the cold start, 2 from the batch warm start.  Measured on the
  // benchmark batch (warm): 1.3 / 1.5 / 1.7 / 2.0 / 2.5 / 3.0 -> 91 / 96 / 95 / 88 / 88 / 115 ms; from the cold
  // start 2.0 costs 0.7 iterations more than 1.5.  kappa_mu and tau_min do not matter.
  O.kappa_eps = o.kappa_eps; O.kappa_mu = 0.2; O.theta_mu = 1.5; O.tau_min = 0.99;
  O.delta_c = o.delta_c; O.tf_guess = o.tf_guess;
  O.max_iter = o.max_iter; O.max_ls = o.max_ls;
  O.mu_min_factor = o.mu_min_factor;
  O.n_polish = o.n_polish >= 0 ? o.n_polish : (use_dc ? 2 : 4);
  // ... 2 from the warm start WITH the move term only.  Without it the control on the singular arc is a nearly flat
  // direction, and the jump 1e-6 -> 1e-12 leaves a few problems in 10 000 on an error plateau until the stall guard
  // gives the warm attempt up -- each holding its warp: 65 536 problems, dcost = 0: 260-560 ms with 2, 66 ms with 1.5.
  O.theta_mu_warm = use_dc ? 2.0 : 1.5;
  const int on = o.objective_nodes > 0 ? o.objective_nodes : nt - 1;
  O.w_dcost = use_dc ? o.obj_scale * o.dcost / (double)on : 0.0;
  return O;
}

// The options of the warm start's reference solve: the batch-mean problem solved down to mu_ref only, without the
// move term (at mu_ref >> w it is immaterial): ~10 iterations from the cold start on the first call, 1-2 from the
// previous call's reference afterwards.
inline Options reference_options(Options O, double mu_ref) {
  O.tol = 10.0 * mu_ref; O.mu_min_factor = 0.1; O.n_polish = 0;
  O.w_dcost = 0.0;
  return O;
}

}  // namespace lmato
