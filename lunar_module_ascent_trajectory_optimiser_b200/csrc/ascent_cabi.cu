// C ABI + kernels of the batched ascent solver (sm_100a).  See include/lmato_b200.h.
//
// Three kernels solve the same NLP with the same IPM driver (ipm_iterate_t, ascent_ipm.cuh):
//   ascent_ipm_kernel   ONE PROBLEM PER THREAD, persistent warps, for batches that fill the GPU (>= ~1 wave of
//                       148 x 256 problems).  The stage data of a problem (55-67 doubles x nt) streams through a
//                       workspace in HBM laid out [stage][warp][field][lane]: every access of a warp is one
//                       coalesced 256-byte row, staged one stage ahead in shared memory with cp.async.  Each sweep
//                       re-evaluates the model, so the HBM traffic stays near 3x the algorithmic minimum.
//   ascent_coop_kernel  EIGHT LANES PER PROBLEM (ascent_coop.cuh), for everything smaller: a single solve, the
//                       1 024 / 4 096-problem configurations, a 65 536 batch strong-scaled over 8 GPUs.  Model
//                       evaluation is stage-parallel over the group and stored per stage; the Riccati recursion
//                       runs on the stored records with the cost-to-go distributed by rows over the group.
//   ascent_colloc_kernel 8 OR 32 LANES PER PROBLEM (ascent_colloc.cuh), the general path for NODES = 3..6.
// Each kernel sets up its shared constants and its workspace view and then runs one loop, solve_queue: it claims
// problems from a device-side queue and never returns to the host during a solve (barrier updates,
// fraction-to-boundary, filter line search and convergence masks live in the owning lanes).  Tensor cores are
// not used: the stage blocks are 8x8 FP64 and the recursion over stages is sequential (DESIGN.md).
// Post-solve checks run one problem per thread: coast_orbit_kernel (the PDF's orbit coast) and fly_control_kernel (the
// solved control flown through the continuous dynamics, ascent_fly.cuh).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <math.h>
#include <new>
#include <vector>

#include "../../include/lmato_b200.h"
#include "ascent_colloc.cuh"
#include "ascent_fly.cuh"
#include "ascent_plan.h"
#include "ascent_result.cuh"

using namespace lmato;

namespace {

thread_local char g_err[512] = "";

void set_err(const char* fmt, const char* a = "", const char* b = "") {
  snprintf(g_err, sizeof(g_err), fmt, a, b);
}

#define CUDA_TRY(expr)                                                        \
  do {                                                                        \
    cudaError_t e__ = (expr);                                                 \
    if (e__ != cudaSuccess) {                                                 \
      set_err("CUDA error: %s at %s", cudaGetErrorString(e__), #expr);        \
      return LMATO_ERR_CUDA;                                                  \
    }                                                                         \
  } while (0)

#ifndef LMATO_SYNC_PERIOD
#define LMATO_SYNC_PERIOD 1
#endif
// dynamic shared memory: the staging tiles, then one workspace view per thread
constexpr size_t kTileSmem = (size_t)(kBlock / 32) * 2 * TILE_ROWS * LANES * sizeof(double) + kBlock * sizeof(Ws);

struct KArgs {
  const double* params;  // [NPARAM][B]
  ResultOut res;         // the outputs; res.B is the batch size B of every [..][B] array here
  const double* guess_traj;  // caller-supplied start point [NVAR][nt][B] and [B], or null
  const double* guess_tf;
  double* ws;            // [N+1][slots/32][N_FIELDS][32]
  long slots;
  int N;
  const double* h;
  const double* tau;
  int* counter;
  int model;             // lmato_model_t
  double* ref;           // reference column (warm start), or null
  int ref_mode;          // 0 cold start; 1 solve and store the reference (starting from the previous one,
                         // if any); 2 start from the reference
  Options O;
  const colloc::Coll* coll;   // collocation rule in device memory (NODES >= 3 only)
};

// Mean of every parameter row over the batch: the reference problem of the warm start.
__global__ void __launch_bounds__(256) mean_params_kernel(const double* __restrict__ p, long B, double* out) {
  __shared__ double red[256];
  const int row = blockIdx.x;
  double acc = 0.0;
  for (long i = threadIdx.x; i < B; i += blockDim.x) acc += p[row * B + i];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[row] = red[0] / (double)B;
}

// Params padded to an odd number of doubles per thread so that the per-thread structs in shared memory
// are bank-conflict free (Params = 19 doubles -> stride 21 doubles = 42 words; 42 mod 32 = 10).
struct alignas(8) ParamsSlot { Params p; double pad[(sizeof(Params) / 8) % 2 == 0 ? 1 : 2]; };

static_assert(GuessSrc::V_Y == LMATO_V_Y && GuessSrc::V_YDOT == LMATO_V_YDOT && GuessSrc::V_X == LMATO_V_X &&
              GuessSrc::V_XDOT == LMATO_V_XDOT && GuessSrc::V_ANGLE == LMATO_V_ANGLE &&
              GuessSrc::V_ANGLEDOT == LMATO_V_ANGLEDOT && GuessSrc::V_U == LMATO_V_ANGLEDOUBLEDOT,
              "the guess uses the output layout of include/lmato_b200.h");

// How a warp leaves the problem queue of solve_queue.
enum QueueExit {
  kBlockBarrier,   // a block-wide vote every LMATO_SYNC_PERIOD-th round, which also keeps the warps of a CTA in step
  kWarpVote        // each warp on its own, once the queue is empty and its last chunk is written
};

// The persistent problem queue of every solve kernel.  A warp holds a chunk of 32 / GP problems, GP =
// SW::LANES_PER_PROBLEM lanes each (1 in the thread kernel); its groups run the IPM driver in lock step (same sweep at
// the same time, each with its own lane mask), finished problems wait until the warp's whole chunk is done, then the
// warp claims the next chunk.  IpmState (filter, barrier parameter, ...) is carried redundantly by the GP lanes of a
// problem: every decision of the driver is a function of group-uniform values.  P is this problem's slot of the
// kernel's shared Params; g and mask are this lane's index and lane mask in its group, as write_results takes them.
// The driver is inlined here with one call site each of ipm_start, ipm_iterate_t, ipm_restart and write_results
// (DESIGN.md section 3a).
template <class SW, QueueExit EXIT, class WS>
__device__ __forceinline__ void solve_queue(const KArgs& a, Params& P, const Mesh& M, const Options& O, const WS& W,
                                            int g, unsigned mask) {
  constexpr int GP = SW::LANES_PER_PROBLEM;
  constexpr int PPW = 32 / GP;                 // problems per warp
  const int lane = threadIdx.x & 31;
  IpmState S;
  bool active = false;        // this lane holds an unfinished problem
  bool pending = false;       // this lane holds a finished problem whose results are not written yet
  bool exhausted = false;     // the queue is empty (warp-uniform)
  bool first = true;
  long b = -1;
  unsigned round = 0;
  while (true) {
    // ---- a warp whose problems are all finished claims the next chunk (warp-uniform branch) ----
    const bool chunk_done = !__any_sync(0xffffffffu, active);
    // ---- a finished chunk writes its results with all 32 lanes together: every row of the
    //      [variable][node][problem] output is then one coalesced store per warp (the output
    //      may be pinned host memory written over PCIe while the other warps keep computing) ----
    if (chunk_done && __any_sync(0xffffffffu, pending)) {
      if (pending) write_results<SW, GP>(a.res, P, M, O.obj_scale, a.model, W, g, mask, S, b);
      pending = false;
    }
    if (!exhausted && chunk_done) {
      // first chunk: static round-robin over CTAs (spreads a small batch over all SMs);
      // afterwards: the device-wide queue
      int chunk = 0;
      if (first) {
        chunk = (threadIdx.x / 32) * gridDim.x + blockIdx.x;
        first = false;
      } else {
        if (lane == 0) chunk = atomicAdd(a.counter, 1) + gridDim.x * (kBlock / 32);
        chunk = __shfl_sync(0xffffffffu, chunk, 0);
      }
      if ((long)chunk * PPW >= a.res.B) {
        exhausted = true;
      } else {
        b = (long)chunk * PPW + lane / GP;
        if (b < a.res.B) {
          if (g == 0) P = derive_params(a.params, a.res.B, b, a.model, SW::MOVE_TERM == 2);
          coop::Grp<GP>::sync(mask);
          // ref_mode 2: start from the batch reference.  ref_mode 1 (the reference solve itself):
          // start from the previous call's reference if the handle has one (consecutive batches of a
          // campaign have nearly the same mean, so it re-converges in one or two iterations).
          ipm_start<SW>(P, M, O, W, GuessSrc{a.guess_traj, a.guess_tf, a.res.B, b}, a.ref_mode != 0 ? a.ref : nullptr, S);
          active = true;
        }
      }
    }
    if constexpr (EXIT == kBlockBarrier) {
      // ---- all eight warps of the SM start each iteration together: they then run the same sweep
      //      (same code) at the same time, which keeps the 32 KB instruction cache effective ----
      // (every LMATO_SYNC_PERIOD-th round: a barrier per iteration costs more in waiting than it
      //  gains, because line-search retries differ between warps; the imbalance averages out over
      //  a few iterations while the warps stay close enough to share the instruction cache)
      if ((round++ % LMATO_SYNC_PERIOD) == 0 && !__syncthreads_or((active || !exhausted) ? 1 : 0)) break;
    } else {
      // (no block barrier per iteration here: the warps of an SM are few and their sweeps are short; a warp that
      //  waits for its neighbours' line-search retries loses more than the instruction cache gains)
      if (exhausted && !__any_sync(0xffffffffu, active || pending)) break;
    }
    if (active && ipm_iterate_t<SW>(P, M, O, W, S)) {
      if (ipm_restart<SW>(P, M, O, W, S)) continue;      // this problem restarts from another start point
      active = false;
      if constexpr (SW::STORES_REF) {
        // ref_mode 1, the reference solve of the batch warm start: store the reference, write no results
        if (a.ref_mode == 1) {
          SolveOut out;
          ipm_result(S, out);
          SW::store_ref(P, M, W, out.cur, S.cur, S.ctl.mu, out.status == ST_CONVERGED, a.ref);
          continue;
        }
      }
      pending = true;      // results are written when the whole chunk is done (see above)
    }
  }
}

// SW = Sweeps7 (dcost = 0) or Sweeps8 (with the reference's move-suppression term, LO:99)
template <class SW>
__global__ void __launch_bounds__(kBlock, kBlocksPerSM) ascent_ipm_kernel(KArgs a) {
  // Per-problem constants are read in every stage of every sweep.  They live in shared memory: as
  // registers they would be spilled (255 are already in use), and a spill is reloaded from local
  // memory, which misses the thrashed L1 every stage.
  __shared__ ParamsSlot sP[kBlock];
  __shared__ Options sO;
  __shared__ Mesh sM;
  if (threadIdx.x == 0) { sO = a.O; sM = Mesh{a.N, a.h, a.tau}; }
  __syncthreads();
  const long slot = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const long nwarps = a.slots / LANES;
  // staging tiles: [warp][2 buffers][TILE_ROWS][32 lanes] doubles of dynamic shared memory
  extern __shared__ __align__(16) double sTiles[];
  const unsigned tile0 = (unsigned)__cvta_generic_to_shared(sTiles) +
                         (unsigned)(((threadIdx.x / 32) * 2 * TILE_ROWS * LANES + lane) * sizeof(double));
  // the workspace view is read inside every stage as well: shared memory for the same reason
  // (24-byte stride: conflict-free per half warp)
  Ws* sW = reinterpret_cast<Ws*>(sTiles + (size_t)(kBlock / 32) * 2 * TILE_ROWS * LANES);   // after the tiles
  sW[threadIdx.x] = Ws{a.ws + ((slot / LANES) * SW::NFIELDS) * LANES + lane, nwarps * SW::NFIELDS * LANES, tile0};
  // (the reference solve of the batch warm start, ref_mode 1, runs on the cooperative kernel)
  solve_queue<SW, kBlockBarrier>(a, sP[threadIdx.x].p, sM, sO, sW[threadIdx.x], 0, 1u << lane);
}

// ---------------------------------------------------------------------------------------
// cooperative kernel: G lanes per problem (ascent_coop.cuh)
// ---------------------------------------------------------------------------------------
constexpr int kCoopScrStride = coop::SCR_DOUBLES;       // per group: record ring + transpose tiles (even: 16-byte aligned)
static_assert(kCoopBlock == kBlock, "solve_queue counts kBlock / 32 warps in every CTA");
constexpr size_t coop_smem(int gp) { return sizeof(double) * (size_t)(kCoopBlock / gp) * kCoopScrStride; }

//   GP = 8 : four problems per warp, for batches that can fill the GPU that way;
//   GP = 32: the whole warp works on one problem (the stage-parallel phases are four times shorter), for
//            the latency regime: up to a few problems per SM.
//   BPS = CTAs per SM: 1 leaves 255 registers per thread (no spills), 2 halves them for twice the problems in flight.
template <int G, int GP, int MOVE, int BPS>      // MOVE: 0 no move term, 1 move term (LO:99), 2 the circular model's (MV = angle)
__global__ void __launch_bounds__(kCoopBlock, BPS) ascent_coop_kernel(KArgs a) {
  using SW = SweepsCoop<G, GP, MOVE>;
  constexpr int GPB = kCoopBlock / GP;         // groups per block
  __shared__ ParamsSlot sP[GPB];
  __shared__ Options sO;
  __shared__ Mesh sM;
  extern __shared__ __align__(16) double sScr[];    // [GPB][kCoopScrStride]
  if (threadIdx.x == 0) { sO = a.O; sM = Mesh{a.N, a.h, a.tau}; }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int grp = threadIdx.x / GP;
  const unsigned gmask = GP == 32 ? 0xffffffffu : (((1u << GP) - 1u) << ((lane / GP) * GP));
  const unsigned smask = ((1u << G) - 1u) << ((lane / GP) * GP);
  const long slot = (long)blockIdx.x * GPB + grp;
  // workspace layout by regime (ascent_coop.cuh, CwsT): stage-major blocks when a whole warp walks one problem
  const coop::CwsT<(GP == 32)> W{a.ws + slot * coop::coop_doubles_per_problem(a.N + 1), a.N + 1, sScr + grp * kCoopScrStride,
                                 lane % GP, gmask, smask, 0.0, 0.0, 0, 0u};
  if (W.g == 0) coop::ring_init_barriers(W.bars());      // the mbarriers of this group's record ring
  __syncthreads();
  solve_queue<SW, kWarpVote>(a, sP[grp].p, sM, sO, W, W.g, W.mask);
}

// ---------------------------------------------------------------------------------------
// higher-order collocation kernel (NODES = 3..6, ascent_colloc.cuh): GP lanes per problem
// ---------------------------------------------------------------------------------------
template <int GP>
__global__ void __launch_bounds__(kCoopBlock, 1) ascent_colloc_kernel(KArgs a) {
  constexpr int GPB = kCoopBlock / GP;
  __shared__ ParamsSlot sP[GPB];
  __shared__ Options sO;
  __shared__ Mesh sM;
  __shared__ colloc::Coll sC;
  if (threadIdx.x == 0) { sO = a.O; sM = Mesh{a.N, a.h, a.tau}; sC = *a.coll; }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int grp = threadIdx.x / GP;
  const unsigned gmask = GP == 32 ? 0xffffffffu : (((1u << GP) - 1u) << ((lane / GP) * GP));
  const long slot = (long)blockIdx.x * GPB + grp;
  colloc::Nws W;
  W.L.init(sC.m);
  W.base = a.ws + slot * colloc::colloc_doubles_per_problem(a.N + 1, sC.m);
  W.N1 = a.N + 1; W.C = &sC; W.g = lane % GP; W.mask = gmask; W.dw = 0.0; W.pimax = 0.0; W.ls_flag = 0;
  solve_queue<SweepsColloc<GP>, kWarpVote>(a, sP[grp].p, sM, sO, W, W.g, W.mask);
}

// Every solve-kernel instantiation a launch plan (ascent_plan.h) can name, with its launch shape.  The thread kernel's
// staging tiles and the cooperative kernel's record rings need the opt-in shared-memory size (thread kernel: 158 KB
// dynamic + 42 KB static per CTA).
struct SolveKernel {
  KernelKey key;
  void (*fn)(KArgs);
  int block;
  size_t smem;         // dynamic shared memory
};
#define COOP_KERNEL(GP, MOVE, BPS) {{kCoopKernel, GP, BPS, MOVE}, ascent_coop_kernel<kCoopG, GP, MOVE, BPS>, kCoopBlock, coop_smem(GP)}
const SolveKernel kSolveKernels[] = {
  {{kThreadKernel, 1, kBlocksPerSM, 0}, ascent_ipm_kernel<Sweeps7>, kBlock, kTileSmem},
  {{kThreadKernel, 1, kBlocksPerSM, 1}, ascent_ipm_kernel<Sweeps8>, kBlock, kTileSmem},
  COOP_KERNEL(8, 0, 1), COOP_KERNEL(8, 1, 1), COOP_KERNEL(8, 2, 1),
  COOP_KERNEL(8, 0, 2), COOP_KERNEL(8, 1, 2), COOP_KERNEL(8, 2, 2),
  COOP_KERNEL(32, 0, 1), COOP_KERNEL(32, 1, 1), COOP_KERNEL(32, 2, 1),
  COOP_KERNEL(32, 0, 2), COOP_KERNEL(32, 1, 2), COOP_KERNEL(32, 2, 2),
  {{kCollocKernel, 8, 1, 0}, ascent_colloc_kernel<8>, kCoopBlock, 0},
  {{kCollocKernel, 32, 1, 0}, ascent_colloc_kernel<32>, kCoopBlock, 0},
};
#undef COOP_KERNEL

// Launches the table's kernel for `key` on `grid` CTAs.
lmato_status_t launch(const KernelKey& key, long grid, cudaStream_t st, const KArgs& a) {
  for (const SolveKernel& k : kSolveKernels)
    if (k.key == key) {
      k.fn<<<(int)grid, k.block, k.smem, st>>>(a);
      CUDA_TRY(cudaGetLastError());
      return LMATO_OK;
    }
  set_err("lmato_solve_batch: no solve kernel is instantiated for the launch plan");
  return LMATO_ERR_INVALID;
}

// Makes *p hold at least `bytes` bytes of device memory, freeing and reallocating it when it is smaller.  A caller
// whose old buffer may still be in use on the device waits for that before it asks for more.
cudaError_t grow(double** p, size_t* cap, size_t bytes) {
  if (bytes <= *cap) return cudaSuccess;
  const cudaError_t e = cudaFree(*p);
  *p = nullptr; *cap = 0;
  if (e != cudaSuccess) return e;
  const cudaError_t m = cudaMalloc(p, bytes);
  if (m == cudaSuccess) *cap = bytes;
  return m;
}

// FP64 FMA peak: 8 independent chains per thread, no memory traffic.
__global__ void __launch_bounds__(256) dfma_peak_kernel(double* out, int iters) {
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5,
         a6 = a0 + 6, a7 = a0 + 7;
  const double m = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; ++i) {
    a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
    a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
  }
  out[(long)blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

// Post-solve orbit check of the reference PDF (p.28-29 src 185-237): explicit Euler two-body coast,
// one problem per thread, everything in registers.  state/out: [4][B] / [6][B], SI, Moon-centred.
__global__ void __launch_bounds__(128) coast_orbit_kernel(const double* __restrict__ state, long B, double gm,
                                                          double dt, long nsteps, double* __restrict__ out) {
  const long b = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  double x = state[0 * B + b], y = state[1 * B + b], vx = state[2 * B + b], vy = state[3 * B + b];
  double r2 = fma(x, x, y * y);
  double r2min = r2, r2max = r2;
  for (long i = 0; i < nsteps; ++i) {
    const double inv = lm_rsqrt(r2);
    const double k = gm * inv * inv * inv;
    const double ax = -k * x, ay = -k * y;            // src 207-208
    x = fma(vx, dt, x);                               // src 231-232 (old velocity)
    y = fma(vy, dt, y);
    vx = fma(ax, dt, vx);                             // src 233-234
    vy = fma(ay, dt, vy);
    r2 = fma(x, x, y * y);
    r2min = fmin(r2min, r2);
    r2max = fmax(r2max, r2);
  }
  out[0 * B + b] = sqrt(r2min); out[1 * B + b] = sqrt(r2max);
  out[2 * B + b] = x; out[3 * B + b] = y; out[4 * B + b] = vx; out[5 * B + b] = vy;
}

// Post-solve flight (ascent_fly.cuh): one problem per thread; every read and write of a [..][B] row is coalesced
// across the warp's 32 problems.
__global__ void __launch_bounds__(128) fly_control_kernel(const double* __restrict__ params, long B, int model,
                                                          const double* __restrict__ tau, int nt,
                                                          const double* __restrict__ traj, const double* __restrict__ tf,
                                                          int substeps, double* __restrict__ fin, double* __restrict__ out) {
  const long b = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const Params P = derive_params(params, B, b, model);
  fly_one(P, model, tau, nt, traj, tf[b], substeps, B, b, fin, out);
}

// Self-test of the branch-free math against the CUDA library: max relative errors of
// rcp, rsqrt, log over [1e-40, 1e3] and max absolute errors of sin, cos over [0, 3.5].
__global__ void math_selftest_kernel(double* out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double t = (double)i / (double)(n - 1);
  const double x = exp(log(1e-40) + t * (log(1e3) - log(1e-40)));
  const double a = 3.5 * t;
  double s, c;
  lm_sincos_small(a, &s, &c);
  const double lx = log(x);
  out[i * 5 + 0] = fabs(lm_rcp(x) * x - 1.0);
  out[i * 5 + 1] = fabs(lm_rsqrt(x) * sqrt(x) - 1.0);
  out[i * 5 + 2] = fabs(lm_log_pos(x) - lx) / fmax(fabs(lx), 1e-3);
  out[i * 5 + 3] = fabs(s - sin(a));
  out[i * 5 + 4] = fabs(c - cos(a));
}

}  // namespace

struct lmato_handle {
  int device = 0;
  int nt = 0;
  int nodes = 2;
  int model = 0;
  int sm_count = 0;
  double* d_h = nullptr;
  double* d_tau = nullptr;
  double* d_ws = nullptr;
  size_t ws_bytes = 0;
  int* d_counter = nullptr;
  // the device copy of a host solve's arrays (stage_and_solve), for lmato_solve_batch_host and the device list
  double* d_stage = nullptr; size_t stage_bytes = 0;
  double* d_ref = nullptr;        // reference column of the warm start: [REF_ROWS][nt]
  double* d_refparams = nullptr;  // [NPARAM] batch-mean parameters + scratch outputs of the reference solve
  lmato_options opt;
  double* sens_out = nullptr;     // optional extra output of the next solves (lmato_set_sensitivity_output)
  double* psens_out = nullptr;    // another one (lmato_set_param_sensitivity_output)
  const double* guess_traj = nullptr;   // optional start point of the next solves (lmato_set_initial_guess)
  const double* guess_tf = nullptr;
  int64_t launches = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaStream_t last_stream = nullptr;
  bool timed = false;
  colloc::Coll coll;              // collocation rule for NODES >= 3 ...
  colloc::Coll* d_coll = nullptr; // ... and its device copy
};

// Collocation rule of GEKKO NODES = n (SURVEY Appendix B.2): Lobatto points on [0,1] including both ends;
// h N f_{1..m} = z_{1..m} - z_0 with N_ij = int_0^{tau_i} l_j(s) ds, l_j the Lagrange basis on tau_1..tau_m.
static bool collocation_rule(int nodes, colloc::Coll* C) {
  if (nodes < 2 || nodes > 6) return false;
  const int m = nodes - 1;
  double pts[6];                         // Lobatto points on [-1, 1]
  switch (nodes) {
    case 2: pts[0] = -1; pts[1] = 1; break;
    case 3: pts[0] = -1; pts[1] = 0; pts[2] = 1; break;
    case 4: { const double a = sqrt(1.0 / 5.0); pts[0] = -1; pts[1] = -a; pts[2] = a; pts[3] = 1; break; }
    case 5: { const double a = sqrt(3.0 / 7.0); pts[0] = -1; pts[1] = -a; pts[2] = 0; pts[3] = a; pts[4] = 1; break; }
    default: {
      const double a = sqrt(1.0 / 3.0 - 2.0 * sqrt(7.0) / 21.0), b = sqrt(1.0 / 3.0 + 2.0 * sqrt(7.0) / 21.0);
      pts[0] = -1; pts[1] = -b; pts[2] = -a; pts[3] = a; pts[4] = b; pts[5] = 1; break;
    }
  }
  double tau[6];
  for (int i = 0; i < nodes; ++i) tau[i] = 0.5 * (pts[i] + 1.0);
  C->m = m;
  for (int i = 0; i < colloc::MAXM; ++i) { C->tau[i] = 0.0; for (int j = 0; j < colloc::MAXM; ++j) C->N[i][j] = 0.0; }
  for (int i = 0; i < m; ++i) C->tau[i] = tau[i + 1];
  for (int j = 0; j < m; ++j) {
    double c[6] = {1, 0, 0, 0, 0, 0};    // coefficients of l_j, ascending powers
    int deg = 0;
    for (int q = 0; q < m; ++q) {
      if (q == j) continue;
      const double den = tau[j + 1] - tau[q + 1];
      double n[6] = {0, 0, 0, 0, 0, 0};
      for (int d = 0; d <= deg; ++d) { n[d + 1] += c[d] / den; n[d] -= c[d] * tau[q + 1] / den; }
      ++deg;
      for (int d = 0; d <= deg; ++d) c[d] = n[d];
    }
    for (int i = 0; i < m; ++i) {
      double s = 0.0, tp = tau[i + 1];
      for (int d = 0; d <= deg; ++d) { s += c[d] * tp / (double)(d + 1); tp *= tau[i + 1]; }
      C->N[i][j] = s;
    }
  }
  return true;
}

// device-side part of lmato_create (every failure path returns through the caller's lmato_destroy)
static lmato_status_t create_device_state(lmato_handle* H, const std::vector<double>& h, const std::vector<double>& tau) {
  const int nt = H->nt;
  CUDA_TRY(cudaSetDevice(H->device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, H->device));
  H->sm_count = prop.multiProcessorCount;
  for (const SolveKernel& k : kSolveKernels)
    if (k.smem > 0) CUDA_TRY(cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.smem));
  CUDA_TRY(cudaMalloc(&H->d_h, sizeof(double) * nt));
  CUDA_TRY(cudaMalloc(&H->d_tau, sizeof(double) * nt));
  CUDA_TRY(cudaMemcpy(H->d_h, h.data(), sizeof(double) * nt, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(H->d_tau, tau.data(), sizeof(double) * nt, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMalloc(&H->d_counter, sizeof(int)));
  CUDA_TRY(cudaMalloc(&H->d_ref, sizeof(double) * (size_t)dc::REF_ROWS * nt));   // dc:: is the larger layout
  CUDA_TRY(cudaMemset(H->d_ref, 0, sizeof(double) * (size_t)dc::REF_ROWS * nt));   // REF_OK = 0: no reference yet
  CUDA_TRY(cudaMalloc(&H->d_refparams, sizeof(double) * (LMATO_NPARAM + 8)));
  CUDA_TRY(cudaMalloc(&H->d_coll, sizeof(colloc::Coll)));
  CUDA_TRY(cudaMemcpy(H->d_coll, &H->coll, sizeof(colloc::Coll), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaEventCreate(&H->ev0));
  CUDA_TRY(cudaEventCreate(&H->ev1));
  return LMATO_OK;
}

extern "C" {

const char* lmato_last_error(void) { return g_err; }
const char* lmato_version(void) { return "lmato_b200 0.1 (sm_100a)"; }

void lmato_default_options(lmato_options* o) {
  if (o) *o = default_options();
}

lmato_status_t lmato_create(lmato_handle** out, int32_t device, int32_t nt, const double* time,
                            int32_t nodes, int32_t model) {
  if (!out) { set_err("lmato_create: out is NULL"); return LMATO_ERR_INVALID; }
  *out = nullptr;
  if (nt < 2) { set_err("lmato_create: nt must be >= 2"); return LMATO_ERR_INVALID; }
  if (nodes < 2 || nodes > 6) { set_err("lmato_create: NODES must be 2..6 (GEKKO's range, LO:25)"); return LMATO_ERR_INVALID; }
  if (model != LMATO_MODEL_ELLIPTICAL && model != LMATO_MODEL_CIRCULAR) {
    set_err("lmato_create: unknown model");
    return LMATO_ERR_INVALID;
  }
  if (nodes > 2 && model != LMATO_MODEL_ELLIPTICAL) {
    set_err("lmato_create: NODES > 2 is implemented for the elliptical model (Launch_Optimiser.py) only");
    return LMATO_ERR_UNSUPPORTED;
  }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    set_err("lmato_create: no CUDA device available (%s); there is no CPU fallback",
            e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    return LMATO_ERR_NO_DEVICE;
  }
  if (device < 0 || device >= ndev) { set_err("lmato_create: bad device ordinal"); return LMATO_ERR_INVALID; }
  std::vector<double> h(nt), tau(nt);
  for (int k = 0; k < nt; ++k) tau[k] = time ? time[k] : (double)k / (double)(nt - 1);   // LO:21
  if (tau[0] != 0.0) { set_err("lmato_create: time[0] must be 0"); return LMATO_ERR_INVALID; }
  h[0] = 0.0;
  for (int k = 1; k < nt; ++k) {
    h[k] = tau[k] - tau[k - 1];
    if (!(h[k] > 0.0)) { set_err("lmato_create: time must be strictly increasing"); return LMATO_ERR_INVALID; }
  }
  lmato_handle* H = new (std::nothrow) lmato_handle();
  if (!H) { set_err("lmato_create: out of host memory"); return LMATO_ERR_INVALID; }
  H->device = device; H->nt = nt; H->nodes = nodes; H->model = model;
  lmato_default_options(&H->opt);
  collocation_rule(nodes, &H->coll);
  const lmato_status_t rc = create_device_state(H, h, tau);
  if (rc != LMATO_OK) { lmato_destroy(H); return rc; }      // frees whatever was allocated before the failure
  *out = H;
  return LMATO_OK;
}

lmato_status_t lmato_destroy(lmato_handle* h) {
  if (!h) return LMATO_OK;
  cudaSetDevice(h->device);
  cudaFree(h->d_h); cudaFree(h->d_tau); cudaFree(h->d_ws); cudaFree(h->d_counter);
  cudaFree(h->d_stage); cudaFree(h->d_ref); cudaFree(h->d_refparams); cudaFree(h->d_coll);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  delete h;
  return LMATO_OK;
}

lmato_status_t lmato_set_options(lmato_handle* h, const lmato_options* o) {
  if (!h || !o) { set_err("lmato_set_options: NULL argument"); return LMATO_ERR_INVALID; }
  if (!(o->tol > 0) || !(o->mu_init > 0) || !(o->obj_scale > 0) || !(o->delta_c > 0) ||
      !(o->tf_guess > 0 && o->tf_guess < 1) || o->max_iter < 0 || o->max_ls < 1 ||
      !(o->mu_min_factor > 0 && o->mu_min_factor <= 1) || o->n_polish < -1 ||
      (o->warm_start < 0 || o->warm_start > 2) || !(o->mu_ref > 0 && o->mu_ref <= o->mu_init) ||
      !(o->dcost >= 0) || o->objective_nodes < 0 || !(o->kappa_eps >= 1.0) ||
      o->kernel < LMATO_KERNEL_AUTO || o->kernel > LMATO_KERNEL_COOP || !(o->otol >= 0) || !(o->rtol >= 0) ||
      (o->coop_lanes != 0 && o->coop_lanes != 8 && o->coop_lanes != 32)) {
    set_err("lmato_set_options: option out of range");
    return LMATO_ERR_INVALID;
  }
  h->opt = *o;
  return LMATO_OK;
}

lmato_status_t lmato_workspace_bytes(lmato_handle* h, int64_t B, int64_t* bytes) {
  if (!h || !bytes || B < 0) { set_err("lmato_workspace_bytes: bad argument"); return LMATO_ERR_INVALID; }
  *bytes = (int64_t)plan_solve(h->sm_count, h->nt, h->nodes, h->model, h->opt, B, h->guess_traj != nullptr, B).ws_bytes;
  return LMATO_OK;
}

lmato_status_t lmato_kernel_launches(lmato_handle* h, int64_t* n) {
  if (!h || !n) { set_err("lmato_kernel_launches: bad argument"); return LMATO_ERR_INVALID; }
  *n = h->launches;
  return LMATO_OK;
}

// What kind of memory a registered optional buffer (sensitivity output, start point) points at.  The device entry
// point needs memory the kernel can address (device, managed, or pinned host memory); the host entry point needs
// memory the host can address.  Answers true when the runtime cannot tell (plain host memory is "unregistered").
static bool kernel_can_address(const void* p) {
  if (!p) return true;
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged ||
         (attr.type == cudaMemoryTypeHost && attr.devicePointer != nullptr);
}
static bool host_can_address(const void* p) {
  if (!p) return true;
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) { cudaGetLastError(); return true; }
  return attr.type != cudaMemoryTypeDevice;
}

// The argument checks of every solve entry point (`fn` names it in the message).  An empty batch is valid.
static lmato_status_t check_batch(const char* fn, const void* handle, const double* params, int64_t B,
                                  const double* out_tf, const double* out_final_mass, const int32_t* out_status,
                                  const int32_t* out_iters) {
  if (!handle) { set_err("%s: NULL handle", fn); return LMATO_ERR_INVALID; }
  if (B < 0) { set_err("%s: negative batch", fn); return LMATO_ERR_INVALID; }
  if (B > 0 && (!params || !out_tf || !out_final_mass || !out_status || !out_iters)) {
    set_err("%s: NULL buffer", fn);
    return LMATO_ERR_INVALID;
  }
  return LMATO_OK;
}

// Solves the out.B > 0 problems of `params` into `out`, starting from guess_traj / guess_tf when they are given, on
// h's device (the current one).  The problems belong to a batch of warm_batch problems (ascent_plan.h, plan_solve).
// Every pointer is a device pointer.
static lmato_status_t solve_batch(lmato_handle* h, const double* params, const double* guess_traj, const double* guess_tf,
                                  const ResultOut& out, cudaStream_t st, int64_t warm_batch) {
  if (h->nodes > 2 && (out.sens || out.psens || guess_traj)) {
    set_err("lmato_solve_batch: sensitivities and caller-supplied start points are implemented for NODES = 2 only");
    return LMATO_ERR_UNSUPPORTED;
  }
  // Every solve on a handle shares its workspace, work-queue counter and warm-start reference.  A solve issued on
  // a different stream than the previous one first waits (on the device) for that one to finish.
  if (h->timed && st != h->last_stream) CUDA_TRY(cudaStreamWaitEvent(st, h->ev1, 0));
  const int64_t B = out.B;
  const LaunchPlan plan = plan_solve(h->sm_count, h->nt, h->nodes, h->model, h->opt, B, guess_traj != nullptr, warm_batch);
  if (plan.alloc_bytes > h->ws_bytes && h->timed) CUDA_TRY(cudaEventSynchronize(h->ev1));   // the previous solve may still be using it
  CUDA_TRY(grow(&h->d_ws, &h->ws_bytes, plan.alloc_bytes));
  CUDA_TRY(cudaMemsetAsync(h->d_counter, 0, sizeof(int), st));
  KArgs a;
  a.params = params;
  a.res = out;
  a.res.params = params;
  a.guess_traj = guess_traj; a.guess_tf = guess_tf;
  a.ws = h->d_ws; a.slots = plan.slots; a.N = h->nt - 1; a.h = h->d_h; a.tau = h->d_tau;
  a.counter = h->d_counter;
  a.model = h->model;
  a.ref = nullptr; a.ref_mode = 0;
  a.O = solve_options(h->opt, h->nt, plan.use_dc);
  a.coll = h->d_coll;
  CUDA_TRY(cudaEventRecord(h->ev0, st));
  if (plan.warm) {
    // the reference problem is the batch mean, solved by ONE group of the cooperative kernel
    mean_params_kernel<<<LMATO_NPARAM, 256, 0, st>>>(params, B, h->d_refparams);
    CUDA_TRY(cudaGetLastError());
    KArgs r = a;
    double* scratch = h->d_refparams + LMATO_NPARAM;
    r.params = h->d_refparams;
    r.res = ResultOut{nullptr, scratch, scratch + 1, (int*)(scratch + 2), (int*)(scratch + 3), scratch + 4, nullptr, 1};
    r.guess_traj = nullptr; r.guess_tf = nullptr;
    r.ref = h->d_ref; r.ref_mode = 1;
    r.O = reference_options(a.O, h->opt.mu_ref);
    const lmato_status_t rc = launch(KernelKey{kCoopKernel, 32, 1, 0}, 1, st, r);
    if (rc != LMATO_OK) return rc;
    CUDA_TRY(cudaMemsetAsync(h->d_counter, 0, sizeof(int), st));
    a.ref = h->d_ref; a.ref_mode = 2;
    h->launches += 2;
  }
  const lmato_status_t rc = launch(plan.kernel, plan.grid, st, a);
  if (rc != LMATO_OK) return rc;
  CUDA_TRY(cudaEventRecord(h->ev1, st));
  h->last_stream = st; h->timed = true;
  h->launches += 1;
  return LMATO_OK;
}

lmato_status_t lmato_solve_batch(lmato_handle* h, const double* params, int64_t B,
                                 double* out_traj, double* out_tf, double* out_final_mass,
                                 int32_t* out_status, int32_t* out_iters, double* out_kkt,
                                 void* stream) {
  const lmato_status_t rc = check_batch("lmato_solve_batch", h, params, B, out_tf, out_final_mass, out_status, out_iters);
  if (rc != LMATO_OK || B == 0) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  if (!kernel_can_address(h->sens_out) || !kernel_can_address(h->psens_out) || !kernel_can_address(h->guess_traj) ||
      !kernel_can_address(h->guess_tf)) {
    set_err("lmato_solve_batch: the registered sensitivity output / start point is not device-addressable memory "
            "(lmato_solve_batch takes DEVICE pointers; use lmato_solve_batch_host for host buffers)");
    return LMATO_ERR_INVALID;
  }
  return solve_batch(h, params, h->guess_traj, h->guess_tf,
                     ResultOut{out_traj, out_tf, out_final_mass, out_status, out_iters, out_kkt, h->sens_out, (long)B,
                               h->psens_out},
                     (cudaStream_t)stream, B);
}

lmato_status_t lmato_last_kernel_ms(lmato_handle* h, double* ms) {
  if (!h || !ms) { set_err("lmato_last_kernel_ms: bad argument"); return LMATO_ERR_INVALID; }
  if (!h->timed) { set_err("lmato_last_kernel_ms: no solve has been launched"); return LMATO_ERR_INVALID; }
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaEventSynchronize(h->ev1));
  float f = 0.f;
  CUDA_TRY(cudaEventElapsedTime(&f, h->ev0, h->ev1));
  *ms = (double)f;
  return LMATO_OK;
}

// Device-usable alias of a host buffer if the caller pinned it (cudaHostAlloc / cudaHostRegister /
// torch pin_memory), else nullptr.  With unified addressing pinned host memory is mapped into the
// device's address space, so the kernel can store results straight into it.
static double* pinned_alias(double* host) {
  if (!host) return nullptr;
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  if (attr.type != cudaMemoryTypeHost || !attr.devicePointer) return nullptr;
  return static_cast<double*>(attr.devicePointer);
}

// The host arrays of one solve (include/lmato_b200.h), each a [rows][B] block: the inputs first, then the outputs.  A
// shard of the batch is the columns [lo, lo + n) of every array.  An array the caller passes as NULL is absent.
enum HostArrayId { kParams, kGuessTraj, kGuessTf, kTraj, kSens, kPsens, kTf, kFinalMass, kKkt, kStatus, kIters, kHostArrays };
constexpr int kHostInputs = kTraj;

struct HostArray {
  void* host;          // the caller's array, or NULL
  size_t rows, elem;   // elem: bytes per element
  void* dev;           // the shard's [rows][n] block that the solve reads or writes (set by stage_and_solve)
};

struct HostSolve {
  HostArray a[kHostArrays];
  int64_t B, lo, n;
};

static HostSolve host_solve(int nt, int64_t B, const double* params, const double* guess_traj, const double* guess_tf,
                            double* traj, double* sens, double* psens, double* tf, double* final_mass, double* kkt,
                            int32_t* status, int32_t* iters) {
  const size_t d = sizeof(double), i = sizeof(int32_t), nv = (size_t)LMATO_NVAR * nt;
  return HostSolve{{{const_cast<double*>(params), LMATO_NPARAM, d}, {const_cast<double*>(guess_traj), nv, d},
                    {const_cast<double*>(guess_tf), 1, d}, {traj, nv, d}, {sens, LMATO_NSENS, d},
                    {psens, LMATO_NPARAM, d}, {tf, 1, d},
                    {final_mass, 1, d}, {kkt, 1, d}, {status, 1, i}, {iters, 1, i}},
                   B, 0, 0};
}

// Copies the shard's columns of one array between the caller's block and the device.  The whole batch, or a single
// row, is one contiguous run and takes one flat copy (the 1 GB of trajectories of a 65 536-problem solve among them);
// the columns of a block of several rows take one 2D copy.
static cudaError_t copy_columns(const HostSolve& s, const HostArray& a, cudaMemcpyKind kind, cudaStream_t st) {
  char* host = static_cast<char*>(a.host) + a.elem * s.lo;
  const size_t w = a.elem * s.n, pitch = a.elem * s.B;
  const bool up = kind == cudaMemcpyHostToDevice;
  if (s.n == s.B || a.rows == 1)
    return up ? cudaMemcpyAsync(a.dev, host, w * a.rows, kind, st) : cudaMemcpyAsync(host, a.dev, w * a.rows, kind, st);
  return up ? cudaMemcpy2DAsync(a.dev, w, host, pitch, w, a.rows, kind, st)
            : cudaMemcpy2DAsync(host, pitch, a.dev, w, w, a.rows, kind, st);
}

// Carves h's staging buffer for the columns [lo, lo + n) of s, uploads their inputs and launches their solve on st
// (h's device is the current one).  Nothing here waits for the device unless the staging buffer has to grow.
// in_place: the shard is the whole batch, and a pinned trajectory array is written by the kernel directly.
static lmato_status_t stage_and_solve(lmato_handle* h, HostSolve& s, int64_t lo, int64_t n, cudaStream_t st,
                                      bool in_place) {
  s.lo = lo; s.n = n;
  // The trajectories are 16 KB per problem (1 GB for 65 536 problems).  If the caller's array is pinned the kernel
  // can write them there directly, chunk by chunk as problems finish, so that the transfer over PCIe overlaps the
  // solve.  The kernel writes rows of stride n, so only a whole batch can be written in place.
  double* alias = in_place ? pinned_alias(static_cast<double*>(s.a[kTraj].host)) : nullptr;
  if (alias) s.a[kTraj].host = nullptr;         // written in place: neither staged nor downloaded
  // every array starts on a 256-byte boundary, as an allocation of its own would
  auto room = [&](const HostArray& a) { return a.host ? (a.elem * a.rows * (size_t)n + 255) & ~(size_t)255 : 0; };
  size_t bytes = 0;
  for (const HostArray& a : s.a) bytes += room(a);
  if (bytes > h->stage_bytes) CUDA_TRY(cudaStreamSynchronize(st));   // the previous call's copies may still use it
  CUDA_TRY(grow(&h->d_stage, &h->stage_bytes, bytes));
  char* p = reinterpret_cast<char*>(h->d_stage);
  for (HostArray& a : s.a) { a.dev = a.host ? p : nullptr; p += room(a); }
  if (alias) s.a[kTraj].dev = alias;
  for (int i = 0; i < kHostInputs; ++i)
    if (s.a[i].host) CUDA_TRY(copy_columns(s, s.a[i], cudaMemcpyHostToDevice, st));
  auto dev = [&](int i) { return static_cast<double*>(s.a[i].dev); };
  const ResultOut out{dev(kTraj), dev(kTf), dev(kFinalMass), static_cast<int*>(s.a[kStatus].dev),
                      static_cast<int*>(s.a[kIters].dev), dev(kKkt), dev(kSens), (long)n, dev(kPsens)};
  return solve_batch(h, dev(kParams), dev(kGuessTraj), dev(kGuessTf), out, st, s.B);
}

// Queues the copies of the shard's outputs into the caller's arrays on st.  A copy into pageable memory returns only
// when it is done, so a caller with several devices issues every launch before the first download.
static lmato_status_t download(const HostSolve& s, cudaStream_t st) {
  for (int i = kHostInputs; i < kHostArrays; ++i)
    if (s.a[i].host) CUDA_TRY(copy_columns(s, s.a[i], cudaMemcpyDeviceToHost, st));
  return LMATO_OK;
}

lmato_status_t lmato_solve_batch_host(lmato_handle* h, const double* params, int64_t B,
                                      double* out_traj, double* out_tf, double* out_final_mass,
                                      int32_t* out_status, int32_t* out_iters, double* out_kkt) {
  lmato_status_t rc = check_batch("lmato_solve_batch_host", h, params, B, out_tf, out_final_mass, out_status, out_iters);
  if (rc != LMATO_OK || B == 0) return rc;
  CUDA_TRY(cudaSetDevice(h->device));
  if (!host_can_address(h->sens_out) || !host_can_address(h->psens_out) || !host_can_address(h->guess_traj) ||
      !host_can_address(h->guess_tf)) {
    set_err("lmato_solve_batch_host: the registered sensitivity output / start point is device memory "
            "(lmato_solve_batch_host takes HOST pointers)");
    return LMATO_ERR_INVALID;
  }
  HostSolve s = host_solve(h->nt, B, params, h->guess_traj, h->guess_tf, out_traj, h->sens_out, h->psens_out, out_tf,
                           out_final_mass, out_kkt, out_status, out_iters);
  cudaStream_t st = nullptr;
  if ((rc = stage_and_solve(h, s, 0, B, st, true)) != LMATO_OK || (rc = download(s, st)) != LMATO_OK) return rc;
  CUDA_TRY(cudaStreamSynchronize(st));
  return LMATO_OK;
}

lmato_status_t lmato_collocation_rule(int32_t nodes, double* tau, double* N) {
  colloc::Coll C;
  if (!tau || !N || !collocation_rule(nodes, &C)) { set_err("lmato_collocation_rule: NODES must be 2..6"); return LMATO_ERR_INVALID; }
  for (int i = 0; i < C.m; ++i) { tau[i] = C.tau[i]; for (int j = 0; j < C.m; ++j) N[i * C.m + j] = C.N[i][j]; }
  return LMATO_OK;
}

lmato_status_t lmato_set_initial_guess(lmato_handle* h, const double* guess_traj, const double* guess_tf) {
  if (!h) { set_err("lmato_set_initial_guess: NULL handle"); return LMATO_ERR_INVALID; }
  if ((guess_traj == nullptr) != (guess_tf == nullptr)) {
    set_err("lmato_set_initial_guess: pass both the trajectories and tf, or NULL for both");
    return LMATO_ERR_INVALID;
  }
  h->guess_traj = guess_traj; h->guess_tf = guess_tf;
  return LMATO_OK;
}

lmato_status_t lmato_set_sensitivity_output(lmato_handle* h, double* out_dtf) {
  if (!h) { set_err("lmato_set_sensitivity_output: NULL handle"); return LMATO_ERR_INVALID; }
  h->sens_out = out_dtf;
  return LMATO_OK;
}

lmato_status_t lmato_set_param_sensitivity_output(lmato_handle* h, double* out_dtf_dp) {
  if (!h) { set_err("lmato_set_param_sensitivity_output: NULL handle"); return LMATO_ERR_INVALID; }
  h->psens_out = out_dtf_dp;
  return LMATO_OK;
}

lmato_status_t lmato_coast_orbit(lmato_handle* h, const double* state, int64_t B, double gm, double dt,
                                 int64_t nsteps, double* out, void* stream) {
  if (!h || B < 0 || nsteps < 0 || !(dt > 0) || !(gm > 0)) { set_err("lmato_coast_orbit: bad argument"); return LMATO_ERR_INVALID; }
  if (B == 0) return LMATO_OK;
  if (!state || !out) { set_err("lmato_coast_orbit: NULL buffer"); return LMATO_ERR_INVALID; }
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  coast_orbit_kernel<<<(unsigned)((B + 127) / 128), 128, 0, st>>>(state, (long)B, gm, dt, (long)nsteps, out);
  CUDA_TRY(cudaGetLastError());
  h->launches += 1;
  return LMATO_OK;
}

lmato_status_t lmato_fly_control(lmato_handle* h, const double* params, int64_t B, const double* traj,
                                 const double* tf, int32_t substeps, double* out_final, double* out_traj, void* stream) {
  if (!h || B < 0 || substeps < 1) { set_err("lmato_fly_control: bad argument"); return LMATO_ERR_INVALID; }
  if (B == 0) return LMATO_OK;
  if (!params || !traj || !tf || !out_final) { set_err("lmato_fly_control: NULL buffer"); return LMATO_ERR_INVALID; }
  CUDA_TRY(cudaSetDevice(h->device));
  fly_control_kernel<<<(unsigned)((B + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      params, (long)B, h->model, h->d_tau, h->nt, traj, tf, substeps, out_final, out_traj);
  CUDA_TRY(cudaGetLastError());
  h->launches += 1;
  return LMATO_OK;
}

lmato_status_t lmato_selftest_math(lmato_handle* h, double* max_err5) {
  if (!h || !max_err5) { set_err("lmato_selftest_math: bad argument"); return LMATO_ERR_INVALID; }
  CUDA_TRY(cudaSetDevice(h->device));
  const int n = 1 << 18;
  double* d = nullptr;
  CUDA_TRY(cudaMalloc(&d, sizeof(double) * 5 * n));
  math_selftest_kernel<<<(n + 255) / 256, 256>>>(d, n);
  CUDA_TRY(cudaGetLastError());
  std::vector<double> hbuf((size_t)5 * n);
  CUDA_TRY(cudaMemcpy(hbuf.data(), d, sizeof(double) * 5 * n, cudaMemcpyDeviceToHost));
  cudaFree(d);
  h->launches += 1;
  for (int j = 0; j < 5; ++j) max_err5[j] = 0.0;
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < 5; ++j)
      if (!(hbuf[(size_t)i * 5 + j] <= max_err5[j])) max_err5[j] = hbuf[(size_t)i * 5 + j];   // NaN-propagating max
  return LMATO_OK;
}

lmato_status_t lmato_measure_fp64_peak(lmato_handle* h, double* gflops) {
  if (!h || !gflops) { set_err("lmato_measure_fp64_peak: bad argument"); return LMATO_ERR_INVALID; }
  CUDA_TRY(cudaSetDevice(h->device));
  const int blocks = h->sm_count * 8, threads = 256, iters = 20000;
  double* d = nullptr;
  CUDA_TRY(cudaMalloc(&d, sizeof(double) * (size_t)blocks * threads));
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0));
  CUDA_TRY(cudaEventCreate(&e1));
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    CUDA_TRY(cudaEventRecord(e0, 0));
    dfma_peak_kernel<<<blocks, threads>>>(d, iters);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(e1, 0));
    CUDA_TRY(cudaEventSynchronize(e1));
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
    const double fl = 2.0 * 8.0 * (double)iters * (double)blocks * threads;
    const double g = fl / (ms * 1e-3) * 1e-9;
    if (rep > 0 && g > best) best = g;
  }
  h->launches += 5;
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
  *gflops = best;
  return LMATO_OK;
}


// ---------------------------------------------------------------------------------------
// device list: one host process, several GPUs (SURVEY 8b/8e).  Problem i goes to device floor(i*G/B)
// (contiguous index ranges); every device solves its shard with its own handle, through that handle's staging
// buffer, concurrently (all launches are asynchronous), and writes its slice of the caller's HOST result arrays.  The
// problems are independent and the results land on the host, so there is no collective to own here; the
// one-process-per-GPU path with its single NCCL allgather is `sharded_solve` in the Python host layer.
// ---------------------------------------------------------------------------------------
struct lmato_multi {
  std::vector<lmato_handle*> h;
  std::vector<cudaStream_t> st;
};

lmato_status_t lmato_multi_destroy(lmato_multi* m) {
  if (!m) return LMATO_OK;
  for (size_t g = 0; g < m->h.size(); ++g) {
    if (m->h[g]) cudaSetDevice(m->h[g]->device);
    if (g < m->st.size() && m->st[g]) cudaStreamDestroy(m->st[g]);
    lmato_destroy(m->h[g]);
  }
  delete m;
  return LMATO_OK;
}

lmato_status_t lmato_multi_create(lmato_multi** out, const int32_t* devices, int32_t ndev, int32_t nt,
                                  const double* time, int32_t nodes, int32_t model) {
  if (!out) { set_err("lmato_multi_create: out is NULL"); return LMATO_ERR_INVALID; }
  *out = nullptr;
  if (!devices || ndev < 1) { set_err("lmato_multi_create: empty device list"); return LMATO_ERR_INVALID; }
  lmato_multi* m = new (std::nothrow) lmato_multi();
  if (!m) { set_err("lmato_multi_create: out of host memory"); return LMATO_ERR_INVALID; }
  m->h.assign(ndev, nullptr); m->st.assign(ndev, nullptr);
  for (int g = 0; g < ndev; ++g) {
    lmato_status_t rc = lmato_create(&m->h[g], devices[g], nt, time, nodes, model);
    if (rc == LMATO_OK && (cudaSetDevice(devices[g]) != cudaSuccess ||
                           cudaStreamCreateWithFlags(&m->st[g], cudaStreamNonBlocking) != cudaSuccess)) {
      set_err("lmato_multi_create: could not create a stream on device %s", g == 0 ? "0" : "n");
      rc = LMATO_ERR_CUDA;
    }
    if (rc != LMATO_OK) { lmato_multi_destroy(m); return rc; }
  }
  *out = m;
  return LMATO_OK;
}

lmato_status_t lmato_multi_set_options(lmato_multi* m, const lmato_options* o) {
  if (!m || !o) { set_err("lmato_multi_set_options: NULL argument"); return LMATO_ERR_INVALID; }
  for (lmato_handle* h : m->h) {
    const lmato_status_t rc = lmato_set_options(h, o);
    if (rc != LMATO_OK) return rc;
  }
  return LMATO_OK;
}

lmato_status_t lmato_multi_device_count(lmato_multi* m, int32_t* n) {
  if (!m || !n) { set_err("lmato_multi_device_count: NULL argument"); return LMATO_ERR_INVALID; }
  *n = (int32_t)m->h.size();
  return LMATO_OK;
}

lmato_status_t lmato_multi_solve_host(lmato_multi* m, const double* params, int64_t B,
                                      double* out_traj, double* out_tf, double* out_final_mass,
                                      int32_t* out_status, int32_t* out_iters, double* out_kkt) {
  lmato_status_t rc = check_batch("lmato_multi_solve_host", m, params, B, out_tf, out_final_mass, out_status, out_iters);
  if (rc != LMATO_OK || B == 0) return rc;
  const int G = (int)m->h.size();
  std::vector<HostSolve> sh(G, host_solve(m->h[0]->nt, B, params, nullptr, nullptr, out_traj, nullptr, nullptr, out_tf,
                                          out_final_mass, out_kkt, out_status, out_iters));
  // every device gets its columns and its launch before anything waits; the shards of one batch keep the batch warm
  // start even when a shard alone is small (stage_and_solve passes the whole batch's size).  Every shard is staged,
  // that of a one-device list too: on a B200 the kernel's stores into pinned memory made a one-device list 8 % faster
  // on 65 536 problems at nt = 200 but 20 % slower on 4 096 problems at nt = 2001 than the copy after the solve.
  for (int g = 0; g < G; ++g) {
    const int64_t lo = (B * g) / G, n = (B * (g + 1)) / G - lo;
    if (n == 0) continue;                      // (sh[g].n stays 0: the later loops skip it)
    CUDA_TRY(cudaSetDevice(m->h[g]->device));
    if ((rc = stage_and_solve(m->h[g], sh[g], lo, n, m->st[g], false)) != LMATO_OK) return rc;
  }
  for (int g = 0; g < G; ++g) {
    if (sh[g].n == 0) continue;
    CUDA_TRY(cudaSetDevice(m->h[g]->device));
    if ((rc = download(sh[g], m->st[g])) != LMATO_OK) return rc;
  }
  for (int g = 0; g < G; ++g) {
    if (sh[g].n == 0) continue;
    CUDA_TRY(cudaSetDevice(m->h[g]->device));
    CUDA_TRY(cudaStreamSynchronize(m->st[g]));
  }
  return LMATO_OK;
}

}  // extern "C"
