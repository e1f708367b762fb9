// Cooperative sweeps: G lanes of a warp per problem (G = 8 on the device; G = 1 is the same code run by
// one lane, which is how tests/test_device_source_on_host.py checks it on the CPU).
//
// Same NLP, same Newton system and same IPM driver (ipm_iterate_t, ascent_ipm.cuh) as the one-thread-per-
// problem sweeps of ascent_ipm_dc.cuh, organised for the regime that kernel cannot serve: batches too
// small to fill the GPU with one thread per problem (a single solve, SURVEY's configs 1-3 and 5, a
// 65 536 batch strong-scaled over 8 GPUs).  There the time is the latency of one thread walking every
// stage of every sweep.  Here
//   * everything that does not depend on the recursion is evaluated STAGE-PARALLEL: lane g of a group
//     takes stages g+1, g+1+G, ...  The trial point, its defects, merit and KKT-error terms, and the
//     model of the next Newton system (dynamics Jacobian with its structured inverse, Lagrangian
//     Hessian, condensed move cost: the "M record") are produced in one such pass per line-search
//     trial and kept, so the model is evaluated once per trial instead of once per sweep;
//   * the block-tridiagonal LDL^T (Riccati recursion) runs over the stored M records with the 8x8
//     cost-to-go distributed by rows over the group: W E^-1 is a row operation, E^-T (W E^-1) is the
//     same row operation after a transpose of the 8x8 block across the group (through shared memory),
//     and the rank-one condensation of the move needs one row broadcast;
//   * the forward substitution and the adjoint recursion for the new multipliers are 8-vector affine
//     recursions (40-70 flops per stage); every lane of the group carries them redundantly, which
//     costs nothing in SIMT time and needs no communication;
//   * fraction-to-boundary ratios, the merit slope and the right-hand sides of the adjoint recursion
//     are again stage-parallel.
// Formulation: always the 8-state one of ascent_ipm_dc.cuh, s = (y, vy, x, vx | angle, angledot, u, tf),
// control = the move v_k = u_k - u_{k-1}.  MOVE = true carries the reference's l1 move-suppression term
// (angledoubledot.DCOST, LO:99) as the slack pair (p, n); MOVE = false is the same NLP with a free move
// (dcost = 0) and also serves the circular model (coup5 = 0), so there is ONE implementation.
//
// Data layout (HBM/L2): per problem one contiguous block of per-stage records,
//   X[2][N+1][24]  iterate (ping-pong)      D[N+1][16]  step (ds, du, dv, pi)
//   M[2][N+1][52]  model at the iterate     K[N+1][10]  feedback law     H[N+1][8]  adjoint right-hand sides
// Records are 16-byte aligned and read with 128-bit loads.  A sequential phase reads one record per
// stage (the same addresses on all lanes of the group: one transaction); a stage-parallel phase reads
// G consecutive records per group.
#pragma once
#include "ascent_ipm_dc.cuh"

namespace lmato {
namespace coop {

enum : int {
  X_Z = 0, X_U = 6, X_LAM = 7 /* 7 */, X_ZLA = 14, X_ZUA = 15, X_ZLU = 16, X_ZUU = 17,
  X_PP = 18, X_PN = 19, X_ZPP = 20, X_ZPN = 21, XR = 24,
  D_DS = 0 /* ds[0..5], du */, D_DV = 7, D_PI = 8 /* 7 */, DR = 16,
  // M record: stage Jacobian with its structured inverse, defects, Hessian and gradient pieces
  J_AL = 0, J_ALA, J_ALB, J_ALC, J_ALD, J_M11, J_M13, J_M31, J_M33, J_GA1, J_GA3,
  J_E0, J_E1, J_E2, J_E3, J_E4, J_E5, J_BETA, JR = 20,
  M_J = 0, M_C = JR /* 6 defects */, M_Q = JR + 8,
  Q_00 = 0, Q_02, Q_22, Q_04, Q_24, Q_44, Q_T0 /* tf column, rows 0..6 */, Q_77 = Q_T0 + 7, Q_RU, Q_D0,
  Q_G4A, Q_G4B /* gradient of angle = A + mu*B */, Q_GUA, Q_GUB /* gradient of u */,
  Q_MVR, Q_MVA, Q_MVB /* condensed move cost: Hessian, gradient A + mu*B */, QR = 24,
  MR = M_Q + QR,
  K_FF = 8, KR = 10,
  HR = 8,
  VR = 72,                                // rows of W_k = P_k + Q_k (64) and g_k = p_k + q_k (8): see VREC below
  PER_STAGE = 2 * XR + DR + 2 * MR + KR + HR + VR,
  SCR_TR1 = 80, SCR_TR2 = 72,                                    // group scratch: the two transpose tiles of backward()
  // record ring of the sequential phases (cp.async, see rg_*): slots of backward / forward / adjoint
  RING_D = 4,                             // slots (a power of two): records travel RING_D-1 stages ahead
  RING_SB = MR,                           // backward: the whole M record
  RING_SF = M_Q + KR,                     // forward: J, c of the M record, then the feedback law
  RING_SA = JR + HR,                      // adjoint: J, then the right-hand side
  RING_DOUBLES = RING_D * RING_SB,
  SCR_DOUBLES = SCR_TR1 + SCR_TR2 + RING_DOUBLES + RING_D      // ... + one mbarrier (8 bytes) per ring slot
};
static_assert((int)X_LAM == NODE_LAM && (int)X_ZLA == NODE_ZLA && (int)X_ZUU == NODE_ZUU && (int)X_PP == NODE_PP &&
              (int)X_ZPN == NODE_ZPN && NODE_N == 22 && XR == 24, "the X record holds a start node (ascent_ipm.cuh) and two pad doubles");

// 128-bit moves of N (even) doubles
template <int N>
LM_HD void ldv(const double* __restrict__ p, double* out) {
#if defined(__CUDA_ARCH__)
#pragma unroll
  for (int i = 0; i < N; i += 2) { const double2 v = *reinterpret_cast<const double2*>(p + i); out[i] = v.x; out[i + 1] = v.y; }
#else
  for (int i = 0; i < N; ++i) out[i] = p[i];
#endif
}
template <int N>
LM_HD void stv(double* __restrict__ p, const double* in) {
#if defined(__CUDA_ARCH__)
#pragma unroll
  for (int i = 0; i < N; i += 2) *reinterpret_cast<double2*>(p + i) = make_double2(in[i], in[i + 1]);
#else
  for (int i = 0; i < N; ++i) p[i] = in[i];
#endif
}

// Group primitives.  A group = G consecutive lanes of a warp (aligned); `m` is its lane mask.
template <int G>
struct Grp {
  LM_HD static double sum(unsigned m, double v) {
#if defined(__CUDA_ARCH__)
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(m, v, o);
#endif
    return v;
  }
  LM_HD static double max(unsigned m, double v) {
#if defined(__CUDA_ARCH__)
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v = dmax(v, __shfl_xor_sync(m, v, o));
#endif
    return v;
  }
  LM_HD static double min(unsigned m, double v) {
#if defined(__CUDA_ARCH__)
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v = dmin(v, __shfl_xor_sync(m, v, o));
#endif
    return v;
  }
  LM_HD static int any(unsigned m, int v) {
#if defined(__CUDA_ARCH__)
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v |= __shfl_xor_sync(m, v, o);
#endif
    return v;
  }
  LM_HD static int bcast_int(unsigned m, int v, int src) {
#if defined(__CUDA_ARCH__)
    if (G > 1) v = __shfl_sync(m, v, src, G);
#endif
    return v;
  }
  // value of lane `src` (index inside the group) on every lane
  LM_HD static double bcast(unsigned m, double v, int src) {
#if defined(__CUDA_ARCH__)
    if (G > 1) v = __shfl_sync(m, v, src, G);
#endif
    return v;
  }
  // running maximum of num/den across the group (the pair travels; ties keep the lower lane's)
  LM_HD static void ratio_max(unsigned m, RatioMax& r) {
#if defined(__CUDA_ARCH__)
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) {
      const double n2 = __shfl_xor_sync(m, r.n, o), d2 = __shfl_xor_sync(m, r.d, o);
      if (n2 * r.d > r.n * d2) { r.n = n2; r.d = d2; }
    }
    r.n = bcast(m, r.n, 0); r.d = bcast(m, r.d, 0);
#endif
  }
  LM_HD static void sync(unsigned m) {
#if defined(__CUDA_ARCH__)
    if (G > 1) __syncwarp(m);
#endif
  }
};

// View of one problem's workspace block for one lane of its group.
// STAGE_MAJOR = false: one array per record kind ([kind][stage][record]) -- a stage-parallel phase reads GP consecutive
// records of one kind, i.e. one contiguous run per group; the layout of the throughput regime (GP = 8).
// STAGE_MAJOR = true: all records of a stage in one contiguous PER_STAGE block ([stage][kind][record]) -- a sequential
// phase walks one block (one or two DRAM pages) per stage instead of one page per record kind; the layout of the
// latency regime (a warp per problem, GP = 32).  Measured on B200: single solve 5.81 -> 5.53 ms, 1 184 problems
// 9.27 -> 8.99 ms with the stage-major layout; 4 096 x nt = 2001 at GP = 8: 242 -> 267 ms (so each regime keeps its own).
template <bool STAGE_MAJOR>
struct CwsT {
  double* base;
  int N1;                // N + 1 records per array
  double* scr;           // group scratch, SCR_DOUBLES doubles (shared memory on the device, 16-byte aligned): ring, then the tiles
  int g;                 // lane inside the group (0 .. GP-1)
  unsigned mask;         // the GP lanes of the group (stage-parallel phases, phase boundaries)
  unsigned smask;        // its first G lanes (sequential phases)
  mutable double dw;     // delta_w of the last factorisation (the adjoint recursion uses the same Hessian)
  mutable double pimax;  // largest new defect multiplier of the last adjoint recursion
  mutable int ls_flag;   // set by the driver while the least-squares multiplier estimate runs
  mutable unsigned rpar; // phase bits of the ring's mbarriers (lanes of the sequential group)
  LM_HD double* ring() const { return scr; }
  LM_HD double* tiles() const { return scr + RING_DOUBLES; }
  LM_HD double* bars() const { return scr + RING_DOUBLES + SCR_TR1 + SCR_TR2; }
  LM_HD double* X(int buf, int k) const {
    return STAGE_MAJOR ? base + (long)k * PER_STAGE + buf * XR : base + ((long)buf * N1 + k) * XR;
  }
  LM_HD double* D(int k) const {
    return STAGE_MAJOR ? base + (long)k * PER_STAGE + 2 * XR : base + (2L * N1) * XR + (long)k * DR;
  }
  LM_HD double* Mo(int buf, int k) const {
    return STAGE_MAJOR ? base + (long)k * PER_STAGE + (2 * XR + DR) + buf * MR
                       : base + (2L * N1) * XR + (long)N1 * DR + ((long)buf * N1 + k) * MR;
  }
  LM_HD double* K(int k) const {
    return STAGE_MAJOR ? base + (long)k * PER_STAGE + (2 * XR + DR + 2 * MR)
                       : base + (2L * N1) * XR + (long)N1 * DR + (2L * N1) * MR + (long)k * KR;
  }
  LM_HD double* H(int k) const {
    return STAGE_MAJOR ? base + (long)k * PER_STAGE + (2 * XR + DR + 2 * MR + KR)
                       : base + (2L * N1) * XR + (long)N1 * DR + (2L * N1) * MR + (long)N1 * KR + (long)k * HR;
  }
  LM_HD double* V(int k) const {
    return STAGE_MAJOR ? base + (long)k * PER_STAGE + (2 * XR + DR + 2 * MR + KR + HR)
                       : base + (2L * N1) * XR + (long)N1 * DR + (2L * N1) * MR + (long)N1 * (KR + HR) + (long)k * VR;
  }
};
using Cws = CwsT<false>;
template <bool STAGE_MAJOR> LM_HD int grp_lane(const CwsT<STAGE_MAJOR>& W) { return W.g; }
template <bool STAGE_MAJOR> LM_HD unsigned grp_mask(const CwsT<STAGE_MAJOR>& W) { return W.mask; }
LM_HD long coop_doubles_per_problem(int nt) { return (long)nt * PER_STAGE; }
static_assert(RING_SF <= RING_SB && RING_SA <= RING_SB, "ring too small");

// Record ring.  A sequential phase reads one small record set per stage, at addresses known in advance; without
// help each stage would start with an exposed L2/HBM round trip (~700 cycles against 100-400 cycles of
// arithmetic).  The group moves the records RING_D-1 stages ahead into its shared-memory ring.  Two back ends:
//   default          cp.async (LDGSTS): the 16-byte chunks of a record are spread over the lanes, one commit
//                    group per stage; a stage waits for its own group, then a group barrier makes every lane's
//                    chunks visible (in the backward sweep that barrier is the symmetrisation tile's).
//   LMATO_RING_BULK  cp.async.bulk.shared.global (the TMA engine; SASS UBLKCP) issued by ONE lane per record,
//                    completing on the slot's mbarrier (expect_tx / complete_tx; SASS SYNCS), on which every
//                    lane of the group waits; records written with ordinary stores in an earlier phase are
//                    published to the asynchronous proxy by a proxy fence of every writer (ring_publish()).
// The records are contiguous and 16-byte aligned, i.e. exactly what a bulk copy wants -- but they are 160-416
// bytes and on the critical path of a single warp: measured on B200 the mbarrier round trip (arrive.expect_tx,
// UBLKCP through the uniform datapath, try_wait) costs ~350 cycles per stage and phase more than four LDGSTS
// and a wait_group (single solve 5.7 -> 8.9 ms, config 5 254 -> 320 ms; a ring of 8 slots instead of 4 changes
// nothing, so it is issue/wait overhead, not uncovered latency).  Hence cp.async by default.
struct Ring {
  double* base;          // slot 0 (generic pointer; shared memory on the device)
#if defined(__CUDA_ARCH__)
  unsigned slot_s;       // shared-space byte address of slot 0
  unsigned bar_s;        // shared-space byte address of the first of RING_D mbarriers
#endif
  int g;                 // lane inside the group
};
#if defined(LMATO_RING_BULK)
constexpr bool kRingBulk = true;
#else
constexpr bool kRingBulk = false;
#endif
LM_HD void ring_publish() {
#if defined(__CUDA_ARCH__) && defined(LMATO_RING_BULK)
  asm volatile("fence.proxy.async.global;" ::: "memory");
#endif
}
LM_HD Ring ring_of(double* base, double* bars, int g) {
  Ring r;
  r.base = base; r.g = g;
#if defined(__CUDA_ARCH__)
  r.slot_s = (unsigned)__cvta_generic_to_shared(base);
  r.bar_s = (unsigned)__cvta_generic_to_shared(bars);
#else
  (void)bars;
#endif
  return r;
}
// once per kernel, by one lane of the group (followed by a CTA barrier)
LM_HD void ring_init_barriers(double* bars) {
#if defined(__CUDA_ARCH__) && defined(LMATO_RING_BULK)
  const unsigned b = (unsigned)__cvta_generic_to_shared(bars);
#pragma unroll
  for (int i = 0; i < RING_D; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(b + 8u * i), "r"(1u) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#else
  (void)bars;
#endif
}
// Fill slot `slot` (stride SLOT doubles) with record A (NA doubles) followed by record B (NB doubles, may be 0);
// valid = false: the stage does not exist (the commit group is still closed, so that groups and stages stay in step).
template <int G, int SLOT, int NA, int NB>
LM_HD void ring_issue(const Ring& r, int slot, const double* a, const double* b, bool valid) {
#if defined(__CUDA_ARCH__)
#if defined(LMATO_RING_BULK)
  if (!valid || r.g != 0) return;
  const unsigned bar = r.bar_s + 8u * (unsigned)slot;
  const unsigned dst = r.slot_s + 8u * (unsigned)(slot * SLOT);
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(8u * (NA + NB)) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(a), "r"(8u * NA), "r"(bar) : "memory");
  if (NB > 0)
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst + 8u * NA), "l"(b), "r"(8u * NB), "r"(bar) : "memory");
#else
  if (valid) {
    const unsigned dst = r.slot_s + 8u * (unsigned)(slot * SLOT) + 16u * (unsigned)r.g;
#pragma unroll
    for (int c = 0; c < (NA / 2 + G - 1) / G; ++c)
      if (c * G + r.g < NA / 2)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16u * (unsigned)(c * G)), "l"(a + 2 * (c * G + r.g)) : "memory");
#pragma unroll
    for (int c = 0; c < (NB / 2 + G - 1) / G; ++c)
      if (c * G + r.g < NB / 2)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 8u * NA + 16u * (unsigned)(c * G)), "l"(b + 2 * (c * G + r.g)) : "memory");
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
#endif
#else
  if (valid && r.g == 0) {
    double* d = r.base + slot * SLOT;
    for (int i = 0; i < NA; ++i) d[i] = a[i];
    for (int i = 0; i < NB; ++i) d[NA + i] = b[i];
  }
#endif
}
// The copies of slot `slot` have landed.  cp.async: all but the PENDING newest commit groups of this lane are
// complete (the caller's next group barrier makes the other lanes' chunks visible); bulk: the slot's mbarrier
// phase is complete (`par` holds one phase bit per slot).
template <int PENDING>
LM_HD void ring_wait(const Ring& r, int slot, unsigned& par, bool valid) {
#if defined(__CUDA_ARCH__)
#if defined(LMATO_RING_BULK)
  if (!valid) return;
  const unsigned bar = r.bar_s + 8u * (unsigned)slot;
  const unsigned ph = (par >> slot) & 1u;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "RW%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra RD%=;\n\t"
      "bra RW%=;\n\t"
      "RD%=:\n\t"
      "}" ::"r"(bar), "r"(ph) : "memory");
  par ^= 1u << slot;
#else
  asm volatile("cp.async.wait_group %0;" ::"n"(PENDING) : "memory");
  (void)slot; (void)par; (void)valid; (void)r;
#endif
#else
  (void)r; (void)slot; (void)par; (void)valid;
#endif
}
// hint: bring the 128-byte lines of a record that a later stage of a stage-parallel loop will read into L2/L1
template <int NDBL>
LM_HD void prefetch_rec(const double* p) {
#if defined(__CUDA_ARCH__) && defined(LMATO_COOP_PREFETCH)
#pragma unroll
  for (int i = 0; i < NDBL; i += 16) asm volatile("prefetch.global.L1 [%0];" ::"l"(p + i));
#endif
}

LM_HD void jac_load(const double* m, StageJac& J) {
  double j[JR];
  ldv<JR>(m + M_J, j);
  J.al = j[J_AL]; J.ala = j[J_ALA]; J.alb = j[J_ALB]; J.alc = j[J_ALC]; J.ald = j[J_ALD];
  J.m11 = j[J_M11]; J.m13 = j[J_M13]; J.m31 = j[J_M31]; J.m33 = j[J_M33];
  J.ga1 = j[J_GA1]; J.ga3 = j[J_GA3];
  J.e0 = j[J_E0]; J.e1 = j[J_E1]; J.e2 = j[J_E2]; J.e3 = j[J_E3]; J.e4 = j[J_E4]; J.e5 = j[J_E5];
  J.beta = j[J_BETA];
}

// MOVE as a template argument of the sweeps: 0 no move term (u is free per stage), 1 the move term on the MV
// angledoubledot (LO:99), 2 the move term of the circular model, where the MV slot IS the pitch angle (mv_is_angle()).
// E^{-1} v and E^{-T} g of the 8-state stage Jacobian (dc::solveE8 / dc::solveET8); MVA: with the extra entry
// d defect_4 / d u = -1 of that last case (angle_k - u_k = 0), a compile-time flag so that it costs the other
// cases nothing on their dependency chains.
template <bool MVA>
LM_HD void solveE8x(const StageJac& J, double* v) {
  const double v7 = v[7], v6 = v[6];
  const double v5 = v[5] + J.beta * v6 + J.e5 * v7;
  const double v4 = (MVA ? v[4] + v6 : v[4]) + J.al * v5 + J.e4 * v7;
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
template <bool MVA>
LM_HD void solveET8x(const StageJac& J, double* g) {
  double w0 = g[0], w1 = g[1], w2 = g[2], w3 = g[3];
  applyA11T(J, w0, w1, w2, w3);
  const double gaw = J.ga1 * w1 + J.ga3 * w3;
  const double gew = J.e0 * w0 + J.e1 * w1 + J.e2 * w2 + J.e3 * w3;
  const double w4 = g[4] + gaw;
  const double w5 = g[5] + J.al * w4;
  const double w6 = (MVA ? g[6] + w4 : g[6]) + J.beta * w5;
  const double w7 = g[7] + gew + J.e4 * w4 + J.e5 * w5;
  g[0] = w0; g[1] = w1; g[2] = w2; g[3] = w3; g[4] = w4; g[5] = w5; g[6] = w6; g[7] = w7;
}

// ---------------------------------------------------------------------------------------
// Model of the Newton system at one stage of one point -> M record.  Gradient pieces that depend
// on the barrier parameter are kept as (A, B) with value A + mu*B, and delta_w is added by the
// consumers, so a record stays valid when mu or delta_w change.  ls: the least-squares multiplier
// estimate of IPOPT section 3.6 (Hessian := I, gradient := grad f - zL + zU), as in stage_hessian().
// ---------------------------------------------------------------------------------------
template <int MOVE>
LM_HD void build_stage(const Params& P, const Options& O, double kap, double taum, double tf, bool ls,
                       const double* z, double u, const double* zp, double up, const double* lam,
                       double zla, double zua, double zlu, double zuu,
                       double pp, double pn, double zpp, double zpn, double* mrec) {
  Accel1 f;
  accel_first(P, z[0], z[2], z[4], taum * tf, f);
  StageJac J;
  stagejac_build(P, kap, tf, taum, f, z[1], z[3], z[5], u, J);
  stagejac_invert(J);
  double j[JR];
  j[J_AL] = J.al; j[J_ALA] = J.ala; j[J_ALB] = J.alb; j[J_ALC] = J.alc; j[J_ALD] = J.ald;
  j[J_M11] = J.m11; j[J_M13] = J.m13; j[J_M31] = J.m31; j[J_M33] = J.m33;
  j[J_GA1] = J.ga1; j[J_GA3] = J.ga3;
  j[J_E0] = J.e0; j[J_E1] = J.e1; j[J_E2] = J.e2; j[J_E3] = J.e3; j[J_E4] = J.e4; j[J_E5] = J.e5;
  j[J_BETA] = J.beta; j[18] = 0.0; j[19] = 0.0;
  stv<JR>(mrec + M_J, j);
  const double al = J.al;
  double c[8];
  c[0] = z[0] - zp[0] - al * z[1];
  c[1] = z[1] - zp[1] - al * f.ay;
  c[2] = z[2] - zp[2] - al * z[3];
  c[3] = z[3] - zp[3] - al * f.ax;
  c[4] = (MOVE == 2) ? z[4] - u - al * z[5]                  // the MV slot is the angle: angle_k - u_k = 0 (angledot = 0)
                     : z[4] - zp[4] - al * z[5];
  c[5] = z[5] - ((MOVE == 1) ? zp[5] : (MOVE == 2) ? 0.0 : P.coup5 * zp[5]) - J.beta * u;
  c[6] = 0.0; c[7] = 0.0;
  stv<8>(mrec + M_C, c);
  StageQ q;
  stage_hessian(P, f, J, kap, taum, lam, z[4], u, zla, zua, zlu, zuu, 1.0, 0.0, ls, q);
  double o[QR];
  o[Q_00] = q.q00; o[Q_02] = q.q02; o[Q_22] = q.q22; o[Q_04] = q.q04; o[Q_24] = q.q24; o[Q_44] = q.q44;
  o[Q_T0 + 0] = q.q06; o[Q_T0 + 1] = q.q16; o[Q_T0 + 2] = q.q26; o[Q_T0 + 3] = q.q36;
  o[Q_T0 + 4] = q.q46; o[Q_T0 + 5] = q.q56; o[Q_T0 + 6] = q.sig;
  o[Q_77] = q.q66; o[Q_RU] = q.R; o[Q_D0] = q.d;
  o[Q_G4A] = ls ? q.q4 : 0.0; o[Q_G4B] = ls ? 0.0 : q.q4;
  o[Q_GUA] = ls ? q.r : 0.0;  o[Q_GUB] = ls ? 0.0 : q.r;
  if (MOVE) {
    dc::Move mv;
    mv.build(pp, pn, zpp, zpn, u - up, O.w_dcost, 0.0, ls);
    o[Q_MVR] = mv.R; o[Q_MVA] = mv.r;
    o[Q_MVB] = ls ? 0.0 : -(mv.ip * mv.Sn - mv.in_ * mv.Sp) * mv.sinv;
  } else {
    o[Q_MVR] = 0.0; o[Q_MVA] = 0.0; o[Q_MVB] = 0.0;
  }
  o[QR - 1] = 0.0;
  stv<QR>(mrec + M_Q, o);
}

// (re)build the M records of buffer `buf` from its X records (start point; least-squares phase)
template <int GP, int MOVE, class CW>
LM_SWEEP void coop_build(const Params& P, const Mesh& M, const Options& O, const CW& W, int buf, double tf, bool ls) {
  const int N = M.N;
  for (int k = 1 + W.g; k <= N; k += GP) {
    double x[XR], xm[8];
    ldv<XR>(W.X(buf, k), x);
    ldv<8>(W.X(buf, k - 1), xm);
    build_stage<MOVE>(P, O, M.h[k] * P.T, P.mT * M.tau[k], tf, ls, x + X_Z, x[X_U], xm + X_Z, xm[X_U], x + X_LAM,
                      x[X_ZLA], x[X_ZUA], x[X_ZLU], x[X_ZUU], x[X_PP], x[X_PN], x[X_ZPP], x[X_ZPN], W.Mo(buf, k));
  }
  ring_publish();
  Grp<GP>::sync(W.mask);
}

// ---------------------------------------------------------------------------------------
// backward sweep: block LDL^T of the KKT matrix in stage order over the stored M records.
// Lane g owns rows g*R .. g*R+R-1 of the 8x8 cost-to-go and the same elements of its affine part
// (R = 8/G).  Per stage
//   W = P_k + Q_k,  g = p_k + q_k
//   X = W E^-1                      row operation on the owned rows
//   transpose [X | g] across the group (shared-memory tile), g becomes known to every lane
//   Wt = X^T E^-1 (= E^-T W E^-1),  g~ = E^-T g
//   symmetrise Wt through a second tile: 0.5 (Wt + Wt^T).  This is not cosmetic: with barrier terms
//   Sigma ~ 1e13 on the diagonal, entries (i,j) and (j,i) computed by different lanes differ by ~1e-3
//   absolute, and un-symmetrised the recursion loses Newton's quadratic convergence near the solution
//   (measured on the host build: 33-35 instead of 28-32 iterations, inertia corrections appear)
//   condense the move (row / column 6, read from the same tile), P_{k-1} = D (Wt - ...) D
// identical, up to rounding, to dc::riccati_backward.  Returns false on wrong inertia.
// ---------------------------------------------------------------------------------------
// VREC: also keep W_k = P_k + Q_k and g_k = p_k + q_k of every stage (72 doubles).  The new multipliers are then
// pi_k = -E_k^-T (W_k ds_k + g_k)  -- a stage-parallel product in forward() -- instead of the sequential adjoint
// recursion: one of the three sequential sweeps per iteration disappears, for 1.1 KB more traffic per stage.
// Used where the sequential sweeps are the critical path (a warp per problem), not where HBM traffic counts.
template <int G, int MOVE, bool VREC, class CW>
LM_SWEEP bool coop_backward_seq(const Params& P, const Mesh& M, const Options& O, const CW& W, int src,
                                const Scal& c0, double mu, double dw, bool ls, double* dtf_out) {
  constexpr int R = 8 / G;
  const int N = M.N;
  const int g = W.g;
  const unsigned gm = W.smask;
  double Pr[R][8], pr[R];
  {
    double zn[8];
    ldv<8>(W.X(src, N), zn);
    TermQP tq;
    terminal_qp(P, O, c0, zn, mu, dw, ls, tq);
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int i = g * R + r;
#pragma unroll
      for (int j = 0; j < 8; ++j) Pr[r][j] = 0.0;
      pr[r] = 0.0;
#pragma unroll
      for (int ii = 0; ii < 4; ++ii)
        if (i == ii) {
#pragma unroll
          for (int j = 0; j < 4; ++j) Pr[r][j] = tq.H[ii][j];
          pr[r] = tq.g[ii];
        }
      if (i == 7) { Pr[r][7] = tq.H66; pr[r] = tq.g6; }
    }
  }
  const double cw = ls ? 0.0 : 1.0;     // defects are dropped in the least-squares mode
  const double cp = (MOVE == 1) ? 1.0 : (MOVE == 2) ? 0.0 : P.coup5, cq4 = (MOVE == 2) ? 0.0 : 1.0;   // (compile-time with the move term)
  double rmask[R][8], rscale[R];        // rmask[r][j] = 1 if this lane's r-th row is row j;  D = diag(1,1,1,1,cq4,coup5,1,1)
#pragma unroll
  for (int r = 0; r < R; ++r) {
#pragma unroll
    for (int j = 0; j < 8; ++j) rmask[r][j] = (g * R + r == j) ? 1.0 : 0.0;
    rscale[r] = (g * R + r == 5) ? cp : (g * R + r == 4) ? cq4 : 1.0;
  }
  double* tr1 = W.tiles();              // 8 x 10: X rows with the affine part as ninth column
  double* tr2 = W.tiles() + SCR_TR1;    // 8 x 9 : Wt rows
  bool ok = true;
  double* ring = W.ring();
  const Ring rg = ring_of(ring, W.bars(), g);
  unsigned par = W.rpar;
  int ki = N, kw = N;                          // next stage to issue / to wait for (descending)
#pragma unroll
  for (int d = 0; d < RING_D - 1; ++d) {
    ring_issue<G, RING_SB, MR, 0>(rg, ki & (RING_D - 1), W.Mo(src, ki), nullptr, ki >= 1);
    --ki;
  }
  ring_wait<RING_D - 2>(rg, kw & (RING_D - 1), par, true); --kw;   // stage N has landed
  if (!kRingBulk) Grp<G>::sync(gm);
  for (int k = N; k >= 1; --k) {
    ring_issue<G, RING_SB, MR, 0>(rg, ki & (RING_D - 1), W.Mo(src, ki), nullptr, ki >= 1);
    --ki;
    const double* m = ring + (k & (RING_D - 1)) * RING_SB;
    StageJac J;
    jac_load(m, J);
    double c[8], q[QR];
    ldv<8>(m + M_C, c);
    ldv<QR>(m + M_Q, q);
    const double dd = q[Q_D0] + dw;
    // ---- W = Q_k + P_k (owned rows), g = q_k + p_k ----
    // Row i of the sparse Q_k is assembled with the lane's 0/1 row masks and FMAs: lane-dependent ternaries were
    // compiled to divergent branches here (BSSY/BSYNC around partially active bodies, 11 % of the loop's stall
    // samples on a single solve); masked FMAs are straight-line code on a pipe that is idle in this regime.
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const double* mk = rmask[r];
      const double q00 = q[Q_00] + dw, q22 = q[Q_22] + dw, q44 = q[Q_44] + dw, qru = q[Q_RU] + dw;
      Pr[r][0] += mk[0] * q00 + mk[2] * q[Q_02] + (mk[4] * q[Q_04] + mk[7] * q[Q_T0 + 0]);
      Pr[r][2] += mk[0] * q[Q_02] + mk[2] * q22 + (mk[4] * q[Q_24] + mk[7] * q[Q_T0 + 2]);
      Pr[r][4] += mk[0] * q[Q_04] + mk[2] * q[Q_24] + (mk[4] * q44 + mk[7] * q[Q_T0 + 4]);
      Pr[r][1] += mk[1] * dd + mk[7] * q[Q_T0 + 1];
      Pr[r][3] += mk[3] * dd + mk[7] * q[Q_T0 + 3];
      Pr[r][5] += mk[5] * dd + mk[7] * q[Q_T0 + 5];
      Pr[r][6] += mk[6] * qru + mk[7] * q[Q_T0 + 6];
      Pr[r][7] += (mk[0] * q[Q_T0 + 0] + mk[1] * q[Q_T0 + 1]) + (mk[2] * q[Q_T0 + 2] + mk[3] * q[Q_T0 + 3]) +
                  ((mk[4] * q[Q_T0 + 4] + mk[5] * q[Q_T0 + 5]) + (mk[6] * q[Q_T0 + 6] + mk[7] * q[Q_77]));
      pr[r] += mk[4] * (q[Q_G4A] + mu * q[Q_G4B]) + mk[6] * (q[Q_GUA] + mu * q[Q_GUB]);
    }
    if (VREC) {
      double* v = W.V(k);
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const int i = g * R + r;
        stv<8>(v + 8 * i, Pr[r]);
        v[64 + i] = pr[r];
      }
    }
    // ---- X = W E^-1 (row operation), transpose [X | g] across the group ----
#pragma unroll
    for (int r = 0; r < R; ++r) solveET8x<(MOVE == 2)>(J, Pr[r]);
    double gt[8];
    if (G > 1) {
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const int i = g * R + r;
#pragma unroll
        for (int j = 0; j < 8; ++j) tr1[i * 10 + j] = Pr[r][j];
        tr1[i * 10 + 8] = pr[r];
      }
      Grp<G>::sync(gm);
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const int i = g * R + r;
#pragma unroll
        for (int j = 0; j < 8; ++j) Pr[r][j] = tr1[j * 10 + i];
      }
#pragma unroll
      for (int l = 0; l < 8; ++l) gt[l] = tr1[l * 10 + 8];
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        gt[i] = pr[i % R];
#pragma unroll
        for (int j = 0; j < i; ++j) { const double t = Pr[i % R][j]; Pr[i % R][j] = Pr[j % R][i]; Pr[j % R][i] = t; }
      }
    }
    // ---- Wt = X^T E^-1,  g~ = E^-T g (every lane) ----
#pragma unroll
    for (int r = 0; r < R; ++r) solveET8x<(MOVE == 2)>(J, Pr[r]);
    solveET8x<(MOVE == 2)>(J, gt);
    // ---- symmetrise; row 6 (= column 6) of Wt to every lane ----
    double w6[8];
    if (G > 1) {
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const int i = g * R + r;
#pragma unroll
        for (int j = 0; j < 8; ++j) tr2[i * 9 + j] = Pr[r][j];
      }
      ring_wait<RING_D - 2>(rg, kw & (RING_D - 1), par, kw >= 1);   // the next stage's record has landed ...
      --kw;
      Grp<G>::sync(gm);                                              // ... and is visible to every lane
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const int i = g * R + r;
#pragma unroll
        for (int j = 0; j < 8; ++j) Pr[r][j] = 0.5 * (Pr[r][j] + tr2[j * 9 + i]);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) w6[j] = tr2[6 * 9 + j] + tr2[j * 9 + 6];     // TWICE row 6: the halves are folded in below
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < i; ++j) { const double v = 0.5 * (Pr[i % R][j] + Pr[j % R][i]); Pr[i % R][j] = v; Pr[j % R][i] = v; }
#pragma unroll
      for (int j = 0; j < 8; ++j) w6[j] = 2.0 * Pr[6 % R][j];
      ring_wait<RING_D - 2>(rg, kw & (RING_D - 1), par, kw >= 1);
      --kw;
    }
    // ---- condense the move: it enters the u row (index 6) with coefficient 1 ----
    double wc6 = 0.0;
#pragma unroll
    for (int j = 0; j < 6; ++j) wc6 = fma(w6[j], c[j], wc6);
    const double rx6 = gt[6] - (0.5 * cw) * wc6;                  // (w6 holds twice the symmetrised row 6)
    const double Ruu = q[Q_MVR] + (MOVE && !ls ? dw : 0.0) + 0.5 * w6[6];
    const double ru = q[Q_MVA] + mu * q[Q_MVB] + rx6;
    if (!(Ruu > 0.0) || !(Ruu < 1e300)) ok = false;
    const double Rinv = lm_rcp(Ruu);
    w6[5] *= cp; if (MOVE == 2) w6[4] = 0.0;            // d defect_k / d s_{k-1} = -D, D = diag(1,1,1,1,cq4,coup5,1,1)
    // the feedback law K_k = -w6 / Ruu, k_k = -ru / Ruu, computed with its sign: it is what gets stored, and the
    // update below subtracts w6_i * w6 / Ruu = adds w6_i * K (no separate negations in the one-lane store branch)
    const double nRinv = -Rinv, nhRinv = -0.5 * Rinv;
    double w6n[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) w6n[j] = w6[j] * nhRinv;
    const double kffn = ru * nRinv;
    if (g == 6 / R) {
      double kk[KR];
#pragma unroll
      for (int j = 0; j < 8; ++j) kk[j] = w6n[j];
      kk[K_FF] = kffn; kk[9] = 0.0;
      stv<KR>(W.K(k), kk);
    }
    // ---- P_{k-1} = D Wt D - (D w6)(D w6)^T / Ruu ,  p_{k-1} = D (g~ - Wt c) - D w6 ru / Ruu ----
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const double* mk = rmask[r];
      double wc = 0.0;
#pragma unroll
      for (int j = 0; j < 6; ++j) wc = fma(Pr[r][j], c[j], wc);
      const double gti = (mk[0] * gt[0] + mk[1] * gt[1]) + (mk[2] * gt[2] + mk[3] * gt[3]) +
                         ((mk[4] * gt[4] + mk[5] * gt[5]) + (mk[6] * gt[6] + mk[7] * gt[7]));
      const double rs = rscale[r];
      const double w6i = rs * Pr[r][6];
      Pr[r][5] *= cp; if (MOVE == 2) Pr[r][4] = 0.0;
#pragma unroll
      for (int j = 0; j < 8; ++j) Pr[r][j] = fma(w6i, w6n[j], rs * Pr[r][j]);
      pr[r] = fma(w6i, kffn, rs * (gti - cw * wc));
    }
    if (!ok) {
      // wrong inertia: leave with the ring drained (every issued copy waited for), the caller retries with delta_w
      if (kRingBulk) while (kw > ki && kw >= 1) { ring_wait<0>(rg, kw & (RING_D - 1), par, true); --kw; }
      W.rpar = par;
      ring_publish();
      return false;
    }
  }
  W.rpar = par;
  ring_publish();                              // K (and the kept rows) are read through the ring / by other lanes next
  // node 0: everything pinned except tf
  const double P77 = Grp<G>::bcast(gm, Pr[7 % R][7], 7 / R);
  const double p7 = Grp<G>::bcast(gm, pr[7 % R], 7 / R);
  if (!(P77 > 0.0)) return false;
  *dtf_out = -p7 / P77;
  return true;
}

// the G lanes of the sequential group factorise; the result goes to all GP lanes of the group
template <int G, int GP, int MOVE, bool VREC, class CW>
LM_SWEEP bool coop_backward(const Params& P, const Mesh& M, const Options& O, const CW& W, int src,
                            const Scal& c0, double mu, double dw, bool ls, double* dtf_out) {
  W.dw = dw;
  double dtf = 0.0;
  int ok = 0;
  if (W.g < G) ok = coop_backward_seq<G, MOVE, VREC>(P, M, O, W, src, c0, mu, dw, ls, &dtf) ? 1 : 0;
  Grp<GP>::sync(W.mask);                     // the feedback law K is read by forward()
  if (GP > G) { ok = Grp<GP>::bcast_int(W.mask, ok, 0); dtf = Grp<GP>::bcast(W.mask, dtf, 0); }
  *dtf_out = dtf;
  return ok != 0;
}

// ---------------------------------------------------------------------------------------
// forward sweep: (1) primal Newton step, an 8-vector recursion carried redundantly by every lane;
// (2) stage-parallel: steps of the move slack pair and of the bound multipliers, fraction-to-boundary
// ratios, merit slope, and the right-hand sides Q_k ds_k + q_k of the adjoint recursion; (3) the adjoint
// recursion E_k^T pi_k = D pi_{k+1} - (Q_k ds_k + q_k) for the new defect multipliers.
// ---------------------------------------------------------------------------------------
template <int G, int GP, int MOVE, bool VREC, class CW>
LM_SWEEP void coop_forward(const Params& P, const Mesh& M, const Options& O, const CW& W, int src,
                           const Scal& c0, double mu, double tau, double dtf, bool ls, TermStep& ts, StepInfo& si) {
  const int N = M.N;
  const int g = W.g;
  const unsigned gm = W.smask;       // sequential group
  const unsigned pmk = W.mask;       // parallel group
  const double cw = ls ? 0.0 : 1.0;
  const double cp = (MOVE == 1) ? 1.0 : (MOVE == 2) ? 0.0 : P.coup5, cq4 = (MOVE == 2) ? 0.0 : 1.0;   // (compile-time with the move term)
  const double dw = W.dw;
  const double wdc = O.w_dcost;
  // ---- (1) ds_k = E_k^-1 (D ds_{k-1} + e_6 dv_k - c_k),  dv_k = k_k + K_k ds_{k-1} ----
  double ds[8] = {0, 0, 0, 0, 0, 0, 0, dtf};
  double* ring = W.ring();
  const Ring rg = ring_of(ring, W.bars(), g);
  unsigned par = W.rpar;
  if (g < G) {
    int ki = 1;
#pragma unroll
    for (int d = 0; d < RING_D - 1; ++d) {
      ring_issue<G, RING_SF, M_Q, KR>(rg, ki & (RING_D - 1), W.Mo(src, ki), W.K(ki), ki <= N);
      ++ki;
    }
    for (int k = 1; k <= N; ++k) {
      if (kRingBulk) Grp<G>::sync(gm);         // every lane is done with the slot that is re-filled now
      ring_issue<G, RING_SF, M_Q, KR>(rg, ki & (RING_D - 1), W.Mo(src, ki), W.K(ki), ki <= N);
      ++ki;
      ring_wait<RING_D - 1>(rg, k & (RING_D - 1), par, true);
      if (!kRingBulk) Grp<G>::sync(gm);        // the other lanes' chunks
      const double* m = ring + (k & (RING_D - 1)) * RING_SF;
      StageJac J;
      jac_load(m, J);
      double c[8], kk[KR];
      ldv<8>(m + M_C, c);
      ldv<KR>(m + M_Q, kk);
    // (a tree, not a chain: the move heads the stage's dependency chain)
    const double dv = ((kk[0] * ds[0] + kk[1] * ds[1]) + (kk[2] * ds[2] + kk[3] * ds[3])) +
                      ((kk[4] * ds[4] + kk[5] * ds[5]) + (kk[6] * ds[6] + fma(kk[7], ds[7], kk[K_FF])));
    double xi[8];
#pragma unroll
    for (int i = 0; i < 4; ++i) xi[i] = ds[i] - cw * c[i];
    xi[4] = (MOVE == 2 ? 0.0 : ds[4]) - cw * c[4];
    xi[5] = cp * ds[5] - cw * c[5];
    xi[6] = ds[6] + dv;
    xi[7] = dtf;
    solveE8x<(MOVE == 2)>(J, xi);
#pragma unroll
    for (int i = 0; i < 7; ++i) ds[i] = xi[i];
      if (g == 0) {
        double o[8];
#pragma unroll
        for (int i = 0; i < 7; ++i) o[i] = ds[i];
        o[D_DV] = dv;
        stv<8>(W.D(k) + D_DS, o);
      }
    }
  }
  Grp<GP>::sync(pmk);
  // ---- (2) stage-parallel ----
  double dphi = 0.0, dxmax = 0.0, pimax_par = 0.0;
  RatioMax rp, rz;
  rp.init(); rz.init();
  TermQP tq;
  if (!VREC && ((N - 1) % GP) == g) {
    double zn[8];
    ldv<8>(W.X(src, N), zn);
    terminal_qp(P, O, c0, zn, mu, dw, ls, tq);
  }
  for (int k = 1 + g; k <= N; k += GP) {
    if (k + GP <= N) { prefetch_rec<XR>(W.X(src, k + GP)); prefetch_rec<8>(W.D(k + GP)); prefetch_rec<QR>(W.Mo(src, k + GP) + M_Q); }
    double x[XR], d[8], q[QR];
    ldv<XR>(W.X(src, k), x);
    ldv<8>(W.D(k), d);
    ldv<QR>(W.Mo(src, k) + M_Q, q);
    const double u = x[X_U], du = d[6], da = d[4], dv = d[D_DV];
    if (MOVE) {
      const double up = W.X(src, k - 1)[X_U];
      dc::Move mv;
      mv.build(x[X_PP], x[X_PN], x[X_ZPP], x[X_ZPN], u - up, wdc, mu, ls);
      double dp, dn;
      mv.steps(dv, dp, dn);
      const double ip = mv.ip, in_ = mv.in_;
      rp.push(-dp, x[X_PP]); rp.push(-dn, x[X_PN]);
      rz.push(-((mu - x[X_ZPP] * dp) * ip - x[X_ZPP]), x[X_ZPP]);
      rz.push(-((mu - x[X_ZPN] * dn) * in_ - x[X_ZPN]), x[X_ZPN]);
      dphi += (wdc - mu * ip) * dp + (wdc - mu * in_) * dn;
      dxmax = dmax(dxmax, dmax(fabs(dp), fabs(dn)) * dmin(1.0, dmax(ip, in_)));
    }
#pragma unroll
    for (int i = 0; i < 7; ++i) dxmax = dmax(dxmax, fabs(d[i]));
    const double a = x[X_Z + 4];
    const double dLa = a, dUa = P.a_ub - a, dLu = u + P.u_ub, dUu = P.u_ub - u;
    rp.push(-da, dLa); rp.push(da, dUa); rp.push(-du, dLu); rp.push(du, dUu);
    const double zla = x[X_ZLA], zua = x[X_ZUA], zlu = x[X_ZLU], zuu = x[X_ZUU];
    double rLa, rUa, rLu, rUu;
    recip4(dLa, dUa, dLu, dUu, rLa, rUa, rLu, rUu);
    rz.push(-((mu - zla * da) * rLa - zla), zla);
    rz.push(-((mu + zua * da) * rUa - zua), zua);
    rz.push(-((mu - zlu * du) * rLu - zlu), zlu);
    rz.push(-((mu + zuu * du) * rUu - zuu), zuu);
    dphi += mu * ((rUa - rLa) * da + (rUu - rLu) * du);
    if (VREC) {
      // new multipliers of this stage from the kept rows: pi_k = -E_k^-T (W_k ds_k + g_k)
      double v[VR], gg[8];
      ldv<VR>(W.V(k), v);
#pragma unroll
      for (int i = 0; i < 7; ++i) {
        double t = fma(v[8 * i + 7], dtf, v[64 + i]);
#pragma unroll
        for (int j = 0; j < 7; ++j) t = fma(v[8 * i + j], d[j], t);
        gg[i] = -t;
      }
      gg[7] = 0.0;
      StageJac J;
      jac_load(W.Mo(src, k), J);
      solveET8x<(MOVE == 2)>(J, gg);
      gg[7] = 0.0;
      stv<8>(W.D(k) + D_PI, gg);
      if (ls) {
#pragma unroll
        for (int i = 0; i < 7; ++i) pimax_par = dmax(pimax_par, fabs(gg[i]));
      }
    } else {
    // right-hand side of the adjoint recursion (same Hessian as the factorisation, delta_w included)
    const double dd = q[Q_D0] + dw;
    double h[8];
    h[0] = (q[Q_00] + dw) * d[0] + q[Q_02] * d[2] + q[Q_04] * d[4] + q[Q_T0 + 0] * dtf;
    h[1] = dd * d[1] + q[Q_T0 + 1] * dtf;
    h[2] = q[Q_02] * d[0] + (q[Q_22] + dw) * d[2] + q[Q_24] * d[4] + q[Q_T0 + 2] * dtf;
    h[3] = dd * d[3] + q[Q_T0 + 3] * dtf;
    h[4] = q[Q_04] * d[0] + q[Q_24] * d[2] + (q[Q_44] + dw) * d[4] + q[Q_T0 + 4] * dtf + q[Q_G4A] + mu * q[Q_G4B];
    h[5] = dd * d[5] + q[Q_T0 + 5] * dtf;
    h[6] = (q[Q_RU] + dw) * du + q[Q_T0 + 6] * dtf + q[Q_GUA] + mu * q[Q_GUB];
    h[7] = 0.0;
    if (k == N) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        h[i] += tq.H[i][0] * d[0] + tq.H[i][1] * d[1] + tq.H[i][2] * d[2] + tq.H[i][3] * d[3] + tq.g[i];
    }
    stv<HR>(W.H(k), h);
    }
  }
  dphi = Grp<GP>::sum(pmk, dphi);
  dxmax = dmax(Grp<GP>::max(pmk, dxmax), fabs(dtf));
  Grp<GP>::ratio_max(pmk, rp);
  Grp<GP>::ratio_max(pmk, rz);
  // ---- terminal slacks and multipliers (every lane) ----
  {
    double zm[8];
    ldv<8>(W.X(src, N), zm);
    ldv<8>(W.D(N), ds);                  // the step of the last node (lanes outside the sequential group did not carry it)
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
  ring_publish();                              // the H records travel through the ring next
  Grp<GP>::sync(pmk);
  // ---- (3) adjoint recursion, every lane of the sequential group ----
  double pin[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  double pimax = 0.0;
  if (VREC) {
    W.rpar = par;
    W.pimax = Grp<GP>::max(pmk, pimax_par);
    return;
  }
  if (g < G) {
  int ki = N;
#pragma unroll
  for (int d = 0; d < RING_D - 1; ++d) {
    ring_issue<G, RING_SA, JR, HR>(rg, ki & (RING_D - 1), W.Mo(src, ki), W.H(ki), ki >= 1);
    --ki;
  }
  for (int k = N; k >= 1; --k) {
    if (kRingBulk) Grp<G>::sync(gm);
    ring_issue<G, RING_SA, JR, HR>(rg, ki & (RING_D - 1), W.Mo(src, ki), W.H(ki), ki >= 1);
    --ki;
    ring_wait<RING_D - 1>(rg, k & (RING_D - 1), par, true);
    if (!kRingBulk) Grp<G>::sync(gm);
    const double* m = ring + (k & (RING_D - 1)) * RING_SA;
    StageJac J;
    jac_load(m, J);
    double h[HR], gg[8];
    ldv<HR>(m + JR, h);
#pragma unroll
    for (int i = 0; i < 7; ++i) gg[i] = pin[i] - h[i];
    gg[4] = (MOVE == 2 ? 0.0 : pin[4]) - h[4];
    gg[5] = cp * pin[5] - h[5];
    gg[7] = 0.0;
    solveET8x<(MOVE == 2)>(J, gg);
#pragma unroll
    for (int i = 0; i < 7; ++i) pin[i] = gg[i];
    if (ls) {        // only the least-squares multiplier estimate looks at the size of the multipliers
#pragma unroll
      for (int i = 0; i < 7; ++i) pimax = dmax(pimax, fabs(gg[i]));
    }
    if (g == 0) { gg[7] = 0.0; stv<8>(W.D(k) + D_PI, gg); }
  }
  }
  W.rpar = par;
  Grp<GP>::sync(pmk);
  W.pimax = GP > G ? Grp<GP>::bcast(pmk, pimax, 0) : pimax;
}

// ---------------------------------------------------------------------------------------
// evaluation pass, stage-parallel: trial point x + alpha dx written to buffer `dst`, its merit and
// KKT-error terms, and the M records of the trial point (the model of the next Newton system).
// The per-stage arithmetic is that of dc::eval_pass.
// ---------------------------------------------------------------------------------------
template <int GP, int MOVE, class CW>
LM_SWEEP void coop_eval(const Params& P, const Mesh& M, const Options& O, const CW& W, int src, int dst,
                        const Scal& c0, const TermStep& ts, double mu, double alpha, double alpha_z,
                        double alpha_lam, Scal& t) {
  const int N = M.N;
  const int g = W.g;
  const unsigned gm = W.mask;
  const double tf0 = c0.tf, dtf = ts.dtf;
  const double tf = tf0 + alpha * dtf;
  const double wdc = O.w_dcost;
  const double cp = (MOVE == 1) ? 1.0 : (MOVE == 2) ? 0.0 : P.coup5, cq4 = (MOVE == 2) ? 0.0 : 1.0;   // (compile-time with the move term)
  t.tf = tf;
  // ---- terminal scalars of the trial point (every lane) ----
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
  double theta = 0, prim = 0, dual = 0, sumlog = 0, cmin = 1e300, cmax = 0, slam = 0, sz = 0, gtf = 0, movecost = 0;
  int bad = 0;
  for (int k = 1 + g; k <= N; k += GP) {
    if (k + GP <= N) { prefetch_rec<XR>(W.X(src, k + GP)); prefetch_rec<DR>(W.D(k + GP)); }
    double xo[XR], d[DR], xm[8], dm[8];
    ldv<XR>(W.X(src, k), xo);
    ldv<DR>(W.D(k), d);
    ldv<8>(W.X(src, k - 1), xm);          // node k-1: z, u (node 0 rows are zeros)
    ldv<8>(W.D(k - 1), dm);
    double z[7], zp[7];                   // index 6 = u
#pragma unroll
    for (int i = 0; i < 7; ++i) { z[i] = fma(alpha, d[i], xo[i]); zp[i] = fma(alpha, dm[i], xm[i]); }
    const double u_old = xo[X_U], du = d[6], u = z[6];
    double lam[7];
#pragma unroll
    for (int i = 0; i < 7; ++i) lam[i] = fma(alpha_lam, d[D_PI + i] - xo[X_LAM + i], xo[X_LAM + i]);
    double zla = xo[X_ZLA], zua = xo[X_ZUA], zlu = xo[X_ZLU], zuu = xo[X_ZUU];
    const double kap = M.h[k] * P.T;
    const double taum = P.mT * M.tau[k];
    // ---- bound multipliers: dz = (mu - z dx)/d - z (old d, old z), then the kappa_Sigma clip ----
    {
      double rLa, rUa, rLu, rUu;
      recip4(xo[4], P.a_ub - xo[4], u_old + P.u_ub, P.u_ub - u_old, rLa, rUa, rLu, rUu);
      const double da = d[4];
      zla += alpha_z * ((mu - zla * da) * rLa - zla);
      zua += alpha_z * ((mu + zua * da) * rUa - zua);
      zlu += alpha_z * ((mu - zlu * du) * rLu - zlu);
      zuu += alpha_z * ((mu + zuu * du) * rUu - zuu);
    }
    const double dLa = z[4], dUa = P.a_ub - z[4], dLu = u + P.u_ub, dUu = P.u_ub - u;
    if (!(dLa > 0 && dUa > 0 && dLu > 0 && dUu > 0)) bad = 1;
    {
      const double c1 = dLa * zla, c2 = dUa * zua, c3 = dLu * zlu, c4 = dUu * zuu;
      const double hi = 1e10 * mu, lo = 1e-10 * mu;
      if (dmax(dmax(c1, c2), dmax(c3, c4)) > hi || dmin(dmin(c1, c2), dmin(c3, c4)) < lo) {
        zla = clip_mult(zla, dLa, mu); zua = clip_mult(zua, dUa, mu);
        zlu = clip_mult(zlu, dLu, mu); zuu = clip_mult(zuu, dUu, mu);
      }
    }
    double slack = (dLa * dUa) * (dLu * dUu);
    {
      const double c1 = dLa * zla, c2 = dUa * zua, c3 = dLu * zlu, c4 = dUu * zuu;
      cmin = dmin(cmin, dmin(dmin(c1, c2), dmin(c3, c4)));
      cmax = dmax(cmax, dmax(dmax(c1, c2), dmax(c3, c4)));
    }
    sz += (zla + zua) + (zlu + zuu);
    // ---- move slack pair ----
    double pp = xo[X_PP], pn = xo[X_PN], zpp = xo[X_ZPP], zpn = xo[X_ZPN];
    if (MOVE) {
      dc::Move mv;
      mv.build(pp, pn, zpp, zpn, u_old - xm[X_U], wdc, mu, false);
      double dp, dn;
      mv.steps(du - dm[6], dp, dn);
      const double ip = mv.ip, in_ = mv.in_;
      zpp += alpha_z * ((mu - zpp * dp) * ip - zpp);
      zpn += alpha_z * ((mu - zpn * dn) * in_ - zpn);
      pp = fma(alpha, dp, pp);
      pn = fma(alpha, dn, pn);
      if (!(pp > 0 && pn > 0)) bad = 1;
      {
        const double c1 = pp * zpp, c2 = pn * zpn;
        if (dmax(c1, c2) > 1e10 * mu || dmin(c1, c2) < 1e-10 * mu) { zpp = clip_mult(zpp, pp, mu); zpn = clip_mult(zpn, pn, mu); }
      }
      slack *= pp * pn;
      {
        const double c1 = pp * zpp, c2 = pn * zpn;
        cmin = dmin(cmin, dmin(c1, c2));
        cmax = dmax(cmax, dmax(c1, c2));
      }
      sz += zpp + zpn;
      movecost += pp + pn;
    }
    sumlog += lm_log_pos(slack);
    // ---- dynamics at the trial point: defects, and the model of the next Newton system ----
    double* mrec = W.Mo(dst, k);
    build_stage<MOVE>(P, O, kap, taum, tf, false, z, u, zp, zp[6], lam, zla, zua, zlu, zuu, pp, pn, zpp, zpn, mrec);
    StageJac J;
    jac_load(mrec, J);
    double c[8];
    ldv<8>(mrec + M_C, c);
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      const double ac = fabs(c[i]);
      theta += ac;
      prim = dmax(prim, ac);
      slam += fabs(lam[i]);
    }
    if (MOVE) {
      slam += fabs(lam[6]);
      const double c6 = fabs((u - zp[6]) - pp + pn);            // move row: u_k - u_{k-1} = p - n
      theta += c6;
      prim = dmax(prim, c6);
    }
    // ---- Lagrangian gradient wrt (s_k, u_k) and wrt the move ----
    double res[7];
    applyET6(J, lam, res);
    res[4] += zua - zla;
    res[6] = -J.beta * lam[5] - (MOVE == 2 ? lam[4] : 0.0) + lam[6] - zlu + zuu;
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
      double xn[8], pn8[8];
      ldv<8>(W.X(src, k + 1) + X_U, xn);     // u, lam_0..6 of node k+1
      ldv<8>(W.D(k + 1) + D_PI, pn8);
#pragma unroll
      for (int i = 0; i < 7; ++i) {
        const double ln = fma(alpha_lam, pn8[i] - xn[1 + i], xn[1 + i]);
        res[i] -= (i == 5 ? cp : i == 4 ? cq4 : 1.0) * ln;
      }
    }
#pragma unroll
    for (int i = 0; i < 7; ++i) dual = dmax(dual, fabs(res[i]));
    if (MOVE) dual = dmax(dual, dmax(fabs(wdc - lam[6] - zpp), fabs(wdc + lam[6] - zpn)));   // d L / d p_k, d L / d n_k
    else dual = dmax(dual, fabs(lam[6]));                                                   // free move: d L / d v_k
    gtf -= J.e0 * lam[0] + J.e1 * lam[1] + J.e2 * lam[2] + J.e3 * lam[3] + J.e4 * lam[4] + J.e5 * lam[5];
    // ---- write the trial iterate ----
    double xo2[XR];
#pragma unroll
    for (int i = 0; i < 7; ++i) { xo2[i] = z[i]; xo2[X_LAM + i] = lam[i]; }
    xo2[X_ZLA] = zla; xo2[X_ZUA] = zua; xo2[X_ZLU] = zlu; xo2[X_ZUU] = zuu;
    xo2[X_PP] = pp; xo2[X_PN] = pn; xo2[X_ZPP] = zpp; xo2[X_ZPN] = zpn;
    xo2[22] = 0.0; xo2[23] = 0.0;
    stv<XR>(W.X(dst, k), xo2);
  }
  theta = Grp<GP>::sum(gm, theta);
  sumlog = Grp<GP>::sum(gm, sumlog) + sumlog0;
  slam = Grp<GP>::sum(gm, slam) + slam0;
  sz = Grp<GP>::sum(gm, sz) + sz0;
  gtf = Grp<GP>::sum(gm, gtf) + gtf0;
  movecost = Grp<GP>::sum(gm, movecost);
  prim = Grp<GP>::max(gm, prim);
  dual = dmax(Grp<GP>::max(gm, dual), fabs(gtf));
  cmin = dmin(Grp<GP>::min(gm, cmin), cmin0);
  cmax = dmax(Grp<GP>::max(gm, cmax), cmax0);
  const bool anybad = Grp<GP>::any(gm, bad) != 0 || bad0;
  t.theta = theta;
  t.fobj = O.obj_scale * tf + wdc * movecost;
  t.sumlog = anybad ? -1e300 : sumlog;
  t.prim_inf = prim; t.dual_inf = dual; t.cmin = cmin; t.cmax = cmax; t.sum_lam = slam; t.sum_z = sz;
  if (anybad || !(theta == theta)) t.theta = 1e300;
  ring_publish();                              // the M records of the trial point travel through the ring next
  Grp<GP>::sync(gm);
}

// Reference column of the batch warm start (ascent_ipm.cuh: REF_*), so that every kernel can start from a reference
// produced here.
template <int G, class CW>
LM_NOINLINE void coop_store_ref(const Params& P, const Mesh& M, const CW& W, int src, const Scal& c, double mu, bool ok,
                                double* ref) {
  const int N1 = M.N + 1;
  for (int k = 1 + W.g; k <= M.N; k += G) {
    double x[XR];
    ldv<XR>(W.X(src, k), x);
    ref_put_node(ref, N1, k, x);
  }
  if (W.g == 0) ref_put_scalars(ref, N1, P, c, mu, ok);
}

}  // namespace coop

// Sweeps policy of the cooperative formulation for the IPM driver (ipm_iterate_t).
//   G  lanes carry the sequential phases (cost-to-go distributed by rows: 8/G rows per lane),
//   GP lanes (a multiple of G, at most a warp) carry the stage-parallel phases of the same problem.
template <int G, int GP, int MOVE, bool VREC = (GP > G)>
struct SweepsCoop {
  enum : int { LANES_PER_PROBLEM = GP, MOVE_TERM = MOVE, STORES_REF = 1 };    // STORES_REF: has store_ref
  template <class CW>
  LM_HD static int n_eq(const CW&, int N) { return (MOVE ? 7 : 6) * N + 3; }
  template <class CW>
  LM_HD static int n_bd(const CW&, int N) { return (MOVE ? 6 : 4) * N + 4; }
  template <class CW>
  LM_HD static bool backward(const Params& P, const Mesh& M, const Options& O, const CW& W, int src, const Scal& c0,
                             double mu, double dw, bool ls, double* dtf) {
    // the least-squares multiplier estimate factorises its own model (Hessian := I) of the start point
    if (ls) coop::coop_build<GP, MOVE>(P, M, O, W, src, c0.tf, true);
    return coop::coop_backward<G, GP, MOVE, VREC>(P, M, O, W, src, c0, mu, dw, ls, dtf);
  }
  template <class CW>
  LM_HD static void forward(const Params& P, const Mesh& M, const Options& O, const CW& W, int src, const Scal& c0,
                            double mu, double tau, double dtf, bool ls, TermStep& ts, StepInfo& si) {
    coop::coop_forward<G, GP, MOVE, VREC>(P, M, O, W, src, c0, mu, tau, dtf, ls, ts, si);
  }
  template <class CW>
  LM_HD static void eval(const Params& P, const Mesh& M, const Options& O, const CW& W, int src, int dst,
                         const Scal& c0, const TermStep& ts, double mu, double /*dw*/, double alpha, double alpha_z,
                         double alpha_lam, int /*mode*/, Scal& t, double* pimax) {
    // (the new multipliers are always read: the adjoint recursion ran at the end of forward())
    coop::coop_eval<GP, MOVE>(P, M, O, W, src, dst, c0, ts, mu, alpha, alpha_z, alpha_lam, t);
    if (pimax) *pimax = W.pimax;
  }
  // start points (ascent_ipm.cuh: start_rollout, ...): node k into the X record of buffer 0 with its step record
  // zeroed; node 0 pinned at zero
  template <class CW>
  LM_HD static void store_node(const CW& W, int k, const double* x) {
    double r[coop::XR], zero[coop::DR];
#pragma unroll
    for (int i = 0; i < NODE_N; ++i) r[i] = x[i];
    r[22] = 0.0; r[23] = 0.0;
    coop::stv<coop::XR>(W.X(0, k), r);
#pragma unroll
    for (int i = 0; i < coop::DR; ++i) zero[i] = 0.0;
    coop::stv<coop::DR>(W.D(k), zero);
  }
  template <class CW>
  LM_HD static void zero_node0(const CW& W) {
    double zero[coop::XR];
#pragma unroll
    for (int i = 0; i < coop::XR; ++i) zero[i] = 0.0;
    coop::stv<coop::XR>(W.X(0, 0), zero); coop::stv<coop::XR>(W.X(1, 0), zero); coop::stv<coop::DR>(W.D(0), zero);
  }
  template <class CW>
  LM_HD static void store_ref(const Params& P, const Mesh& M, const CW& W, int src, const Scal& c, double mu, bool ok,
                              double* ref) { coop::coop_store_ref<GP>(P, M, W, src, c, mu, ok, ref); }
  // node k of iterate `cur`: x = the six states and the control, lam = the multipliers of the ydot, xdot and angledot
  // rows; either may be null
  template <class CW>
  LM_HD static void node(const CW& W, int cur, int k, double* x, double* lam) {
    double r[coop::XR];
    coop::ldv<coop::XR>(W.X(cur, k), r);
    if (x) for (int i = 0; i < 7; ++i) x[i] = r[coop::X_Z + i];     // states, then X_U
    if (!lam) return;
    lam[0] = r[coop::X_LAM + 1]; lam[1] = r[coop::X_LAM + 3]; lam[2] = r[coop::X_LAM + 5];
  }
  // the multipliers of node k (as ws_node_duals): the six defect rows, the angle's upper bound, the control's bounds
  template <class CW>
  LM_HD static void node_duals(const CW& W, int cur, int k, double* d) {
    double r[coop::XR];
    coop::ldv<coop::XR>(W.X(cur, k), r);
    for (int i = 0; i < 6; ++i) d[i] = r[coop::X_LAM + i];
    d[6] = r[coop::X_ZUA]; d[7] = r[coop::X_ZLU]; d[8] = r[coop::X_ZUU];
  }
  template <class CW>
  LM_HD static void remerit(const Mesh&, const Options&, const CW&, int, double, Scal&) {}
};

}  // namespace lmato
