// Convex-MPC stance QP: one CTA per env, float64, everything on chip (sm_100a).
//
// Replaces mpc_osqp.ConvexMpc::ComputeContactForces of motion_imitation==0.0.5 (third-party;
// call site robot_gym/controllers/mpc/mpc_controller.py:47-56,105).  The reference builds a
// dense 13h x 3kh condensed system with a Pade matrix exponential and hands it to OSQP
// (ADMM to 1e-3 + polish).  This kernel reaches the same unique optimum differently:
//
//  * [[A,B],[0,0]] is nilpotent of index 3, so the discretisation is exact in closed form and
//    the state deviation depends on the forces only through the 6-dim acceleration
//    a_t = B_nu u_t.  The condensed Hessian is  P = 2 alpha I + W^T K W  with
//    W = I_h (x) B_nu (6h x 12h) and K = c1 (x) K1 + c2 (x) K2 (6h x 6h, Kronecker in time).
//  * Newton systems (P + G^T D G) dx = r are solved through the Woodbury identity with the
//    block-diagonal 3x3 part E = 2 alpha I + G^T D G:  only a 6h x 6h SPD matrix
//    Psi = K^-1 + W E^-1 W^T is factorised (60 x 60 at h = 10 instead of 120 x 120).
//  * K^-1 comes from a host-precomputed generalised eigen-decomposition of (c2, c1).
//  * The solver (DESIGN.md 3.3): verified active-set rounds -- the equality-constrained QP on the
//    guessed active rows is solved exactly in the per-block null space and the guess is checked
//    against primal feasibility, multiplier signs and stationarity (the analogue of OSQP's polish);
//    a verified round is the optimum.  They start cold (fz >= fz_min active in the last horizon
//    step) or from the set the same env verified one control step earlier, and refactorise only the
//    time blocks whose rows moved.  Problems on which the rounds cycle fall back to a Mehrotra
//    predictor-corrector interior point from a strictly feasible start, which hands its active rows
//    back to the rounds; an escalation ladder drives the interior point deeper when they do not verify.
//  * Two kernels per solve (DESIGN.md 3.8): mpc_solve_kernel<H, LEAN = true> holds the active-set rounds only and
//    queues the envs they do not verify; mpc_fallback_kernel<H> (the complete solver) runs on that queue, launched
//    programmatically behind the first.  Batches that fit one wave of CTAs run mpc_solve_kernel<H, false> alone.
//  * h = 20 factorises Psi by a Riccati sweep over the horizon instead of the dense Cholesky (DESIGN.md 3.9).
//  * A warp alone on its scheduler issues one instruction every ~4 cycles: the serial phases (sweeps, late Cholesky
//    panels) are written for instruction COUNT, not for short dependent chains (DESIGN.md 3.10).
//
// Thread roles inside a CTA (NT = 32 * ceil(6h / 32) threads on the dense path, 32 * ceil(4h / 32) on the Riccati path):
//   "block" threads  tid < 4h : own one (time step, leg) force triple (and, in the complete solver only, its 10
//                               slacks and multipliers) in registers; 4 adjacent lanes = the 4 legs of a step,
//                               so per-step sums over legs are two __shfl_xor rounds.
//   "row"   threads  tid < 6h : own one row of Psi during the Cholesky factorisation.
//   one warp (rotated over the SM sub-partitions, sm.solver_warp) runs the triangular / Riccati sweeps.
#include "rg_common.cuh"
#include <math.h>
#include <map>
#include <mutex>

#ifdef RG_DEBUG_TRACE
// debug builds only (RG_DEBUG_TRACE=1 python -m robot_gym.cuda.build): per-iteration trace of one env
__device__ double* g_trace = nullptr;
__device__ int g_trace_env = -1;
extern "C" int rg_debug_set_trace(double* dev_buf, int env) {
  cudaMemcpyToSymbol(g_trace, &dev_buf, sizeof(dev_buf));
  cudaMemcpyToSymbol(g_trace_env, &env, sizeof(env));
  return 0;
}
#endif
#if defined(RG_DEBUG_TRACE) && !defined(RG_DEBUG_TIMELINE_ONLY)
#define RG_TRACE(slot, value) do { if (g_trace && env == g_trace_env && threadIdx.x == 0) g_trace[slot] = (value); } while (0)
// phase timers: cycles accumulated in g_trace[900 + phase] by thread 0 of the traced env
#define RG_TIC() long long rg_t0_ = clock64()
#define RG_TRESET() rg_t0_ = clock64()
#define RG_TOCL(phase, thr) do { if (g_trace && (int)blockIdx.x == g_trace_env && threadIdx.x == (thr)) g_trace[900 + (phase)] += (double)(clock64() - rg_t0_); rg_t0_ = clock64(); } while (0)
#define RG_TOC(phase) do { if (g_trace && (int)blockIdx.x == g_trace_env && threadIdx.x == 0) g_trace[900 + (phase)] += (double)(clock64() - rg_t0_); rg_t0_ = clock64(); } while (0)
#else
#define RG_TRACE(slot, value) do { } while (0)
#define RG_TIC() do { } while (0)
#define RG_TRESET() do { } while (0)
#define RG_TOC(phase) do { } while (0)
#define RG_TOCL(phase, thr) do { } while (0)
#endif

namespace {

constexpr unsigned kFull = 0xffffffffu;

// Linear algebra behind the Newton / active-set systems:  horizons >= kRiccatiMinH factorise Psi by a backward
// Riccati sweep over the horizon (O(h) work and storage: riccati_factor / riccati_solve), shorter ones by the dense
// packed Cholesky (O(h^3), but 60 rows keep 64 threads busy and the panel routine is faster up to h = 10; measured
// in profiles/r02_riccati_vs_cholesky.md).
constexpr int kRiccatiMinH = 20;

template <int H>
struct Cfg {
  static constexpr int N6 = 6 * H;
  static constexpr int NB = 4 * H;
  static constexpr bool RICCATI = H >= kRiccatiMinH;
  // Threads per CTA.  Dense path: one per row of Psi (6h) for the Cholesky.  Riccati path: the sweeps run in one warp,
  // so only the 4h (step, leg) block threads are needed -- the 6h "rows" of K-products are looped over (h = 20: 96
  // threads instead of 128, i.e. 5 resident CTAs per SM at 128 registers instead of 4).
  static constexpr int NT = RICCATI ? ((NB + 31) / 32) * 32 : ((N6 + 31) / 32) * 32;
  static constexpr int NW = NT / 32;
  static constexpr int NPSI = N6 * (N6 + 1) / 2 + 64;   // slack: the pipelined loads of the factor routines over-read (values unused)
  static constexpr int NA = 3 * H;
  static constexpr int NKA = NA * (NA + 1) / 2;
  static constexpr int RPL = (N6 + 31) / 32;   // Psi rows per lane in the triangular sweeps
  // the gradient at the particular solution is evaluated as "pass -1" of the solve / refine loop (one inlined copy of
  // apply_p instead of two: less code on the round's path; +1.5 % at h = 10, -3 % at h = 5 where the kernel spills)
  static constexpr bool GRAD_IN_PASS_LOOP = H == 10;
  // resident CTAs per SM the register allocation is sized for (launch bound and shared-memory carveout; shared memory
  // allows 9 / 2 at h = 10 / 20).  h = 10: 8 until the instruction-count pass of round 2 had loaded the shared-memory pipe
  // to 60 % of its wavefront peak; since then 7 is faster (+2.5 % at 65536 envs, +3.5 % at 4096, where 4096 / (148 x 7)
  // is almost a whole number of waves); 6: -6 %, 9: -4 %.
  static constexpr int MIN_BLOCKS = H <= 5 ? 24 : (H <= 10 ? 7 : 5);
};

template <int H, bool RIC = Cfg<H>::RICCATI>
struct Smem {
  // dense path: Psi and its Cholesky factor
  __align__(16) double psi[RIC ? 2 : Cfg<H>::NPSI];   // lower triangle, row-major, packed (prow)
  double kinv_ang[RIC ? 1 : Cfg<H>::NKA];    // K^-1 angular block, packed, index a = 3 j + c
  __align__(16) double rdiag[RIC ? 1 : Cfg<H>::N6];
  // Riccati path (see riccati_factor): per stage P_{t+1} Gam (12 x 6), J_t, N_t (6 x 6), and the sweep's scratch
  // (the dense path declares them with one or two elements: they must not cost it shared memory)
  __align__(16) double fac_pg[RIC ? H : 1][RIC ? 72 : 2];
  __align__(16) double fac_j[RIC ? H : 1][RIC ? 36 : 2];
  __align__(16) double fac_n[RIC ? H : 1][RIC ? 36 : 2];
  __align__(16) double pm[RIC ? 144 : 2];      // P_{t+1}: full symmetric storage, row-major 12 x 12, order (pi; sigma)
  __align__(16) double pm2[RIC ? 144 : 2];     // P_{t+1} - PG N PG^T before the time update
  __align__(16) double m6[RIC ? 6 : 1][RIC ? 36 : 2];    // 6 x 6 scratch matrices: D, S, U = D S, Y, Y^-1, G
  __align__(16) double t1[RIC ? 72 : 2];       // PG N
  __align__(16) double rvec[RIC ? H * 6 : 2];   // r_t of the backward sweep of the current solve
  double gt[H * 6];                // g~ : gradient in acceleration space
  __align__(16) double avec[H * 6];   // W u, right-hand sides and Woodbury solutions
  double kvec[H * 6];              // K (W u)
  __align__(16) double blk44[36];  // updated 4x4 diagonal block of the current Cholesky panel (36: the tuned smem layout)
  double bang[4][9];               // A_leg = I_world^-1 [r_leg]x
  double k2ang[9];
  double k1[6];
  double k2lin[3];
  double nblk[H][21];              // per time step: lower triangle of sum_legs B E^-1 B^T (setup: (K1 + gamma_t K2)^-1 scratch)
  double red[3][8];
  int flag;
  int solver_warp;                 // the warp that runs the single-warp phases (sweeps): see solve_env
};

__device__ __forceinline__ int tri(int i, int k) { return i * (i + 1) / 2 + k; }

// offset of row i of the lower-triangular Psi storage.
// packed triangle: T(i) mod 16 is a permutation over 16 consecutive rows, so the per-column 64-bit
// accesses of a half-warp (same column, consecutive rows) are bank-conflict free
__device__ __forceinline__ int prow(int i) { return i * (i + 1) / 2; }
__device__ __forceinline__ double2 ld2(const double* p) { return make_double2(p[0], p[1]); }
// 128-bit load of two consecutive doubles; the caller guarantees 16-byte alignment
__device__ __forceinline__ double2 ld2v(const double* p) { return *reinterpret_cast<const double2*>(p); }

__device__ __forceinline__ double c1f(int h, int j, int k) { return (double)(h - (j > k ? j : k)); }

// Interior-point start (used only when the cold start gives up; A/B in tools/ab_gaits.py):
//   mu0 = kIpmLam0 * max(|q|, |P u0 + q|)   centred start s lam = mu0
//   u0  = safe point + kIpmWarm * (largest strictly feasible step towards the last active-set iterate)
constexpr double kIpmLam0 = 0.01;
constexpr double kIpmWarm = 0.99;
// interior point: iterations without halving the best residual before a close iterate is handed to the rounds
constexpr int kIpmSlowIters = 5;
// cold start: fz >= fz_min is guessed active in the last kColdGuessLast steps of the horizon
constexpr int kColdGuessLast = 1;
// ... and in the last kColdGuessLast4 steps when all four legs stand: the redundant legs are unloaded earlier
// (fz_min is active at step h-2 on 78 % of the legs of four-stance trot states against 50 % with two stance legs,
// and a four-stance problem never verifies from the one-step guess alone: tools/experiments/guess_stats.py)
constexpr int kColdGuessLast4 = 2;
// cold start: its last round hands over when more than this many rows still move
constexpr double kColdLastRoundNchg = 4.0;
// multiplier tolerance (relative to the gradient scale) below which a STICKY row -- one that was dropped and came back --
// is still held: it stops the in / out cycling of weakly active rows, at the price of a point that may sit up to
// tol / (2 alpha) away from the optimum along a weakly curved direction
constexpr double kStickyTol = 1e-9;
// After the first solve of an active-set round the refinement pass is skipped when the projected
// gradient is already below this (relative to the gradient scale): the error it leaves in the
// weakly curved directions is <= tol / (2 alpha).
constexpr double kSkipRefineTol = 1e-10;

// ---- block-wide reductions (all threads call; result valid in all threads) -------------------
// WHAT: bit 0 = the sum, bit 1 = the maximum, bit 2 = the minimum is wanted (the others are left untouched)
template <int NW, int WHAT = 7>
__device__ __forceinline__ void block_reduce(double& sum, double& mx, double& mn, double (*red)[8]) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    if (WHAT & 1) sum += __shfl_xor_sync(kFull, sum, o);
    if (WHAT & 2) mx = fmax(mx, __shfl_xor_sync(kFull, mx, o));
    if (WHAT & 4) mn = fmin(mn, __shfl_xor_sync(kFull, mn, o));
  }
  if (NW == 1) return;
  const int w = threadIdx.x >> 5;
  __syncthreads();   // protect red[] from the previous use
  if ((threadIdx.x & 31) == 0) {
    if (WHAT & 1) red[0][w] = sum;
    if (WHAT & 2) red[1][w] = mx;
    if (WHAT & 4) red[2][w] = mn;
  }
  __syncthreads();
  if (WHAT & 1) sum = red[0][0];
  if (WHAT & 2) mx = red[1][0];
  if (WHAT & 4) mn = red[2][0];
#pragma unroll
  for (int i = 1; i < NW; ++i) {
    if (WHAT & 1) sum += red[0][i];
    if (WHAT & 2) mx = fmax(mx, red[1][i]);
    if (WHAT & 4) mn = fmin(mn, red[2][i]);
  }
}

__device__ __forceinline__ double quad_sum(double v) {   // sum over the 4 legs of a time step
  v += __shfl_xor_sync(kFull, v, 1);
  v += __shfl_xor_sync(kFull, v, 2);
  return v;
}

// 1 / sqrt(d) for the Cholesky pivots: hardware seed (MUFU.RSQ64H, ~2^-21 relative) and one third-order step
// y (1 + e/2 + 3 e^2/8), e = 1 - d y^2  (error 5 e^3 / 16 < 2^-60): 6 instructions on the pivot chain instead of the 12
// of rsqrt() with its range checks.  No special cases: d <= 0 gives NaN / inf, which the caller tests for once per panel.
__device__ __forceinline__ double rsqrt_pivot(double d) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
  const double e = fma(-(d * y), y, 1.0);
  return fma(y * e, fma(0.375, e, 0.5), y);
}

// ---- in-place Cholesky of the packed SPD matrix: one thread per row, panels of 4 columns --------
// Left-looking by panels J = {j0..j0+3}:
//   phase 1  every row thread i >= j0 accumulates its four dot products  A[i][j0+c] - sum_{k<j0} L[i][k] L[j0+c][k]
//            with ONE load of its own L[i][k] and four broadcast loads of the panel rows per k
//            (the four accumulators are independent chains), and the panel rows publish theirs;
//   barrier
//   phase 2  every thread factors the 4x4 diagonal block redundantly in registers (10 broadcast
//            loads, 4 rsqrt) and solves its own row against it; nobody waits for an owner thread;
//   barrier
// -> 2 barriers per 4 columns and ~2.6 instructions per useful FMA instead of 60 barriers and ~5.5.
// The factor's diagonal lives in sm.rdiag as 1 / L[j][j]; the triangular sweeps need nothing else.
// __noinline__: one copy of the code, called from every phase of the solver.
// j_begin (a multiple of 4): columns before it already hold the factor and are kept -- a matrix that
// changed only in rows/columns >= j_begin has the same leading factor columns (left-looking order).
template <int H, class SM>
__device__ __noinline__ void cholesky_rows(SM& sm, int j_begin) {
  constexpr int N6 = Cfg<H>::N6;
  const int i = threadIdx.x;
  const bool row_ok = i < N6;
  double* row_i = sm.psi + prow(row_ok ? i : 0);
  if (i == 0) sm.flag = 0;   // published by the first barrier below
  RG_TIC();
#pragma unroll 1
  for (int j0 = j_begin; j0 < N6; j0 += 4) {
    RG_TOCL(32, N6 - 1);
    // panel width: always 4 when 6h is a multiple of 4 (h = 10, 20); the last panel of N6 = 30 has 2 columns
    const int w = (N6 % 4 == 0) ? 4 : (N6 - j0 < 4 ? N6 - j0 : 4);
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    const bool in_play = row_ok && i >= j0;
    if (in_play) {
      const double* r2 = sm.psi + prow(i);
      const double* p0 = sm.psi + prow(j0);
      const double* p1 = sm.psi + prow(j0 + (w > 1 ? 1 : 0));
      const double* p2 = sm.psi + prow(j0 + (w > 2 ? 2 : 0));
      const double* p3 = sm.psi + prow(j0 + (w > 3 ? 3 : 0));
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[c] = (c < w && j0 + c <= i) ? row_i[j0 + c] : 0.0;
      const int ng = j0 >> 1;                          // pairs of columns already factored (j0 % 4 == 0)
      if (w == 4) {
        // 128-bit broadcast loads of the panel rows.  T(r) = r(r+1)/2 is even for r = 0, 3 (mod 4) and odd for
        // r = 1, 2 (mod 4): rows j0 and j0+3 are 16-byte aligned at even k, rows j0+1 and j0+2 at odd k.  The
        // latter two are read as the pairs (2g+1, 2g+2) and consumed with a one-element lag.  All loads of step
        // g+1 are in flight while step g's eight FMAs retire; the last prefetch over-reads by <= 2 doubles
        // (still inside Psi / its slack, values unused).
        double2 a = ld2(r2);
        double2 b0 = ld2v(p0), b3 = ld2v(p3);
        double b1x = p1[0], b2x = p2[0];
        double2 q1 = ld2v(p1 + 1), q2 = ld2v(p2 + 1);
        // unrolled 4 times: a trip moves five pointers and rotates the lagged operands, ~10 of 38 instructions at 2
#pragma unroll 4
        for (int g = 0; g < ng; ++g) {
          const double2 an = ld2(r2 + 2 * g + 2);
          const double2 c0 = ld2v(p0 + 2 * g + 2), c3 = ld2v(p3 + 2 * g + 2);
          const double2 n1 = ld2v(p1 + 2 * g + 3), n2 = ld2v(p2 + 2 * g + 3);
          acc[0] = fma(-a.x, b0.x, acc[0]); acc[1] = fma(-a.x, b1x, acc[1]);
          acc[2] = fma(-a.x, b2x, acc[2]);  acc[3] = fma(-a.x, b3.x, acc[3]);
          acc[0] = fma(-a.y, b0.y, acc[0]); acc[1] = fma(-a.y, q1.x, acc[1]);
          acc[2] = fma(-a.y, q2.x, acc[2]); acc[3] = fma(-a.y, b3.y, acc[3]);
          b1x = q1.y; b2x = q2.y;
          a = an; b0 = c0; b3 = c3; q1 = n1; q2 = n2;
        }
      } else {
        // scalar pair loads, software-pipelined one stage ahead
        double2 a = ld2(r2), b0 = ld2(p0), b1 = ld2(p1), b2 = ld2(p2), b3 = ld2(p3);
#pragma unroll 2
        for (int g = 0; g < ng; ++g) {
          const int gn = g + 1 < ng ? g + 1 : g;
          const double2 an = ld2(r2 + 2 * gn), c0 = ld2(p0 + 2 * gn), c1 = ld2(p1 + 2 * gn), c2 = ld2(p2 + 2 * gn), c3 = ld2(p3 + 2 * gn);
          acc[0] = fma(-a.x, b0.x, acc[0]); acc[1] = fma(-a.x, b1.x, acc[1]);
          acc[2] = fma(-a.x, b2.x, acc[2]); acc[3] = fma(-a.x, b3.x, acc[3]);
          acc[0] = fma(-a.y, b0.y, acc[0]); acc[1] = fma(-a.y, b1.y, acc[1]);
          acc[2] = fma(-a.y, b2.y, acc[2]); acc[3] = fma(-a.y, b3.y, acc[3]);
          a = an; b0 = c0; b1 = c1; b2 = c2; b3 = c3;
        }
      }
      if (i < j0 + w) {                                // a panel row: publish the updated entries A'[i][j0..i]
        // into the side buffer, NOT into Psi: phase 2 overwrites the panel rows of Psi with the factor
        // while other warps may still be reading the block (that was a cross-warp race)
#pragma unroll
        for (int c = 0; c < 4; ++c) if (j0 + c <= i) sm.blk44[4 * (i - j0) + c] = acc[c];
      }
    }
    RG_TOCL(30, N6 - 1);
    __syncthreads();
    RG_TOCL(33, N6 - 1);
    if (in_play) {
      // 4x4 diagonal block A' (lower triangle), broadcast loads; entries beyond the panel width read as identity
      double a[4][4];
      {
        // six 128-bit broadcast loads instead of ten 64-bit ones (entries above the diagonal are stale, unused)
        const double2 r0 = ld2v(sm.blk44), r1 = ld2v(sm.blk44 + 4), r2a = ld2v(sm.blk44 + 8), r2b = ld2v(sm.blk44 + 10),
                      r3a = ld2v(sm.blk44 + 12), r3b = ld2v(sm.blk44 + 14);
        a[0][0] = r0.x;
        a[1][0] = r1.x; a[1][1] = r1.y;
        a[2][0] = r2a.x; a[2][1] = r2a.y; a[2][2] = r2b.x;
        a[3][0] = r3a.x; a[3][1] = r3a.y; a[3][2] = r3b.x; a[3][3] = r3b.y;
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
          for (int c = 0; c <= r; ++c) if (r >= w) a[r][c] = (r == c ? 1.0 : 0.0);
      }
      // factor: l[r][c] for c < r, inverse diagonal in rd[r].  A non-positive pivot turns rd[] into NaN / inf (no clamp on
      // the chain): the test behind the panel loop catches it, the caller gives the factorisation up (sm.flag).
      double rd[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        double d = a[c][c];
#pragma unroll
        for (int k = 0; k < c; ++k) d = fma(-a[c][k], a[c][k], d);
        rd[c] = rsqrt_pivot(d);
#pragma unroll
        for (int r = c + 1; r < 4; ++r) {
          double v = a[r][c];
#pragma unroll
          for (int k = 0; k < c; ++k) v = fma(-a[r][k], a[c][k], v);
          a[r][c] = v * rd[c];
        }
      }
      // x L_JJ^T = acc: forward substitution over the panel columns.  A panel row runs the same code: its acc[] are the
      // block entries A'[r][0..r], so x[c] = L[r][c] for c < r -- only the entries strictly left of the diagonal are stored.
      double x[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        double v = acc[c];
#pragma unroll
        for (int k = 0; k < c; ++k) v = fma(-x[k], a[c][k], v);
        x[c] = v * rd[c];
      }
#pragma unroll
      for (int c = 0; c < 4; ++c) if (c < w && j0 + c < i) row_i[j0 + c] = x[c];
      if (i == j0) {
        // every in-play thread holds the block's four inverse pivots: the first panel row publishes all of them (one
        // thread, two 16-byte stores) instead of every panel row selecting its own
        if constexpr (N6 % 4 == 0) {
          *reinterpret_cast<double2*>(sm.rdiag + j0) = make_double2(rd[0], rd[1]);
          *reinterpret_cast<double2*>(sm.rdiag + j0 + 2) = make_double2(rd[2], rd[3]);
        } else {
#pragma unroll
          for (int c = 0; c < 4; ++c) if (c < w) sm.rdiag[j0 + c] = rd[c];
        }
      }
    }
    RG_TOCL(31, N6 - 1);
    __syncthreads();
  }
  // A non-positive pivot turns its column into NaN / inf and, the matrix being dense, every later pivot with it: one
  // test of the last two inverse pivots after the loop sees a failure anywhere in the factorisation (it used to cost
  // ten instructions in every panel).  The caller's barrier publishes the flag.
  if (i == 0 && !(sm.rdiag[N6 - 2] * sm.rdiag[N6 - 1] < 1e300)) sm.flag = 1;
}

// ---- Psi x = b with the factor, b/x in sm.avec; executed by one warp ---------------------------
// Each lane owns RPL CONSECUTIVE rows (30 lanes x 1, 2 or 4 rows).  One step eliminates the RPL pivots
// of one lane: a lane-local RPL x RPL triangular solve with the own diagonal reciprocals held in
// registers, RPL shuffles in flight together, then RPL FMAs per owned row.  A single warp issues an
// instruction every ~4 cycles, so the sweep's time is its instruction count: the updates are predicated
// FMAs with negated operands (no negate / select pairs), the pivot lane is not patched per step (its rows
// stop changing at its own step: every lane solves its own diagonal block ONCE after the sweep), and the
// pivot rows of the backward sweep are addressed by additions.  27 / 30 instructions per step instead of
// 40 / 45 (tools/microbench/chol_bench.cu t5: 6.2k cycles per solve alone on an SM against 9.3k, 11.1k
// against 14.0k with 8 CTAs resident per SM; one pivot per step with strided rows: 14.8k).
// T(i) mod 16 is a permutation over the even and over the odd rows of 16 consecutive lanes, so the
// per-column loads stay bank-conflict free with this ownership too.
template <int H, class SM>
__device__ __noinline__ void tri_solve_warp0(SM& sm) {
  constexpr int N6 = Cfg<H>::N6;
  constexpr int RPL = Cfg<H>::RPL;
  constexpr int NL = N6 / RPL;
  static_assert(NL * RPL == N6 && NL <= 32, "rows must split evenly over the lanes of one warp");
  const int lane = threadIdx.x & 31;   // one warp runs this routine (sm.solver_warp)
  const bool active = lane < NL;
  const int i0 = active ? lane * RPL : 0;
  double x[RPL], rd[RPL], lb[RPL][RPL];
  const double* rowp[RPL];
#pragma unroll
  for (int r = 0; r < RPL; ++r) {
    x[r] = active ? sm.avec[i0 + r] : 0.0;
    rd[r] = sm.rdiag[i0 + r];
    rowp[r] = sm.psi + prow(i0 + r);
#pragma unroll
    for (int c = 0; c < r; ++c) lb[r][c] = rowp[r][i0 + c];
  }
  // forward: L y = b
#pragma unroll 1
  for (int p = 0; p < NL - 1; ++p) {
    double l[RPL][RPL];
#pragma unroll
    for (int r = 0; r < RPL; ++r)
#pragma unroll
      for (int c = 0; c < RPL; ++c) l[r][c] = rowp[r][p * RPL + c];   // lanes <= p read past their diagonal: value unused
    double y[RPL], yb[RPL];
#pragma unroll
    for (int c = 0; c < RPL; ++c) {
      double v = x[c];
#pragma unroll
      for (int cc = 0; cc < c; ++cc) v = fma(-lb[c][cc], y[cc], v);
      y[c] = v * rd[c];
    }
#pragma unroll
    for (int c = 0; c < RPL; ++c) yb[c] = __shfl_sync(kFull, y[c], p);
    if (lane > p) {
#pragma unroll
      for (int c = 0; c < RPL; ++c)
#pragma unroll
        for (int r = 0; r < RPL; ++r) x[r] = fma(-l[r][c], yb[c], x[r]);
    }
  }
  // every lane: y of its own rows (x has been final since the lane's own pivot step)
#pragma unroll
  for (int c = 0; c < RPL; ++c) {
    double v = x[c];
#pragma unroll
    for (int cc = 0; cc < c; ++cc) v = fma(-lb[c][cc], x[cc], v);
    x[c] = v * rd[c];
  }
  // backward: L^T x = y
  const double* rp = sm.psi + prow((NL - 1) * RPL) + i0;        // first row of the pivot lane, my columns
  int rlen = (NL - 1) * RPL;                                     // prow(i) - prow(i - 1) = i
#pragma unroll 1
  for (int p = NL - 1; p > 0; --p) {
    double l[RPL][RPL];
    {
      const double* q = rp;
#pragma unroll
      for (int c = 0; c < RPL; ++c) {
#pragma unroll
        for (int r = 0; r < RPL; ++r) l[c][r] = q[r];
        q += rlen + c + 1;                                        // next row of the packed triangle
      }
    }
    double z[RPL], zb[RPL];
#pragma unroll
    for (int c = RPL - 1; c >= 0; --c) {
      double v = x[c];
#pragma unroll
      for (int cc = c + 1; cc < RPL; ++cc) v = fma(-lb[cc][c], z[cc], v);
      z[c] = v * rd[c];
    }
#pragma unroll
    for (int c = 0; c < RPL; ++c) zb[c] = __shfl_sync(kFull, z[c], p);
    if (lane < p) {
#pragma unroll
      for (int c = RPL - 1; c >= 0; --c)
#pragma unroll
        for (int r = 0; r < RPL; ++r) x[r] = fma(-l[c][r], zb[c], x[r]);
    }
    // step back RPL rows: prow(i - 1) = prow(i) - i
#pragma unroll
    for (int k = 0; k < RPL; ++k) { rp -= rlen; --rlen; }
  }
#pragma unroll
  for (int c = RPL - 1; c >= 0; --c) {
    double v = x[c];
#pragma unroll
    for (int cc = c + 1; cc < RPL; ++cc) v = fma(-lb[cc][c], x[cc], v);
    x[c] = v * rd[c];
  }
  if (active) {
#pragma unroll
    for (int r = 0; r < RPL; ++r) sm.avec[i0 + r] = x[r];
  }
}

// Row p of Psi := scale * K^-1[p][:] + (diagonal 6x6 block of sm.nblk), thread per row.
// Only the time blocks >= t_begin (rows and columns) are written; the rest keeps the factor.
template <int H>
__device__ __forceinline__ void psi_build_rows(Smem<H>& sm, const RgMpcDev* __restrict__ ws, int t_begin) {
  constexpr int N6 = Cfg<H>::N6;
  const int p = threadIdx.x;
  if (p < N6 && p >= 6 * t_begin) {
    const int j = p / 6, c = p - 6 * j;
    double* row = sm.psi + prow(p);
    // K^-1 couples channel c with the three angular channels (c < 3) or only with itself (c >= 3)
    if (c < 3) {
      const double* ka = sm.kinv_ang + tri(3 * j + c, 0);
#pragma unroll 2
      for (int k = t_begin; k < j; ++k) {
        double* dst = row + 6 * k;
        const double v0 = ka[3 * k], v1 = ka[3 * k + 1], v2 = ka[3 * k + 2];
        dst[0] = v0; dst[1] = v1; dst[2] = v2; dst[3] = 0.0; dst[4] = 0.0; dst[5] = 0.0;
      }
    } else {
      const double* kl = ws->kinv_lin[c - 3] + tri(j, 0);
#pragma unroll 2
      for (int k = t_begin; k < j; ++k) {
        double* dst = row + 6 * k;
        const double v = kl[k];
        dst[0] = 0.0; dst[1] = 0.0; dst[2] = 0.0;
        dst[3] = c == 3 ? v : 0.0; dst[4] = c == 4 ? v : 0.0; dst[5] = c == 5 ? v : 0.0;
      }
    }
    // diagonal time block: columns d <= c, plus this step's sum_legs B E^-1 B^T
    const double* nb = sm.nblk[j] + c * (c + 1) / 2;
    double* dst = row + 6 * j;
    for (int d = 0; d <= c; ++d) {
      double v = nb[d];
      if (c < 3) v += sm.kinv_ang[tri(3 * j + c, 3 * j + d)];
      else if (d == c) v += ws->kinv_lin[c - 3][tri(j, j)];
      dst[d] = v;
    }
  }
}


// =====================================================================================================================
// State-space (Riccati) linear algebra, used for long horizons (Cfg<H>::RICCATI).
//
// Every system of the solver has the form  Psi v = b,  Psi = K^-1 + blkdiag_t(D_t)  (6h x 6h).  K is the Hessian, in
// acceleration space, of the tracking cost of the linear system
//     x_{i+1} = Phi x_i + Gam a_i,   x = (pi; sigma) in R^12,   sigma_i = sum_{j<i} a_j,   pi_i = sum_{j<i} (i-j-1/2) a_j,
//     Phi = [[I, I], [0, I]],   Gam = [I/2; I],   1/2 a^T K a = sum_{i=1..h} 1/2 x_i^T Q x_i,   Q = blkdiag(K2, K1),
// so with a = K^-1 v the equation is the two-point boundary value problem
//     a_t = b_t - D_t v_t,   v_t = Gam^T lam_{t+1},   lam_i = Q x_i + Phi^T lam_{i+1},   x_0 = 0,  lam_{h+1} = 0,
// which the backward Riccati sweep  lam_i = P_i x_i + p_i  factorises in O(h) operations on 6 x 6 / 12 x 12 matrices:
//     P_h = Q;   for t = h-1 .. 0:   PG = P_{t+1} Gam,   S = Gam^T PG,   J_t = (I + S D_t)^-1 = S (S + S D_t S)^-1,
//                                    N_t = D_t J_t,   P_t = Q + Phi^T (P_{t+1} - PG N_t PG^T) Phi.
// Neither K^-1 nor any 6h x 6h matrix is formed: 144 h doubles of factors instead of 18 h^2 (23 KB instead of 73 KB of
// shared memory at h = 20).  Y = S + S D S is symmetric positive definite (S is: every acceleration channel carries a
// velocity or a position weight, rg_mpc_setup checks it) whatever the rank of D_t, so its inverse is taken by 3 x 3
// blocks in closed form -- no pivoting, no square roots.  Phi and Gam consist of 0, 1/2 and 1: the time update of P and
// the products with Gam are additions.
//
// One warp runs the sweep.  Every step is spread over the lanes so that a lane computes one or two 6-term dot products
// (lane (r, cp) = row r, columns 2 cp and 2 cp + 1 of a 6 x 6 product; 128-bit shared-memory loads), results go through
// shared memory, __syncwarp between steps: about 400 warp instructions per stage.
// =====================================================================================================================
enum { RM_D = 0, RM_S = 1, RM_U = 2, RM_Y = 3, RM_YI = 4, RM_G = 5 };

__device__ __forceinline__ double2 ldd2(const double* p) { return *reinterpret_cast<const double2*>(p); }

// out[r][2cp..2cp+1] = add[r][..] + sum_k a[r][k] b[k][..]  for the 6 x 6 row-major matrices a, b (add may be null)
__device__ __forceinline__ double2 row_times_cols(const double* __restrict__ a, const double* __restrict__ b, int r, int cp) {
  const double2 a01 = ldd2(a + 6 * r), a23 = ldd2(a + 6 * r + 2), a45 = ldd2(a + 6 * r + 4);
  const double2 b0 = ldd2(b + 2 * cp), b1 = ldd2(b + 6 + 2 * cp), b2 = ldd2(b + 12 + 2 * cp);
  const double2 b3 = ldd2(b + 18 + 2 * cp), b4 = ldd2(b + 24 + 2 * cp), b5 = ldd2(b + 30 + 2 * cp);
  double2 o;
  o.x = (a01.x * b0.x + a01.y * b1.x + a23.x * b2.x) + (a23.y * b3.x + a45.x * b4.x + a45.y * b5.x);
  o.y = (a01.x * b0.y + a01.y * b1.y + a23.x * b2.y) + (a23.y * b3.y + a45.x * b4.y + a45.y * b5.y);
  return o;
}

// inverse of a symmetric positive definite 3 x 3 matrix m = (00, 01, 02, 11, 12, 22) by cofactors; false if not SPD
__device__ __forceinline__ bool inv3_spd(const double* m, double* o) {
  const double c00 = m[3] * m[5] - m[4] * m[4], c01 = m[2] * m[4] - m[1] * m[5], c02 = m[1] * m[4] - m[2] * m[3];
  const double det = m[0] * c00 + m[1] * c01 + m[2] * c02;
  const bool ok = det > 0.0 && m[0] > 0.0 && c00 > 0.0;
  const double id = 1.0 / (ok ? det : 1.0);
  o[0] = c00 * id; o[1] = c01 * id; o[2] = c02 * id;
  o[3] = (m[0] * m[5] - m[2] * m[2]) * id; o[4] = (m[1] * m[2] - m[0] * m[4]) * id;
  o[5] = (m[0] * m[3] - m[1] * m[1]) * id;
  return ok;
}

// entry (r, c) of a symmetric 3 x 3 matrix packed (00, 01, 02, 11, 12, 22), by selects (no local-memory indexing)
__device__ __forceinline__ double pick_sym3(const double* m, int r, int c) {
  const int lo = r < c ? r : c, hi = r < c ? c : r;
  const double row0 = hi == 0 ? m[0] : (hi == 1 ? m[1] : m[2]);
  const double row1 = hi == 1 ? m[3] : m[4];
  return lo == 0 ? row0 : (lo == 1 ? row1 : m[5]);
}

template <int H, class SM>
__device__ __noinline__ void riccati_factor(SM& sm) {
  const int lane = threadIdx.x & 31;   // one warp runs this routine (sm.solver_warp)
  // Lane roles (indices of lanes without the role are clamped to 0: every lane computes, only role lanes store --
  // predicated stores instead of divergent branches around each step)
  const bool l18 = lane < 18, l24 = lane < 24, l9 = lane < 9, l22 = lane >= 9 && lane < 18;
  const int r6 = l18 ? lane / 3 : 0, cp = l18 ? lane - 3 * (lane / 3) : 0;     // 6 x 6 products: row r6, columns 2 cp, 2 cp + 1
  const int k12 = l24 ? lane >> 1 : 0, ch = lane & 1;                           // 12 x 6 products: row k12, columns 3 ch ..
  const int gr = l9 ? lane / 3 : 0, gc = l9 ? lane - 3 * (lane / 3) : 0;        // 3 x 3 blocks 11 / 21 of Y^-1
  const int r22 = l22 ? (lane - 9) / 3 : 0, c22 = l22 ? (lane - 9) - 3 * ((lane - 9) / 3) : 0;   // block 22
  // the (k, l), l <= k, entries of the 12 x 12 lower triangle this lane updates in step 8 (78 entries, <= 3 per lane)
  int pk[3], pl[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const int e = lane + 32 * i;
    int k = 0;
    while ((k + 1) * (k + 2) / 2 <= e) ++k;
    pk[i] = e < 78 ? k : 0;
    pl[i] = e < 78 ? e - k * (k + 1) / 2 : 0;
  }
  // stage cost Q = blkdiag(K2, K1) at this lane's two (r6, c) pairs
  double qa[2], qc[2];
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const int c = 2 * cp + j;
    qa[j] = (r6 < 3 && c < 3) ? sm.k2ang[3 * r6 + c] : ((r6 == c && r6 >= 3) ? sm.k2lin[r6 - 3] : 0.0);
    qc[j] = r6 == c ? sm.k1[r6] : 0.0;
  }
  double* __restrict__ md = sm.m6[RM_D];
  double* __restrict__ ms = sm.m6[RM_S];
  double* __restrict__ mu = sm.m6[RM_U];
  double* __restrict__ my = sm.m6[RM_Y];
  double* __restrict__ myi = sm.m6[RM_YI];
  double* __restrict__ mg = sm.m6[RM_G];
  // P_h = Q, and from it the inputs of the first stage (t = H - 1):  PG = P Gam,  S = Gam^T P Gam,  D_t unpacked
  for (int e = lane; e < 144; e += 32) sm.pm[e] = 0.0;
  if (lane == 0) sm.flag = 0;
  __syncwarp();
  {
    double* __restrict__ pg = sm.fac_pg[H - 1];
    const double* __restrict__ nb = sm.nblk[H - 1];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int c = 2 * cp + j;
      if (l18) {
        sm.pm[12 * r6 + c] = qa[j];
        sm.pm[12 * (6 + r6) + 6 + c] = qc[j];
        pg[6 * r6 + c] = 0.5 * qa[j];
        pg[6 * (6 + r6) + c] = qc[j];
        ms[6 * r6 + c] = 0.25 * qa[j] + qc[j];
        md[6 * r6 + c] = r6 >= c ? nb[r6 * (r6 + 1) / 2 + c] : nb[c * (c + 1) / 2 + r6];
      }
    }
  }
  __syncwarp();
#pragma unroll 1
  for (int t = H - 1; t >= 0; --t) {
    double* __restrict__ pg = sm.fac_pg[t];
    // (2) U = D S
    {
      const double2 o = row_times_cols(md, ms, r6, cp);
      if (l18) *reinterpret_cast<double2*>(mu + 6 * r6 + 2 * cp) = o;
    }
    __syncwarp();
    // (3) Y = S + S U   (symmetric positive definite)
    {
      double2 o = row_times_cols(ms, mu, r6, cp);
      const double2 s0 = ldd2(ms + 6 * r6 + 2 * cp);
      o.x += s0.x; o.y += s0.y;
      if (l18) *reinterpret_cast<double2*>(my + 6 * r6 + 2 * cp) = o;
    }
    __syncwarp();
    // (4) Y^-1 by 3 x 3 blocks, Y = [[A, B^T], [B, C]]:  G = B A^-1,  Sc = C - G B^T,
    //     Y^-1 = [[A^-1 + G^T Sc^-1 G, -G^T Sc^-1], [-Sc^-1 G, Sc^-1]].   (4a) G (lanes 0..8), A^-1 in every lane
    double ai[6];
    bool ok;
    {
      const double am[6] = {my[0], my[6], my[12], my[7], my[13], my[14]};      // lower triangle of A
      ok = inv3_spd(am, ai);
      const double b0 = my[6 * (3 + gr)], b1 = my[6 * (3 + gr) + 1], b2 = my[6 * (3 + gr) + 2];   // row gr of B
      const double a0 = gc == 0 ? ai[0] : (gc == 1 ? ai[1] : ai[2]);
      const double a1 = gc == 0 ? ai[1] : (gc == 1 ? ai[3] : ai[4]);
      const double a2 = gc == 0 ? ai[2] : (gc == 1 ? ai[4] : ai[5]);
      const double g = b0 * a0 + b1 * a1 + b2 * a2;
      if (l9) mg[3 * gr + gc] = g;
    }
    __syncwarp();
    // (4b) Sc and Sc^-1 in every lane; lanes 0..8 write -Sc^-1 G (blocks 21 and 12), lanes 9..17 Sc^-1 (block 22)
    double sci[6];
    {
      double g[9], bm[9];
#pragma unroll
      for (int i = 0; i < 9; ++i) g[i] = mg[i];
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) bm[3 * r + c] = my[6 * (3 + r) + c];
      double scm[6];
      scm[0] = my[21] - (g[0] * bm[0] + g[1] * bm[1] + g[2] * bm[2]);
      scm[1] = my[27] - (g[0] * bm[3] + g[1] * bm[4] + g[2] * bm[5]);
      scm[2] = my[33] - (g[0] * bm[6] + g[1] * bm[7] + g[2] * bm[8]);
      scm[3] = my[28] - (g[3] * bm[3] + g[4] * bm[4] + g[5] * bm[5]);
      scm[4] = my[34] - (g[3] * bm[6] + g[4] * bm[7] + g[5] * bm[8]);
      scm[5] = my[35] - (g[6] * bm[6] + g[7] * bm[7] + g[8] * bm[8]);
      ok = inv3_spd(scm, sci) && ok;
      if (!ok && lane == 0) sm.flag = 1;
      const double s0 = gr == 0 ? sci[0] : (gr == 1 ? sci[1] : sci[2]);
      const double s1 = gr == 0 ? sci[1] : (gr == 1 ? sci[3] : sci[4]);
      const double s2 = gr == 0 ? sci[2] : (gr == 1 ? sci[4] : sci[5]);
      const double v21 = -(s0 * mg[gc] + s1 * mg[3 + gc] + s2 * mg[6 + gc]);   // -(Sc^-1 G)[gr][gc]
      const double v22 = pick_sym3(sci, r22, c22);
      if (l9) { myi[6 * (3 + gr) + gc] = v21; myi[6 * gc + 3 + gr] = v21; }
      if (l22) myi[6 * (3 + r22) + 3 + c22] = v22;
    }
    __syncwarp();
    // (4c) block 11: A^-1 - G^T Y21   (Y21 = -Sc^-1 G just written)
    {
      const double v11 = pick_sym3(ai, gr, gc) - (mg[gr] * myi[18 + gc] + mg[3 + gr] * myi[24 + gc] + mg[6 + gr] * myi[30 + gc]);
      if (l9) myi[6 * gr + gc] = v11;
    }
    __syncwarp();
    // (5) J = S Y^-1
    {
      const double2 o = row_times_cols(ms, myi, r6, cp);
      if (l18) *reinterpret_cast<double2*>(sm.fac_j[t] + 6 * r6 + 2 * cp) = o;
    }
    __syncwarp();
    // (6) N = D J
    {
      const double2 o = row_times_cols(md, sm.fac_j[t], r6, cp);
      if (l18) *reinterpret_cast<double2*>(sm.fac_n[t] + 6 * r6 + 2 * cp) = o;
    }
    if (t == 0) break;                       // P_0 is never needed: x_0 = 0
    __syncwarp();
    // (7) T1 = PG N   (12 x 6): lane (k12, ch) computes columns 3 ch .. 3 ch + 2 of row k12
    {
      const double* __restrict__ nn = sm.fac_n[t] + 3 * ch;
      const double2 p01 = ldd2(pg + 6 * k12), p23 = ldd2(pg + 6 * k12 + 2), p45 = ldd2(pg + 6 * k12 + 4);
      double v[3];
#pragma unroll
      for (int c = 0; c < 3; ++c)
        v[c] = (p01.x * nn[c] + p01.y * nn[6 + c] + p23.x * nn[12 + c]) + (p23.y * nn[18 + c] + p45.x * nn[24 + c] + p45.y * nn[30 + c]);
      if (l24) { sm.t1[6 * k12 + 3 * ch] = v[0]; sm.t1[6 * k12 + 3 * ch + 1] = v[1]; sm.t1[6 * k12 + 3 * ch + 2] = v[2]; }
    }
    __syncwarp();
    // (8) P' = P - T1 PG^T: lower triangle (78 entries, <= 3 per lane), mirrored into pm2
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const int k = pk[i], l = pl[i];
      const double2 t01 = ldd2(sm.t1 + 6 * k), t23 = ldd2(sm.t1 + 6 * k + 2), t45 = ldd2(sm.t1 + 6 * k + 4);
      const double2 g01 = ldd2(pg + 6 * l), g23 = ldd2(pg + 6 * l + 2), g45 = ldd2(pg + 6 * l + 4);
      const double v = sm.pm[12 * k + l] - ((t01.x * g01.x + t01.y * g01.y + t23.x * g23.x) + (t23.y * g23.y + t45.x * g45.x + t45.y * g45.y));
      if (lane + 32 * i < 78) { sm.pm2[12 * k + l] = v; sm.pm2[12 * l + k] = v; }
    }
    __syncwarp();
    // (9) P_t = Q + Phi^T P' Phi:  A_t = A' + K2,  B_t = A' + B',  C_t = A' + B' + B'^T + C' + K1 -- and, from the same
    //     four entries, the inputs of the next stage:  PG = P_t Gam,  S = Gam^T P_t Gam;  D_{t-1} unpacked
    {
      double* __restrict__ pgn = sm.fac_pg[t - 1];
      const double* __restrict__ nb = sm.nblk[t - 1];
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int r = r6, c = 2 * cp + j;
        const double a = sm.pm2[12 * r + c], bb = sm.pm2[12 * r + 6 + c], bt = sm.pm2[12 * c + 6 + r], cc = sm.pm2[12 * (6 + r) + 6 + c];
        const double at = a + qa[j], brc = a + bb, bcr = a + bt, ct = a + bb + bt + cc + qc[j];
        const double dv = r >= c ? nb[r * (r + 1) / 2 + c] : nb[c * (c + 1) / 2 + r];
        if (l18) {
          sm.pm[12 * r + c] = at;
          sm.pm[12 * r + 6 + c] = brc;
          sm.pm[12 * (6 + c) + r] = brc;
          sm.pm[12 * (6 + r) + 6 + c] = ct;
          pgn[6 * r + c] = 0.5 * at + brc;
          pgn[6 * (6 + r) + c] = 0.5 * bcr + ct;
          ms[6 * r + c] = 0.25 * at + 0.5 * (brc + bcr) + ct;
          md[6 * r + c] = dv;
        }
      }
    }
    __syncwarp();
  }
}

// ---- Psi v = b with the Riccati factors; b / v in sm.avec; executed by warp 0 only ------------------------------
// backward:  r_t = Gam^T (PG_t b_t + p_{t+1}),  w_t = b_t - N_t r_t,  p_t = Phi^T (p_{t+1} + PG_t w_t),  p_h = 0
// forward :  v_t = J_t (PG_t^T Phi x_t + r_t),  a_t = b_t - D_t v_t,  x_{t+1} = Phi x_t + Gam a_t,  x_0 = 0
// The 12-vectors p and x live in lanes 0..11 (pi part in lanes 0..5, sigma part in lanes 6..11), the 6-vectors in
// lanes 0..5; everything moves by warp shuffles: no barrier and no shared-memory round trip on the chain.
template <int H, class SM>
__device__ __noinline__ void riccati_solve(SM& sm) {
  const int lane = threadIdx.x & 31;   // one warp runs this routine (sm.solver_warp)
  const int k12 = lane < 12 ? lane : 0, c6 = lane < 6 ? lane : 0;
  // The 6- and 12-vectors a stage hands from one product to the next go through shared memory (one predicated store,
  // __syncwarp, 128-bit broadcast loads) instead of one shuffle pair per element and lane: a single warp issues an
  // instruction every ~4 cycles, and the shuffle version needed 95 / 192 instructions per backward / forward stage.
  double* __restrict__ bc6 = sm.t1;          // scratch of the factor sweep, free here: [0..5] w or y, [16..27] Phi x
  double p = 0.0;
#pragma unroll 1
  for (int t = H - 1; t >= 0; --t) {
    const double* __restrict__ pgk = sm.fac_pg[t] + 6 * k12;
    const double* __restrict__ bt = sm.avec + 6 * t;
    const double2 p01 = ldd2(pgk), p23 = ldd2(pgk + 2), p45 = ldd2(pgk + 4);
    const double2 b01 = ldd2(bt), b23 = ldd2(bt + 2), b45 = ldd2(bt + 4);
    const double z = (p01.x * b01.x + p01.y * b01.y + p23.x * b23.x) + (p23.y * b23.y + p45.x * b45.x + p45.y * b45.y) + p;   // (PG b + p)_k
    const double zs = __shfl_down_sync(kFull, z, 6);
    const double r = 0.5 * z + zs;                        // lanes 0..5: r_c = (Gam^T .)_c
    if (lane < 6) sm.rvec[6 * t + lane] = r;
    __syncwarp();
    const double* __restrict__ rt = sm.rvec + 6 * t;
    const double2 r01 = ldd2(rt), r23 = ldd2(rt + 2), r45 = ldd2(rt + 4);
    const double* __restrict__ nr = sm.fac_n[t] + 6 * c6;
    const double2 n01 = ldd2(nr), n23 = ldd2(nr + 2), n45 = ldd2(nr + 4);
    const double bc = c6 == 0 ? b01.x : (c6 == 1 ? b01.y : (c6 == 2 ? b23.x : (c6 == 3 ? b23.y : (c6 == 4 ? b45.x : b45.y))));
    const double w = bc - ((n01.x * r01.x + n01.y * r01.y + n23.x * r23.x) + (n23.y * r23.y + n45.x * r45.x + n45.y * r45.y));
    if (lane < 6) bc6[lane] = w;
    __syncwarp();
    const double2 w01 = ldd2(bc6), w23 = ldd2(bc6 + 2), w45 = ldd2(bc6 + 4);
    const double u = p + ((p01.x * w01.x + p01.y * w01.y + p23.x * w23.x) + (p23.y * w23.y + p45.x * w45.x + p45.y * w45.y));
    const double uu = __shfl_up_sync(kFull, u, 6);
    p = lane < 6 ? u : u + uu;                            // Phi^T: (u_pi; u_pi + u_sigma)
    __syncwarp();                                         // bc6 is rewritten by the next stage
  }
  // row c6 of the packed symmetric D_t: element offsets inside nblk[t], the same at every stage
  int doff[6];
#pragma unroll
  for (int j = 0; j < 6; ++j) doff[j] = c6 >= j ? tri(c6, j) : tri(j, c6);
  double x = 0.0;
#pragma unroll 1
  for (int t = 0; t < H; ++t) {
    const double* __restrict__ pgt = sm.fac_pg[t];
    const double xs = __shfl_down_sync(kFull, x, 6);
    const double zx = lane < 6 ? x + xs : x;              // Phi x = (pi + sigma; sigma)
    if (lane < 12) bc6[16 + lane] = zx;
    __syncwarp();
    double y0 = lane < 6 ? sm.rvec[6 * t + lane] : 0.0, y1 = 0.0, y2 = 0.0;
#pragma unroll
    for (int k = 0; k < 12; k += 6) {
      const double2 z01 = ldd2(bc6 + 16 + k), z23 = ldd2(bc6 + 18 + k), z45 = ldd2(bc6 + 20 + k);
      y0 = fma(pgt[6 * k + c6], z01.x, y0);       y1 = fma(pgt[6 * (k + 1) + c6], z01.y, y1);
      y2 = fma(pgt[6 * (k + 2) + c6], z23.x, y2); y0 = fma(pgt[6 * (k + 3) + c6], z23.y, y0);
      y1 = fma(pgt[6 * (k + 4) + c6], z45.x, y1); y2 = fma(pgt[6 * (k + 5) + c6], z45.y, y2);
    }
    const double y = y0 + (y1 + y2);
    if (lane < 6) bc6[lane] = y;
    __syncwarp();
    const double2 q01 = ldd2(bc6), q23 = ldd2(bc6 + 2), q45 = ldd2(bc6 + 4);
    const double* __restrict__ jr = sm.fac_j[t] + 6 * c6;
    const double2 j01 = ldd2(jr), j23 = ldd2(jr + 2), j45 = ldd2(jr + 4);
    const double v = (j01.x * q01.x + j01.y * q01.y + j23.x * q23.x) + (j23.y * q23.y + j45.x * q45.x + j45.y * q45.y);
    const double bc = lane < 6 ? sm.avec[6 * t + lane] : 0.0;   // every lane touches only the slots it writes itself
    __syncwarp();                                                // everybody has read y before v overwrites bc6[0..5]
    if (lane < 6) bc6[lane] = v;
    __syncwarp();
    const double2 v01 = ldd2(bc6), v23 = ldd2(bc6 + 2), v45 = ldd2(bc6 + 4);
    const double* __restrict__ nb = sm.nblk[t];
    const double a = bc - ((nb[doff[0]] * v01.x + nb[doff[1]] * v01.y + nb[doff[2]] * v23.x) +
                           (nb[doff[3]] * v23.y + nb[doff[4]] * v45.x + nb[doff[5]] * v45.y));
    const double as = __shfl_up_sync(kFull, a, 6);
    x = lane < 6 ? zx + 0.5 * a : x + as;                 // Phi x + Gam a
    if (lane < 6) sm.avec[6 * t + lane] = v;
    __syncwarp();                                         // bc6 is rewritten by the next stage
  }
}

// ---- the per-block 3x3 part --------------------------------------------------------------------
struct Block3 { double e00, e11, e22, e20, e21; };   // symmetric with e10 == 0; reused for E^-1

// E = 2 alpha I + sum_r D_r g_r g_r^T  ->  E^-1 via a cancellation-free Cholesky.
// g rows: (-1,0,mu0) (1,0,mu1) (0,-1,mu2) (0,1,mu3) (0,0,1).
__device__ __forceinline__ void block_inverse(const double* dd, const double* mu, double two_alpha, double* einv) {
  const double sx = dd[0] + dd[1] + two_alpha;
  const double sy = dd[2] + dd[3] + two_alpha;
  const double exz = -mu[0] * dd[0] + mu[1] * dd[1];
  const double eyz = -mu[2] * dd[2] + mu[3] * dd[3];
  // Schur complement of the z pivot, expanded so that every term is non-negative
  const double ms = mu[0] + mu[1], mt = mu[2] + mu[3];
  const double zz = two_alpha + dd[4] +
                    (dd[0] * dd[1] * ms * ms + two_alpha * (mu[0] * mu[0] * dd[0] + mu[1] * mu[1] * dd[1])) / sx +
                    (dd[2] * dd[3] * mt * mt + two_alpha * (mu[2] * mu[2] * dd[2] + mu[3] * mu[3] * dd[3])) / sy;
  // L = [[sqrt(sx),0,0],[0,sqrt(sy),0],[exz/sqrt(sx), eyz/sqrt(sy), sqrt(zz)]]
  // E^-1 = L^-T L^-1 with L^-1 = [[1/l00,0,0],[0,1/l11,0],[-l20/(l00 l22), -l21/(l11 l22), 1/l22]]
  const double izz = 1.0 / zz;
  const double ax = exz / sx, ay = eyz / sy;   // l20/l00, l21/l11
  // einv packed as (xx, yy, zz, xz, yz, xy)
  einv[0] = 1.0 / sx + ax * ax * izz;
  einv[1] = 1.0 / sy + ay * ay * izz;
  einv[2] = izz;
  einv[3] = -ax * izz;
  einv[4] = -ay * izz;
  einv[5] = ax * ay * izz;
}

__device__ __forceinline__ void sym3_mul(const double* m, const double* v, double* o) {
  // m packed as (xx, yy, zz, xz, yz, xy)
  o[0] = m[0] * v[0] + m[5] * v[1] + m[3] * v[2];
  o[1] = m[5] * v[0] + m[1] * v[1] + m[4] * v[2];
  o[2] = m[3] * v[0] + m[4] * v[1] + m[2] * v[2];
}

// G^T w for the 10 rows (upper 0..4, lower 5..9 with negated normals)
__device__ __forceinline__ void gt_mul(const double* w, const double* mu, double* o) {
  const double e0 = w[0] - w[5], e1 = w[1] - w[6], e2 = w[2] - w[7], e3 = w[3] - w[8], e4 = w[4] - w[9];
  o[0] = e1 - e0;
  o[1] = e3 - e2;
  o[2] = mu[0] * e0 + mu[1] * e1 + mu[2] * e2 + mu[3] * e3 + e4;
}

// c_r = g_r . f  (5 values)
__device__ __forceinline__ void g_mul(const double* f, const double* mu, double* c) {
  c[0] = -f[0] + mu[0] * f[2];
  c[1] = f[0] + mu[1] * f[2];
  c[2] = -f[1] + mu[2] * f[2];
  c[3] = f[1] + mu[3] * f[2];
  c[4] = f[2];
}

// ---- per-thread context of a "block" thread: one (time step, leg) force triple ---------------------
struct Blk {
  double ba[9];       // A_leg = I_world^-1 [r]x   (zero for inactive threads)
  double inv_mass;
  double two_alpha;
  int t, leg;
  bool is_blk, act;   // act: this thread's leg is in stance
};

// out = P u for the triple held by this thread, P = 2 alpha I + W^T K W.  All threads call.
template <int H>
__device__ __forceinline__ void apply_p(Smem<H>& sm, const RgMpcDev* __restrict__ ws, const Blk& b, const double* uu, double* out) {
  constexpr int N6 = Cfg<H>::N6;
  const int tid = threadIdx.x;
  double a6[6];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    a6[c] = b.ba[3 * c] * uu[0] + b.ba[3 * c + 1] * uu[1] + b.ba[3 * c + 2] * uu[2];
    a6[3 + c] = b.inv_mass * uu[c];
  }
#pragma unroll
  for (int c = 0; c < 6; ++c) a6[c] = quad_sum(b.act ? a6[c] : 0.0);
  if (b.is_blk && b.leg == 0) {
#pragma unroll
    for (int c = 0; c < 6; ++c) sm.avec[6 * b.t + c] = a6[c];
  }
  __syncthreads();
  for (int row = tid; row < N6; row += Cfg<H>::NT) {
    const int j = row / 6, c = row - 6 * j;
    double s1 = 0.0;
    for (int k = 0; k < H; ++k) s1 = fma(c1f(H, j, k), sm.avec[6 * k + c], s1);
    double val = sm.k1[c] * s1;
    if (c < 3) {
      double s20 = 0.0, s21 = 0.0, s22 = 0.0;
      for (int k = 0; k < H; ++k) {
        const double cc = ws->c2tab[j * H + k];
        s20 = fma(cc, sm.avec[6 * k + 0], s20);
        s21 = fma(cc, sm.avec[6 * k + 1], s21);
        s22 = fma(cc, sm.avec[6 * k + 2], s22);
      }
      val += sm.k2ang[3 * c] * s20 + sm.k2ang[3 * c + 1] * s21 + sm.k2ang[3 * c + 2] * s22;
    } else {
      double s2 = 0.0;
      for (int k = 0; k < H; ++k) s2 = fma(ws->c2tab[j * H + k], sm.avec[6 * k + c], s2);
      val += sm.k2lin[c - 3] * s2;
    }
    sm.kvec[row] = val;
  }
  __syncthreads();
  if (b.act) {
    const double* kv = sm.kvec + 6 * b.t;
#pragma unroll
    for (int d = 0; d < 3; ++d)
      out[d] = b.two_alpha * uu[d] + b.ba[d] * kv[0] + b.ba[3 + d] * kv[1] + b.ba[6 + d] * kv[2] + b.inv_mass * kv[3 + d];
  } else {
    out[0] = out[1] = out[2] = 0.0;
  }
}

// Psi = K^-1 + sum_legs B M B^T (M = per-block symmetric 3x3, packed xx,yy,zz,xz,yz,xy), then its
// Cholesky factor.  All threads call.
template <int H>
// t_begin (even): time blocks before it are unchanged since the previous factorisation, whose leading
// 6 t_begin columns are reused (6 t_begin is a multiple of the Cholesky panel width).
__device__ __forceinline__ void factor_psi(Smem<H>& sm, const RgMpcDev* __restrict__ ws, const Blk& b, const double* m, int t_begin = 0) {
  RG_TIC();
  double am[9];   // A M
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const double a0 = b.ba[3 * a], a1 = b.ba[3 * a + 1], a2 = b.ba[3 * a + 2];
    am[3 * a + 0] = a0 * m[0] + a1 * m[5] + a2 * m[3];
    am[3 * a + 1] = a0 * m[5] + a1 * m[1] + a2 * m[4];
    am[3 * a + 2] = a0 * m[3] + a1 * m[4] + a2 * m[2];
  }
  double n[21];   // lower triangle of the 6x6 block [[A M A^T, .],[M A^T / m, M / m^2]], row-major
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c <= r; ++c)
      n[r * (r + 1) / 2 + c] = am[3 * r] * b.ba[3 * c] + am[3 * r + 1] * b.ba[3 * c + 1] + am[3 * r + 2] * b.ba[3 * c + 2];
  const double mfull[9] = {m[0], m[5], m[3], m[5], m[1], m[4], m[3], m[4], m[2]};
#pragma unroll
  for (int r = 3; r < 6; ++r) {
#pragma unroll
    for (int c = 0; c < 3; ++c) n[r * (r + 1) / 2 + c] = am[3 * c + (r - 3)] * b.inv_mass;
#pragma unroll
    for (int c = 3; c <= r; ++c) n[r * (r + 1) / 2 + c] = mfull[3 * (r - 3) + (c - 3)] * b.inv_mass * b.inv_mass;
  }
#pragma unroll
  for (int i = 0; i < 21; ++i) n[i] = quad_sum(b.act ? n[i] : 0.0);
  if (b.is_blk && b.leg == 0) {
#pragma unroll
    for (int i = 0; i < 21; ++i) sm.nblk[b.t][i] = n[i];
  }
  __syncthreads();
  RG_TOC(12);
  if constexpr (Cfg<H>::RICCATI) {
    if ((int)(threadIdx.x >> 5) == sm.solver_warp) riccati_factor<H>(sm);      // the backward sweep has no reusable prefix: t_begin is not used
    __syncthreads();
  } else {
    psi_build_rows<H>(sm, ws, t_begin);
    __syncthreads();
    RG_TOC(10);
    cholesky_rows<H>(sm, 6 * t_begin);
  }
  RG_TOC(11);
}

// First half of x = (E + W^T K W)^-1 rhs through the Woodbury identity: given the per-block E^-1
// (packed) and the factor of Psi = K^-1 + W E^-1 W^T it returns  b' = rhs - W^T v,
// v = Psi^-1 W E^-1 rhs; the caller finishes with the block solve x = E^-1 b'.  All threads call.
template <int H>
__device__ __forceinline__ void woodbury_solve(Smem<H>& sm, const Blk& b, const double* einv, const double* rhs, double* bprime) {
  double w[3];
  sym3_mul(einv, rhs, w);   // E^-1 rhs
  double t6[6];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    t6[c] = b.ba[3 * c] * w[0] + b.ba[3 * c + 1] * w[1] + b.ba[3 * c + 2] * w[2];
    t6[3 + c] = b.inv_mass * w[c];
  }
#pragma unroll
  for (int c = 0; c < 6; ++c) t6[c] = quad_sum(b.act ? t6[c] : 0.0);
  if (b.is_blk && b.leg == 0) {
#pragma unroll
    for (int c = 0; c < 6; ++c) sm.avec[6 * b.t + c] = t6[c];
  }
  __syncthreads();
  if ((int)(threadIdx.x >> 5) == sm.solver_warp) {
    if constexpr (Cfg<H>::RICCATI) riccati_solve<H>(sm);
    else tri_solve_warp0<H>(sm);
  }
  __syncthreads();
  if (b.act) {
    const double* v = sm.avec + 6 * b.t;
#pragma unroll
    for (int d = 0; d < 3; ++d)
      bprime[d] = rhs[d] - (b.ba[d] * v[0] + b.ba[3 + d] * v[1] + b.ba[6 + d] * v[2] + b.inv_mass * v[3 + d]);
  } else {
    bprime[0] = bprime[1] = bprime[2] = 0.0;
  }
  __syncthreads();   // avec is reused by the next caller
}

// ---- accurate block solve for the interior point -------------------------------------------------
// E = 2 alpha I + sum_r D_r g_r g_r^T.  Solving E dx = b' with an explicit 3x3 inverse loses the
// constraint-space products c_r = g_r . dx of strongly active rows (D_r ~ 1e10) to cancellation,
// and those are exactly what the slack update ds = -/+ c needs.  The 5x5 form
//     S z = G b',  S = 2 alpha D^-1 + G G^T,   c = D^-1 z,   dx = (b' - G^T z) / (2 alpha)
// delivers c without cancellation (DESIGN.md 3.5).  chol5 factors S in registers.
struct Chol5 { double l[15]; };   // lower triangle, row-major; diagonal entries hold 1 / L[i][i]

__device__ __forceinline__ void chol5_factor(const double* mu, const double* inv_d, double two_alpha, Chol5& c) {
  // Gram matrix of the rows (-1,0,mu0) (1,0,mu1) (0,-1,mu2) (0,1,mu3) (0,0,1)
  double a[15];
  a[0] = 1.0 + mu[0] * mu[0];
  a[1] = -1.0 + mu[0] * mu[1]; a[2] = 1.0 + mu[1] * mu[1];
  a[3] = mu[0] * mu[2]; a[4] = mu[1] * mu[2]; a[5] = 1.0 + mu[2] * mu[2];
  a[6] = mu[0] * mu[3]; a[7] = mu[1] * mu[3]; a[8] = -1.0 + mu[2] * mu[3]; a[9] = 1.0 + mu[3] * mu[3];
  a[10] = mu[0]; a[11] = mu[1]; a[12] = mu[2]; a[13] = mu[3]; a[14] = 1.0;
#pragma unroll
  for (int i = 0; i < 5; ++i) a[i * (i + 1) / 2 + i] += two_alpha * inv_d[i];
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    double d = a[j * (j + 1) / 2 + j];
#pragma unroll
    for (int k = 0; k < j; ++k) d = fma(-c.l[j * (j + 1) / 2 + k], c.l[j * (j + 1) / 2 + k], d);
    const double r = rsqrt(fmax(d, 1e-300));
    c.l[j * (j + 1) / 2 + j] = r;
#pragma unroll
    for (int i = j + 1; i < 5; ++i) {
      double v = a[i * (i + 1) / 2 + j];
#pragma unroll
      for (int k = 0; k < j; ++k) v = fma(-c.l[i * (i + 1) / 2 + k], c.l[j * (j + 1) / 2 + k], v);
      c.l[i * (i + 1) / 2 + j] = v * r;
    }
  }
}

// z = S^-1 (G b'), c5 = D^-1 z (= G dx), dx = (b' - G^T z) / (2 alpha)
__device__ __forceinline__ void chol5_block_solve(const Chol5& c, const double* mu, const double* inv_d, double two_alpha,
                                                  const double* bprime, double* dx, double* c5) {
  double z[5];
  g_mul(bprime, mu, z);
#pragma unroll
  for (int i = 0; i < 5; ++i) {
#pragma unroll
    for (int k = 0; k < i; ++k) z[i] = fma(-c.l[i * (i + 1) / 2 + k], z[k], z[i]);
    z[i] *= c.l[i * (i + 1) / 2 + i];
  }
#pragma unroll
  for (int i = 4; i >= 0; --i) {
#pragma unroll
    for (int k = i + 1; k < 5; ++k) z[i] = fma(-c.l[k * (k + 1) / 2 + i], z[k], z[i]);
    z[i] *= c.l[i * (i + 1) / 2 + i];
  }
  const double inv2a = 1.0 / two_alpha;
  dx[0] = (bprime[0] - (z[1] - z[0])) * inv2a;
  dx[1] = (bprime[1] - (z[3] - z[2])) * inv2a;
  dx[2] = (bprime[2] - (mu[0] * z[0] + mu[1] * z[1] + mu[2] * z[2] + mu[3] * z[3] + z[4])) * inv2a;
#pragma unroll
  for (int i = 0; i < 5; ++i) c5[i] = z[i] * inv_d[i];
}

// Orthonormal basis of the active normals of one (step, leg) block (Gram-Schmidt in bit order, at most three rows):
//   a_i = sum_k rr[k][i] e_k,  targets bt_i,  row ids;  dependent normals and rows beyond the third are cleared from act.
// Everything lives in named registers (slot 0 / 1 / 2 chosen by predication): indexing small arrays with the run-time
// count put them into a 480-byte local-memory frame per thread whose write-back was most of the kernel's DRAM traffic.
// Built twice per round from the same bit mask -- before the factorisation (particular solution, projector) and in the
// verification (multipliers) -- instead of being kept live across the heavy phases: 21 doubles fewer in flight.
struct BlockBasis {
  double e0[3], e1[3], e2[3];
  double ir00, r01, r02, ir11, r12, ir22;   // the triangular factor's diagonal is kept as its reciprocals (only ever divided by)
  double bt0, bt1, bt2;
  int row0, row1, row2, na;
};

__device__ __forceinline__ void build_basis(unsigned& act, bool active_blk, const double* mu, const double* hv_up, const double* lo_b,
                                            BlockBasis& B) {
#pragma unroll
  for (int d = 0; d < 3; ++d) { B.e0[d] = 0.0; B.e1[d] = 0.0; B.e2[d] = 0.0; }
  B.ir00 = 1.0; B.r01 = 0.0; B.r02 = 0.0; B.ir11 = 1.0; B.r12 = 0.0; B.ir22 = 1.0;
  B.bt0 = B.bt1 = B.bt2 = 0.0;
  B.row0 = B.row1 = B.row2 = -1;
  B.na = 0;
  // One Gram-Schmidt body, run once per set bit (in bit order) until three independent rows are held: an unrolled scan
  // of the ten rows was 1300 instructions of code for the same handful of executed steps.
  unsigned bits = active_blk ? (act & 0x3ffu) : 0u;
#pragma unroll 1
  while (bits != 0u && B.na < 3) {
    const int r = __ffs((int)bits) - 1;
    bits &= bits - 1u;
    const int rw = r < 5 ? r : r - 5;
    double a0 = rw == 0 ? -1.0 : (rw == 1 ? 1.0 : 0.0), a1 = rw == 2 ? -1.0 : (rw == 3 ? 1.0 : 0.0);
    double a2 = rw == 0 ? mu[0] : (rw == 1 ? mu[1] : (rw == 2 ? mu[2] : (rw == 3 ? mu[3] : 1.0)));
    const double target = r < 5 ? (rw < 4 ? hv_up[0] : hv_up[4]) : (rw < 4 ? lo_b[0] : lo_b[4]);   // the four cone rows share their bounds
    const double c0 = B.na > 0 ? a0 * B.e0[0] + a1 * B.e0[1] + a2 * B.e0[2] : 0.0;
    a0 -= c0 * B.e0[0]; a1 -= c0 * B.e0[1]; a2 -= c0 * B.e0[2];
    const double c1 = B.na > 1 ? a0 * B.e1[0] + a1 * B.e1[1] + a2 * B.e1[2] : 0.0;
    a0 -= c1 * B.e1[0]; a1 -= c1 * B.e1[1]; a2 -= c1 * B.e1[2];
    const double n2 = a0 * a0 + a1 * a1 + a2 * a2;
    if (n2 < 1e-18) {
      act &= ~(1u << r);                                               // dependent normal: drop
    } else {
      const double inrm = rsqrt_pivot(n2);   // 1 / |a|: scales the basis vector and IS the reciprocal diagonal entry
      if (B.na == 0) { B.e0[0] = a0 * inrm; B.e0[1] = a1 * inrm; B.e0[2] = a2 * inrm; B.ir00 = inrm; B.bt0 = target; B.row0 = r; }
      else if (B.na == 1) { B.e1[0] = a0 * inrm; B.e1[1] = a1 * inrm; B.e1[2] = a2 * inrm; B.r01 = c0; B.ir11 = inrm; B.bt1 = target; B.row1 = r; }
      else { B.e2[0] = a0 * inrm; B.e2[1] = a1 * inrm; B.e2[2] = a2 * inrm; B.r02 = c0; B.r12 = c1; B.ir22 = inrm; B.bt2 = target; B.row2 = r; }
      ++B.na;
    }
  }
  // rows beyond the third independent one cannot be held: drop them from the guess
  unsigned keep = 0u;
  if (B.row0 >= 0) keep |= 1u << B.row0;
  if (B.row1 >= 0) keep |= 1u << B.row1;
  if (B.row2 >= 0) keep |= 1u << B.row2;
  act &= keep;
}

// Inverse of an env's 3x3 body inertia (row major) by cofactors, the formula and the rounding of the host's inv3
// (rg_api.cu): no contracted multiply-adds, one IEEE division -- a row equal to the workspace's inertia gives the
// workspace's inverse bit for bit.  The caller has checked |det| >= 1e-300.
__device__ __forceinline__ void env_inv3(const double* __restrict__ m, double* o) {
  const double c00 = __dsub_rn(__dmul_rn(m[4], m[8]), __dmul_rn(m[5], m[7]));
  const double c01 = __dsub_rn(__dmul_rn(m[5], m[6]), __dmul_rn(m[3], m[8]));
  const double c02 = __dsub_rn(__dmul_rn(m[3], m[7]), __dmul_rn(m[4], m[6]));
  const double det = __dadd_rn(__dadd_rn(__dmul_rn(m[0], c00), __dmul_rn(m[1], c01)), __dmul_rn(m[2], c02));
  const double id = 1.0 / det;
  o[0] = __dmul_rn(c00, id);
  o[1] = __dmul_rn(__dsub_rn(__dmul_rn(m[2], m[7]), __dmul_rn(m[1], m[8])), id);
  o[2] = __dmul_rn(__dsub_rn(__dmul_rn(m[1], m[5]), __dmul_rn(m[2], m[4])), id);
  o[3] = __dmul_rn(c01, id);
  o[4] = __dmul_rn(__dsub_rn(__dmul_rn(m[0], m[8]), __dmul_rn(m[2], m[6])), id);
  o[5] = __dmul_rn(__dsub_rn(__dmul_rn(m[2], m[3]), __dmul_rn(m[0], m[5])), id);
  o[6] = __dmul_rn(c02, id);
  o[7] = __dmul_rn(__dsub_rn(__dmul_rn(m[1], m[6]), __dmul_rn(m[0], m[7])), id);
  o[8] = __dmul_rn(__dsub_rn(__dmul_rn(m[0], m[4]), __dmul_rn(m[1], m[3])), id);
}

// number of stance legs (nonzero bytes) in a 4-byte contact word
__device__ __forceinline__ int stance_count(const unsigned w) {
  return (int)((w & 0xffu) != 0) + (int)((w & 0xff00u) != 0) + (int)((w & 0xff0000u) != 0) + (int)((w & 0xff000000u) != 0);
}

// One env's stance QP, executed by the whole CTA.
// LEAN = true : the verified active-set rounds only -- no interior-point state or code (the registers that frees
//               are most of the kernel's local-memory frame).  An env whose rounds do not verify within the
//               cold-start budget is appended to the fallback queue and gets no output from this call.
// LEAN = false: the complete solver (cold start unless skip_cold, interior point, escalation ladder).
// ENV_MODEL = true: mass, inertia and friction coefficients come from the env's row of `model` where its array is not
//               NULL (rg_mpc_env_model).  A compile-time flag, so that the model-free instantiations -- whose schedule
//               was tuned instruction by instruction (DESIGN.md 3.10-3.11) -- carry none of its code (DESIGN.md 3.12).
// PLAN = true : the stance of block (t, leg) comes from byte `leg` of row t of the env's contact schedule `plan`
//               ([N,h,4], rg_mpc_build_solve_schedule) instead of one contact word held over the horizon; the com
//               height is taken over the stance feet of row 0, or of the first row that has one (DESIGN.md 3.15).
// FEET = true (with PLAN): the lever arm of block (t, leg) is foot `leg` of row t of the env's foothold plan `feet`
//               ([N,h,12], rg_mpc_build_solve_footholds) instead of the current foot at every step, and the com height
//               is taken over the stance feet of the same row r* the schedule names (DESIGN.md 3.16).
template <int H, bool LEAN, bool ENV_MODEL, bool PLAN = false, bool FEET = false>
__device__ __forceinline__ void solve_env(Smem<H>& sm, const RgMpcDev* __restrict__ ws, RgMpcScratch* __restrict__ scratch,
                                          const int env, const bool skip_cold,
                                          const rg_mpc_io& io, const rg_mpc_env_model& model,
                                          const uint8_t* __restrict__ plan = nullptr,
                                          const float* __restrict__ feet = nullptr) {
  using C = Cfg<H>;
  const float* __restrict__ g_com_vel = io.com_velocity_body;
  const float* __restrict__ g_rpy = io.base_rpy;
  const float* __restrict__ g_rpy_rate = io.base_rpy_rate;
  const uint8_t* __restrict__ g_contacts = io.foot_contact_state;
  const float* __restrict__ g_feet = io.foot_positions_base;
  const float* __restrict__ g_cmd = io.command;
  const float* __restrict__ g_com_height = io.com_height;
  const int zero_yaw = io.zero_yaw;
  float* __restrict__ g_forces = io.contact_forces;
  float* __restrict__ g_hforces = io.horizon_forces;
  double* __restrict__ g_hforces64 = io.horizon_forces_f64;
  int32_t* __restrict__ g_info = io.solve_info;
  uint16_t* __restrict__ g_active = io.active_set_io;
  constexpr int N6 = C::N6;
  const int tid = threadIdx.x;
#ifdef RG_DEBUG_TRACE
  const long long rg_tstart_ = clock64();
  // timeline mode (trace env == -2): per-CTA start / end in ns and the SM id, 4 doubles per env after slot 1024
  if (g_trace && g_trace_env == -2 && tid == 0) {
    unsigned long long ns; unsigned smid;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    g_trace[1024 + 4 * env] = (double)ns; g_trace[1024 + 4 * env + 2] = (double)smid;
  }
#endif
  const int t_blk = tid >> 2, leg = tid & 3;
  const bool is_blk = tid < C::NB;
#ifdef RG_DEBUG_POISON_SMEM
  // debug builds: overwrite this CTA's shared memory with a byte pattern before the env is solved, so that a read of
  // a value left by the previous env on the SM shows up as a result that depends on the pattern
  for (size_t i = tid; i < sizeof(Smem<H>); i += blockDim.x) reinterpret_cast<unsigned char*>(&sm)[i] = (unsigned char)(RG_DEBUG_POISON_SMEM);
  __syncthreads();
#endif

  // the host record of this workspace may be stale (memory reused without rg_mpc_release): never index the
  // tables with the wrong horizon
  if (ws->magic != RG_WS_MAGIC_MPC || ws->horizon != H) {
    for (int i = tid; i < 12; i += blockDim.x) g_forces[12 * (size_t)env + i] = 0.f;
    if (g_hforces) for (int i = tid; i < 12 * H; i += blockDim.x) g_hforces[12 * H * (size_t)env + i] = 0.f;
    if (g_hforces64) for (int i = tid; i < 12 * H; i += blockDim.x) g_hforces64[12 * H * (size_t)env + i] = 0.0;
    if (g_info && tid < 4) g_info[4 * (size_t)env + tid] = tid == RG_INFO_STATUS ? RG_STATUS_BAD_WORKSPACE : 0;
    return;
  }

  // ---------------------------------------------------------------- parameters (uniform loads)
  const double dt = ws->dt, two_alpha = 2.0 * ws->alpha;
  double inv_mass = ws->inv_mass;
  double fzmax = ws->fz_max, fzmin = ws->fz_min;
  double mu[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) mu[r] = ws->mu[r];
  // per-env model: every thread loads the env's mass and friction row (one address across the CTA: a broadcast) --
  // all of them use 1/m, the bounds and mu; the inertia is read by the lever-arm threads (tid < 4) only, except for
  // the determinant every thread takes here so that the validity test is uniform over the CTA without a barrier.
  // The bounds scale by mass_e / mass: exactly the workspace's bounds when the env's mass is the workspace's.
  bool model_ok = true;
  if constexpr (ENV_MODEL) {
    if (model.mass) {
      const double m = model.mass[env];
      model_ok = m > 0.0 && m <= 1.79769313486231570e308;   // > 0 and finite (NaN fails both)
      inv_mass = 1.0 / m;
      const double scale = m / ws->mass;
      fzmax *= scale;
      fzmin *= scale;
    }
    if (model.friction_coeffs) {
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        mu[r] = model.friction_coeffs[4 * (size_t)env + r];
        model_ok = model_ok && mu[r] > 0.0;
      }
    }
    if (model.inertia) {
      const double* __restrict__ in = model.inertia + 9 * (size_t)env;
      double fin = 0.0;
#pragma unroll
      for (int i = 0; i < 9; ++i) fin += in[i] * 0.0;      // NaN unless all nine are finite
      const double det = in[0] * (in[4] * in[8] - in[5] * in[7]) + in[1] * (in[5] * in[6] - in[3] * in[8]) +
                         in[2] * (in[3] * in[7] - in[4] * in[6]);
      model_ok = model_ok && fin == 0.0 && fabs(det) >= 1e-300;
    }
  }
  const double big_u = (mu[0] + 1.0) * fzmax;

  // ---------------------------------------------------------------- per-env inputs
  // every load is issued here, before anything depends on one of them: one DRAM latency, not four
  // PLAN: every thread reads the env's h row words (one address across the CTA: broadcasts) for the schedule-wide
  // quantities -- the number of stance blocks and the first non-empty row -- and its own block's row word
  unsigned contact_word = 0u, row_word = 0u;
  int plan_blocks = 0, r_star = 0;   // FEET: r_star = the row contact_word comes from
  if constexpr (PLAN) {
    const unsigned* __restrict__ rows = reinterpret_cast<const unsigned*>(plan + 4 * (size_t)H * env);
#pragma unroll
    for (int k = 0; k < H; ++k) {
      const unsigned w = rows[k];
      if (contact_word == 0u) {
        contact_word = w;
        if constexpr (FEET) r_star = k;
      }
      plan_blocks += stance_count(w);
    }
    if (is_blk) row_word = rows[t_blk];
  } else {
    contact_word = *reinterpret_cast<const unsigned*>(g_contacts + 4 * (size_t)env);
  }
  // The attitude, the feet, the rates and the command are consumed by threads of warp 0 only (setup_warp below): the
  // other warps do not load them.  The twelve foot coordinates of an env are 48 contiguous, 16-byte aligned bytes:
  // three 128-bit loads.
  float in_roll = 0.f, in_pitch = 0.f, in_yaw = 0.f, in_com_h = 0.f;
  float in_feet[12] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float in_w[3] = {0.f, 0.f, 0.f}, in_v[3] = {0.f, 0.f, 0.f}, in_cmd[3] = {0.f, 0.f, 0.f};
  // FEET: every block thread loads its own foot of its own row, consumed by itself alone (per-block constants below);
  // the entries of swing blocks are loaded but never used
  float blk_foot[3] = {0.f, 0.f, 0.f};
  if constexpr (FEET) {
    if (is_blk) {
      const float* __restrict__ bf = feet + 12 * ((size_t)H * env + t_blk) + 3 * leg;
      blk_foot[0] = bf[0]; blk_foot[1] = bf[1]; blk_foot[2] = bf[2];
    }
  }
  if (tid < 32) {
    in_roll = g_rpy[3 * (size_t)env + 0]; in_pitch = g_rpy[3 * (size_t)env + 1]; in_yaw = g_rpy[3 * (size_t)env + 2];
    // FEET: the feet of row 0 of the plan, issued with the other loads; reloaded from row r* when the schedule's first
    // stance row is a later one (their only use is the com height)
    const float4* __restrict__ f4 = reinterpret_cast<const float4*>(FEET ? feet + 12 * (size_t)H * env : g_feet + 12 * (size_t)env);
    float4 fa = f4[0], fb = f4[1], fc = f4[2];
    if constexpr (FEET) {
      if (r_star != 0) { fa = f4[3 * r_star]; fb = f4[3 * r_star + 1]; fc = f4[3 * r_star + 2]; }
    }
    in_feet[0] = fa.x; in_feet[1] = fa.y; in_feet[2] = fa.z; in_feet[3] = fa.w;
    in_feet[4] = fb.x; in_feet[5] = fb.y; in_feet[6] = fb.z; in_feet[7] = fb.w;
    in_feet[8] = fc.x; in_feet[9] = fc.y; in_feet[10] = fc.z; in_feet[11] = fc.w;
    if (g_com_height) in_com_h = g_com_height[env];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      in_w[a] = g_rpy_rate[3 * (size_t)env + a];
      in_v[a] = g_com_vel[3 * (size_t)env + a];
      in_cmd[a] = g_cmd[3 * (size_t)env + a];
    }
  }
  const unsigned warm_act = (g_active && is_blk) ? (unsigned)g_active[(size_t)env * C::NB + tid] : (unsigned)RG_ACTIVE_SET_UNKNOWN;
  // stage the rank-h weights of K^-1 (host table) in the Psi buffer, which is free until the first factorisation
  if constexpr (!C::RICCATI) {
    for (int i = tid; i < H * (H + 1) / 2 * H; i += blockDim.x) sm.psi[i] = ws->eig_uu[i];
  }
  const bool stance_leg[4] = {(contact_word & 0xffu) != 0, (contact_word & 0xff00u) != 0,
                              (contact_word & 0xff0000u) != 0, (contact_word & 0xff000000u) != 0};
  const int n_stance = (int)stance_leg[0] + stance_leg[1] + stance_leg[2] + stance_leg[3];
  // stance legs of this block's own horizon step (= n_stance without a schedule)
  const int n_step = PLAN ? stance_count(row_word) : n_stance;
  const bool active_blk = is_blk && (((PLAN ? row_word : contact_word) >> (8 * leg)) & 0xffu) != 0;

  if constexpr (ENV_MODEL) {
    if (!model_ok) {     // this env's model row fails the rg_mpc_setup checks: nothing is solved
      for (int i = tid; i < 12; i += blockDim.x) g_forces[12 * (size_t)env + i] = 0.f;
      if (g_hforces) for (int i = tid; i < 12 * H; i += blockDim.x) g_hforces[12 * H * (size_t)env + i] = 0.f;
      if (g_hforces64) for (int i = tid; i < 12 * H; i += blockDim.x) g_hforces64[12 * H * (size_t)env + i] = 0.0;
      if (g_info && tid < 4) g_info[4 * (size_t)env + tid] = tid == RG_INFO_STATUS ? RG_STATUS_BAD_MODEL : 0;
      if (g_active && is_blk) g_active[(size_t)env * C::NB + tid] = RG_ACTIVE_SET_UNKNOWN;
      return;
    }
  }
  if (PLAN ? plan_blocks == 0 : n_stance == 0) {   // every force pinned to zero by the bounds
    for (int i = tid; i < 12; i += blockDim.x) g_forces[12 * (size_t)env + i] = 0.f;
    if (g_hforces) for (int i = tid; i < 12 * H; i += blockDim.x) g_hforces[12 * H * (size_t)env + i] = 0.f;
    if (g_hforces64) for (int i = tid; i < 12 * H; i += blockDim.x) g_hforces64[12 * H * (size_t)env + i] = 0.0;
    if (g_info && tid < 4) g_info[4 * (size_t)env + tid] = tid == RG_INFO_STATUS ? (RG_STATUS_NO_STANCE | RG_STATUS_POLISHED) : 0;
    if (g_active && is_blk) g_active[(size_t)env * C::NB + tid] = RG_ACTIVE_SET_UNKNOWN;
    return;
  }

  RG_TIC();
  const double roll = in_roll, pitch = in_pitch, yaw = zero_yaw ? 0.0 : (double)in_yaw;
  // Everything derived from the attitude (trigonometry, T(rpy), lever arms, I_w^-1) is consumed by threads of warp 0
  // only (tid < 9 / 4 / H): the other warps skip the computation -- a warp pays for an instruction whether one lane
  // needs the result or all of them.
  const bool setup_warp = tid < 32;
  double sr = 0.0, cr = 1.0, sp = 0.0, cp = 1.0, sy = 0.0, cy = 1.0;
  if (setup_warp) {
    // one sincos call: lanes 0 / 1 / 2 take roll / pitch / yaw, the six results are broadcast
    double sn, cs;
    sincos(tid == 0 ? roll : (tid == 1 ? pitch : yaw), &sn, &cs);
    sr = __shfl_sync(kFull, sn, 0); cr = __shfl_sync(kFull, cs, 0);
    sp = __shfl_sync(kFull, sn, 1); cp = __shfl_sync(kFull, cs, 1);
    sy = __shfl_sync(kFull, sn, 2); cy = __shfl_sync(kFull, cs, 2);
  }

  // ---------------------------------------------------------------- setup (thread 0..; tiny)
  if (tid == 0) {
    sm.flag = 0;
    // The triangular / Riccati sweeps are executed by ONE warp of the CTA.  Warp slots map onto the four SM
    // sub-partitions by (slot mod 4), and the first warp of every CTA lands on the same one or two of them: with
    // "warp 0 sweeps" all resident envs would queue their serial phases on one scheduler.  Rotate the choice with
    // the CTA's position among the SM's warp slots so that the sweeps of co-resident envs spread over all four.
    unsigned slot;
    asm volatile("mov.u32 %0, %%warpid;" : "=r"(slot));
    const unsigned group = slot / C::NW;
    sm.solver_warp = C::NW >= 4 ? (int)(group % C::NW) : (C::NW == 2 ? (int)((group >> 1) & 1u) : 0);
  }

  RG_TOC(40);
  // T(rpy): angular velocity -> rpy rate;  K2_ang = 2 dt^4 T^T diag(w_rpy) T
  double tm[9] = {1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0};
  if (setup_warp) {
    const double icp = 1.0 / cp;
    tm[0] = cy * icp; tm[1] = sy * icp; tm[3] = -sy; tm[4] = cy; tm[6] = cy * sp * icp; tm[7] = sy * sp * icp;
  }
  const double dt2 = dt * dt, dt4 = dt2 * dt2;
  if (tid < 9) {
    const int c = tid / 3, d = tid % 3;
    double v = 0.0;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      // columns c and d of T by selects (a run-time index would put tm[] into local memory)
      const double tc = c == 0 ? tm[3 * r] : (c == 1 ? tm[3 * r + 1] : tm[3 * r + 2]);
      const double td = d == 0 ? tm[3 * r] : (d == 1 ? tm[3 * r + 1] : tm[3 * r + 2]);
      v += ws->w_rho[r] * tc * td;
    }
    sm.k2ang[tid] = 2.0 * dt4 * v;
  }
  if (tid < 6) sm.k1[tid] = 2.0 * dt2 * ws->w_nu[tid];
  if (tid < 3) sm.k2lin[tid] = 2.0 * dt4 * ws->w_rho[3 + tid];

  // foot lever arms in the (yaw aligned) world frame: R = Rx Ry Rz (sic, see oracle/convex_mpc.py)
  // R_body = Rz Ry Rx for the inertia
  double com_z = 0.0;
  if (setup_warp) {
    const double rf[9] = {cp * cy, -cp * sy, sp,
                          sr * sp * cy + cr * sy, -sr * sp * sy + cr * cy, -sr * cp,
                          -cr * sp * cy + sr * sy, cr * sp * sy + sr * cy, cr * cp};
    double zsum = 0.0;
    double fw[4][3];
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      const double px = in_feet[3 * l], py = in_feet[3 * l + 1], pz = in_feet[3 * l + 2];
#pragma unroll
      for (int r = 0; r < 3; ++r) fw[l][r] = rf[3 * r] * px + rf[3 * r + 1] * py + rf[3 * r + 2] * pz;
      if (stance_leg[l]) zsum += fw[l][2];
    }
    com_z = g_com_height ? (double)in_com_h : fabs(zsum / n_stance);
    // FEET: thread 0 publishes rf and I_w^-1 (18 doubles, in the storage of sm.bang) for the block threads, which form
    // their own lever-arm products after the barrier below
    if (tid < (FEET ? 1 : 4)) {
      const double rb[9] = {cy * cp, cy * sp * sr - sy * cr, cy * sp * cr + sy * sr,
                            sy * cp, sy * sp * sr + cy * cr, sy * sp * cr - cy * sr,
                            -sp, cp * sr, cp * cr};
      // I_w^-1 = R I_b^-1 R^T
      double ib[9];
      if constexpr (ENV_MODEL) {
        if (model.inertia) {
          env_inv3(model.inertia + 9 * (size_t)env, ib);
        } else {
#pragma unroll
          for (int i = 0; i < 9; ++i) ib[i] = ws->inv_inertia[i];
        }
      }
      double tmp[9], iw[9];
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) {
          double v = 0.0;
#pragma unroll
          for (int c = 0; c < 3; ++c) v += rb[3 * a + c] * (ENV_MODEL ? ib[3 * c + b] : ws->inv_inertia[3 * c + b]);
          tmp[3 * a + b] = v;
        }
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) {
          double v = 0.0;
#pragma unroll
          for (int c = 0; c < 3; ++c) v += tmp[3 * a + c] * rb[3 * b + c];
          iw[3 * a + b] = v;
        }
      if constexpr (FEET) {
        double* __restrict__ pub = &sm.bang[0][0];
#pragma unroll
        for (int i = 0; i < 9; ++i) { pub[i] = rf[i]; pub[9 + i] = iw[i]; }
      } else {
        // own leg's lever arm by selects: a run-time index into fw[][] would put it (and in_feet[]) into a local-memory frame
        const double rx = tid == 0 ? fw[0][0] : (tid == 1 ? fw[1][0] : (tid == 2 ? fw[2][0] : fw[3][0]));
        const double ry = tid == 0 ? fw[0][1] : (tid == 1 ? fw[1][1] : (tid == 2 ? fw[2][1] : fw[3][1]));
        const double rz = tid == 0 ? fw[0][2] : (tid == 1 ? fw[1][2] : (tid == 2 ? fw[2][2] : fw[3][2]));
        const double sk[9] = {0.0, -rz, ry, rz, 0.0, -rx, -ry, rx, 0.0};
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
          for (int b = 0; b < 3; ++b) {
            double v = 0.0;
#pragma unroll
            for (int c = 0; c < 3; ++c) v += iw[3 * a + c] * sk[3 * c + b];
            sm.bang[tid][3 * a + b] = v;
          }
      }
    }
  }
  __syncthreads();
  RG_TOC(41);

  if constexpr (!C::RICCATI) {   // the dense path needs K^-1 explicitly; the Riccati sweep works from K1, K2 alone
  // Q_t = (K1 + gamma_t K2)^-1 : 3x3 SPD angular block (packed xx,yy,zz,xz,yz,xy) + 3 scalars
  if (tid < H) {
    const double gm = ws->eig_gamma[tid];
    const double m00 = sm.k1[0] + gm * sm.k2ang[0], m11 = sm.k1[1] + gm * sm.k2ang[4], m22 = sm.k1[2] + gm * sm.k2ang[8];
    const double m01 = gm * sm.k2ang[1], m02 = gm * sm.k2ang[2], m12 = gm * sm.k2ang[5];
    const double c00 = m11 * m22 - m12 * m12, c01 = m02 * m12 - m01 * m22, c02 = m01 * m12 - m02 * m11;
    const double det = m00 * c00 + m01 * c01 + m02 * c02;
    const double id = 1.0 / det;
    sm.nblk[tid][0] = c00 * id;
    sm.nblk[tid][1] = (m00 * m22 - m02 * m02) * id;
    sm.nblk[tid][2] = (m00 * m11 - m01 * m01) * id;
    sm.nblk[tid][3] = c02 * id;                       // xz
    sm.nblk[tid][4] = (m01 * m02 - m00 * m12) * id;   // yz
    sm.nblk[tid][5] = c01 * id;                       // xy
  }
  __syncthreads();
  RG_TOC(42);

  // K^-1 = (U (x) I) blkdiag(Q_t) (U^T (x) I): one item per ((j,k) time block, packed 3x3 component),
  // a rank-h sum with the host-tabulated weights U[j][t] U[k][t]
  for (int it = tid; it < H * (H + 1) / 2 * 6; it += blockDim.x) {
    const int p = it / 6, pk = it - 6 * p;
    int j = (int)((sqrtf(8.f * p + 1.f) - 1.f) * 0.5f);
    while (tri(j + 1, 0) <= p) ++j;
    while (tri(j, 0) > p) --j;
    const int k = p - tri(j, 0);
    const double* uu = sm.psi + p * H;
    double v = 0.0;
#pragma unroll
    for (int t = 0; t < H; ++t) v = fma(uu[t], sm.nblk[t][pk], v);
    // packed (xx,yy,zz,xz,yz,xy) -> (c,d), c <= d
    const int c = pk < 3 ? pk : (pk == 4 ? 1 : 0), d = pk < 3 ? pk : (pk == 5 ? 1 : 2);
    sm.kinv_ang[tri(3 * j + d, 3 * k + c)] = v;
    if (j > k && c != d) sm.kinv_ang[tri(3 * j + c, 3 * k + d)] = v;
  }
  RG_TOC(43);
  }
  // g~_j = 2 sum_{i>j} [ dt L_nu e_nu(i) + dt^2 (i-j-1/2) G6^T L_rho e_rho(i) ]
  // stage 1 (thread per horizon step i): the weighted errors of the free response against the reference
  // trajectory, in sm.kvec (velocity part) and sm.avec (position part) -- both are free during the setup;
  // stage 2 (thread per (j,c)): the two-term sums.
  {
    const double wx = in_w[0], wy = in_w[1], wz = in_w[2];
    const double vx = in_v[0], vy = in_v[1], vz = in_v[2];
    const double dvx = in_cmd[0], dvy = in_cmd[1], dwz = in_cmd[2];
    const double grav = -ws->gravity;
    if (tid < H) {
      const double ti = (tid + 1) * dt;
      // rpy rate at t0:  T w
      const double rr0 = tm[0] * wx + tm[1] * wy + tm[2] * wz;
      const double rr1 = tm[3] * wx + tm[4] * wy + tm[5] * wz;
      const double rr2 = tm[6] * wx + tm[7] * wy + tm[8] * wz;
      const double er0 = roll + ti * rr0 - 0.0;
      const double er1 = pitch + ti * rr1 - 0.0;
      const double er2 = yaw + ti * rr2 - (yaw + ti * dwz);
      const double ep[3] = {0.0 + ti * vx - ti * dvx, 0.0 + ti * vy - ti * dvy, com_z + ti * vz + 0.5 * ti * ti * grav - ws->height};
      const double en[6] = {wx - 0.0, wy - 0.0, wz - dwz, vx - dvx, vy - dvy, vz + ti * grav - 0.0};
      const double lr0 = ws->w_rho[0] * er0, lr1 = ws->w_rho[1] * er1, lr2 = ws->w_rho[2] * er2;
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        sm.kvec[6 * tid + c] = ws->w_nu[c] * en[c];
        sm.avec[6 * tid + c] = c < 3 ? tm[c] * lr0 + tm[3 + c] * lr1 + tm[6 + c] * lr2 : ws->w_rho[c] * ep[c - 3];   // (T^T L e)_c
      }
    }
    __syncthreads();
    for (int row = tid; row < N6; row += C::NT) {
      const int j = row / 6, c = row % 6;
      double acc = 0.0;
      for (int i = j + 1; i <= H; ++i) acc += 2.0 * (dt * sm.kvec[6 * (i - 1) + c] + dt2 * (i - j - 0.5) * sm.avec[6 * (i - 1) + c]);
      sm.gt[row] = acc;
    }
  }
  __syncthreads();
  RG_TOC(44);

  RG_TRESET();
#ifdef RG_DEBUG_TRACE
  if (g_trace && (int)blockIdx.x == g_trace_env && threadIdx.x == 0) g_trace[900 + 8] += (double)(clock64() - rg_tstart_);
#endif
  // ---------------------------------------------------------------- per-block constants
  Blk blk;
  if constexpr (FEET) {
    // I_w^-1 [r]x from this block's own foot, in the expressions of the per-leg products of the setup (a plan whose rows
    // all equal the current feet gives the same bits)
#pragma unroll
    for (int i = 0; i < 9; ++i) blk.ba[i] = 0.0;
    if (active_blk) {
      const double* __restrict__ rf = &sm.bang[0][0];
      const double* __restrict__ iw = rf + 9;
      const double px = blk_foot[0], py = blk_foot[1], pz = blk_foot[2];
      double fw[3];
#pragma unroll
      for (int r = 0; r < 3; ++r) fw[r] = rf[3 * r] * px + rf[3 * r + 1] * py + rf[3 * r + 2] * pz;
      const double rx = fw[0], ry = fw[1], rz = fw[2];
      const double sk[9] = {0.0, -rz, ry, rz, 0.0, -rx, -ry, rx, 0.0};
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) {
          double v = 0.0;
#pragma unroll
          for (int c = 0; c < 3; ++c) v += iw[3 * a + c] * sk[3 * c + b];
          blk.ba[3 * a + b] = v;
        }
    }
  } else {
#pragma unroll
    for (int i = 0; i < 9; ++i) blk.ba[i] = active_blk ? sm.bang[leg][i] : 0.0;
  }
  blk.inv_mass = inv_mass;
  blk.two_alpha = two_alpha;
  blk.t = t_blk;
  blk.leg = leg;
  blk.is_blk = is_blk;
  blk.act = active_blk;
  double q[3] = {0.0, 0.0, 0.0};
  if (active_blk) {
    const double* g6 = sm.gt + 6 * t_blk;
#pragma unroll
    for (int d = 0; d < 3; ++d)
      q[d] = blk.ba[d] * g6[0] + blk.ba[3 + d] * g6[1] + blk.ba[6 + d] * g6[2] + inv_mass * g6[3 + d];
  }

  // upper bounds hv (rows 0..4) and lower bounds (rows 5..9 as -g.f <= -l)
  const double hv_up[5] = {big_u, big_u, big_u, big_u, fzmax};
  const double lo_b[5] = {0.0, 0.0, 0.0, 0.0, fzmin};

  // ---------------------------------------------------------------- interior point
  // (the lean instantiation declares the interior-point state with one element and never touches it)
  double u[3] = {0.0, 0.0, 0.0}, s[LEAN ? 1 : 10], lam[LEAN ? 1 : 10];
  // strictly feasible start: every stance foot carries its share of the weight
  const double fz0 = fmin(0.5 * (fzmin + fzmax), fmax(2.0 * fzmin, ws->gravity / (inv_mass * n_step)));
  u[2] = active_blk ? fz0 : 0.0;
  double qmax = active_blk ? fmax(fabs(q[0]), fmax(fabs(q[1]), fabs(q[2]))) : 0.0;
  {
    double dsum = 0.0, dmn = 0.0;
    block_reduce<C::NW, 2>(dsum, qmax, dmn, sm.red);
  }
  const double qscale = fmax(1.0, qmax);
  if constexpr (!LEAN) {
    double c5[5];
    g_mul(u, mu, c5);
#pragma unroll
    for (int r = 0; r < 5; ++r) {
      s[r] = hv_up[r] - c5[r];
      s[5 + r] = c5[r] - lo_b[r];
    }
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      if (!active_blk) s[r] = 1.0;
      lam[r] = active_blk ? kIpmLam0 * qscale / s[r] : 1.0;   // inactive threads carry harmless 1/1 pairs
    }
  }
  const double m_total = PLAN ? 10.0 * plan_blocks : 10.0 * H * n_stance;
  const int max_iters = ws->max_ipm_iters;
  const int max_polish = ws->max_polish_rounds;
  double tol = ws->ipm_tol;
  int iters = 0, polish_rounds = 0, status = 0, n_active_out = 0;
  unsigned act_out = RG_ACTIVE_SET_UNKNOWN;
  double u_out[3] = {u[0], u[1], u[2]};

  // Escalation ladder: interior point to `tol`, then the active-set polish; if the polish does not
  // verify within its round budget (weakly active constraints: multipliers of order alpha), drive
  // the interior point 100x further and try again.  Last resort: the best interior-point iterate.
  int trace_n = 0;
  (void)trace_n;
  double best_res = 1e300, prev_res = 1e300;
  double u_best[3] = {u[0], u[1], u[2]};
  int stall = 0, slow = 0;
  bool done = false;
  // Attempt -1 is the cold start: the same active-set iteration started from the empty set (round 0
  // is the unconstrained minimiser), with no interior point before it.  Most trot-like problems have
  // a handful of active rows and verify within 2-3 rounds (DESIGN.md 3.3); the ones that do not fall
  // through to the interior point untouched.
  const int cold_rounds = ws->cold_start_rounds;
  const double cold_max_viol = (double)ws->cold_start_max_violations;
  // Weakly active rows (multiplier ~ 0 at the optimum: strict complementarity fails) flip for ever between "dropped
  // because its multiplier is -1e-10" and "violated by 1e-9 without it".  A row that was dropped and came back is
  // sticky: it then only leaves for a multiplier that is wrong by more than kStickyTol (1e-9) of the gradient scale.
  unsigned dropped_rows = 0u, sticky_rows = 0u;
#pragma unroll 1
  for (int attempt = (cold_rounds > 0 && !skip_cold) ? -1 : 0; attempt < (LEAN ? 0 : 3) && !done; ++attempt) {
    bool converged = false, ipm_dead = false, handed_over = false;
    const bool cold = LEAN || attempt < 0;
    if constexpr (!LEAN) {
    if (!cold) {
    if (iters == 0) {
      // Centred start s lam = mu0 with mu0 commensurate with the dual residual at the start: with mu0 far
      // below |r_d| the first iterations crawl along the boundary (pace / bound problems: |r_d| ~ 100 |q|).
      double pu0[3];
      apply_p<H>(sm, ws, blk, u, pu0);
      double dsum = 0.0, rd0 = 0.0, dmn = 0.0;
      if (active_blk) {
#pragma unroll
        for (int d = 0; d < 3; ++d) rd0 = fmax(rd0, fabs(pu0[d] + q[d]));
      }
      block_reduce<C::NW, 2>(dsum, rd0, dmn, sm.red);
      const double mu0 = kIpmLam0 * fmax(qscale, rd0);
#pragma unroll
      for (int r = 0; r < 10; ++r) lam[r] = active_blk ? mu0 / s[r] : 1.0;
    }
#pragma unroll 1
    while (true) {
      double pu[3], rd[3], gl[3];
      RG_TOC(0);
      apply_p<H>(sm, ws, blk, u, pu);
      RG_TOC(1);
      gt_mul(lam, mu, gl);
      double sl = 0.0, rdmax = 0.0, dmn = 0.0;
#pragma unroll
      for (int d = 0; d < 3; ++d) { rd[d] = pu[d] + q[d] + gl[d]; rdmax = fmax(rdmax, fabs(rd[d])); }
      // sl_r = s lam and its reciprocal: the only ten divisions of the iteration
      // only isl stays live across the factorisation and the solves: 1/s = lam isl, 1/lam = s isl
      double isl[10];
#pragma unroll
      for (int r = 0; r < 10; ++r) {
        const double slr = s[r] * lam[r];
        isl[r] = 1.0 / slr;
        sl += slr;
      }
      if (!active_blk) { sl = 0.0; rdmax = 0.0; }
      block_reduce<C::NW, 3>(sl, rdmax, dmn, sm.red);
      const double mu_c = sl / m_total;
      const double res = fmax(rdmax, mu_c) / qscale;
      RG_TRACE(4 * trace_n + 0, res); RG_TRACE(4 * trace_n + 1, mu_c); RG_TRACE(4 * trace_n + 2, (double)iters); RG_TRACE(4 * trace_n + 3, tol);
      ++trace_n;
      // slow lane: the best residual has not halved for kIpmSlowIters iterations although the iterate is
      // already close (mu oscillating around 1e-5 on a few pace / bound problems, 40 iterations to the cap):
      // hand over to the active-set rounds, which verify from such a point in a round or two
      slow = (res < 0.5 * best_res) ? 0 : slow + 1;
      if (res < best_res) {
        best_res = res;
#pragma unroll
        for (int d = 0; d < 3; ++d) u_best[d] = u[d];
      }
      if (res < tol) { converged = true; break; }
      if (slow >= kIpmSlowIters && res < 1e-3 && max_polish > 0) { handed_over = true; slow = 0; break; }
      stall = (res > 0.9 * prev_res && res < 1e-7) ? stall + 1 : 0;   // only near the numerical floor
      prev_res = res;
      // dead: budget spent, stalled at the numerical floor, NaN, or diverging (deep iterates lose the
      // tiny slacks of active rows to cancellation in ds = -G dx; see DESIGN.md 3.5)
      if (iters >= max_iters || stall >= 4 || !(res == res) || res > 1e3 * best_res) {
        ipm_dead = true;
        break;
      }
      ++iters;

      // block 3x3 parts and Psi
      double dd[5], einv[6];
#pragma unroll
      for (int r = 0; r < 5; ++r) dd[r] = lam[r] * lam[r] * isl[r] + lam[5 + r] * lam[5 + r] * isl[5 + r];
      block_inverse(dd, mu, two_alpha, einv);
      double inv_d[5];
#pragma unroll
      for (int r = 0; r < 5; ++r) inv_d[r] = 1.0 / dd[r];
      Chol5 ch;
      chol5_factor(mu, inv_d, two_alpha, ch);
      RG_TOC(2);
      factor_psi<H>(sm, ws, blk, einv);
      RG_TOC(3);
      if (sm.flag) { status |= RG_STATUS_NUMERIC; ipm_dead = true; break; }

      // Mehrotra predictor (phase 0: r_c = s lam, rhs = -(P u + q)) and corrector (phase 1:
      // r_c = s lam + ds_a dl_a - sigma mu, rhs = -r_d + G^T (r_c / s)); one copy of the solve code.
      double wv[10], dx[3], c5[5];
      double sigmu = 0.0;
#pragma unroll
      for (int r = 0; r < 10; ++r) wv[r] = 0.0;
#pragma unroll 1
      for (int phase = 0; phase < 2; ++phase) {
        double rhs[3];
        if (phase == 0) {
#pragma unroll
          for (int d = 0; d < 3; ++d) rhs[d] = -(pu[d] + q[d]);
        } else {
          double gw[3];
          gt_mul(wv, mu, gw);
#pragma unroll
          for (int d = 0; d < 3; ++d) rhs[d] = -rd[d] + gw[d];
        }
        double bprime[3];
        RG_TOC(4);
        woodbury_solve<H>(sm, blk, einv, rhs, bprime);
        RG_TOC(5);
        chol5_block_solve(ch, mu, inv_d, two_alpha, bprime, dx, c5);   // c5 = G dx without cancellation
        if (phase == 0) {
          // x_r = ds_r / s_r ; dl_r / lam_r = -1 - x_r: the largest feasible affine step is 1 / max(-x, 1 + x)
          double tmax = 1.0, dsum = 0.0, dmn2 = 0.0;
          double xr[10];
#pragma unroll
          for (int r = 0; r < 10; ++r) {
            xr[r] = (r < 5 ? -c5[r] : c5[r - 5]) * (lam[r] * isl[r]);
            if (active_blk) tmax = fmax(tmax, fmax(-xr[r], 1.0 + xr[r]));
          }
          block_reduce<C::NW, 2>(dsum, tmax, dmn2, sm.red);
          const double amax = 1.0 / tmax;
          double mu_aff = 0.0;
#pragma unroll
          for (int r = 0; r < 10; ++r) {
            const double slr = s[r] * lam[r];
            mu_aff += slr * (1.0 + amax * xr[r]) * (1.0 - amax * (1.0 + xr[r]));
            wv[r] = -slr * xr[r] * (1.0 + xr[r]);             // ds_a dl_a
          }
          if (!active_blk) mu_aff = 0.0;
          double dmx3 = 0.0, dmn3 = 0.0;
          block_reduce<C::NW, 1>(mu_aff, dmx3, dmn3, sm.red);
          mu_aff /= m_total;
          const double ratio = mu_aff / mu_c;
          sigmu = ratio * ratio * ratio * mu_c;
#pragma unroll
          for (int r = 0; r < 10; ++r) wv[r] = (s[r] * lam[r] + wv[r] - sigmu) * (lam[r] * isl[r]);   // r_c / s
        }
      }
      // step to the boundary: -ds/s = -y, -dl/lam = w/lam + y with y = ds/s
      double tmax = 0.0, dsum = 0.0, dmn2 = 0.0;
      double yr[10];
#pragma unroll
      for (int r = 0; r < 10; ++r) {
        yr[r] = (r < 5 ? -c5[r] : c5[r - 5]) * (lam[r] * isl[r]);
        if (active_blk) tmax = fmax(tmax, fmax(-yr[r], wv[r] * (s[r] * isl[r]) + yr[r]));
      }
      block_reduce<C::NW, 2>(dsum, tmax, dmn2, sm.red);
      // fraction to the boundary: 0.99 throughout.  (0.999 once the residuals are small saved nothing measurable
      // and made two bound-gait problems in 1.5 M oscillate at mu ~ 1e-4; steps closer to 1 collapse the slacks
      // while the dual residual is still finite and de-centre the iterate.)
      const double tau = 0.99;
      const double step = tmax > tau ? tau / tmax : 1.0;
      if (active_blk) {
#pragma unroll
        for (int r = 0; r < 10; ++r) {
          const double ds = yr[r] * s[r];
          const double dl = -wv[r] - lam[r] * yr[r];
          s[r] += step * ds;
          lam[r] += step * dl;
        }
#pragma unroll
        for (int d = 0; d < 3; ++d) u[d] += step * dx[d];
      }
    }
    if (converged) status |= RG_STATUS_IPM_CONVERGED; else status &= ~RG_STATUS_IPM_CONVERGED;
    if (max_polish <= 0) {
      if (ipm_dead || tol <= 1e-9) break;
      tol = 1e-9;        // without the polish the interior point itself has to resolve the alpha-directions
      continue;
    }
    }   // !cold
    }   // !LEAN

    RG_TOC(6);
    // -------------------------------------------------------------- active-set polish
    unsigned act = 0;
    if (!cold) {
      if constexpr (!LEAN) {
#pragma unroll
        for (int r = 0; r < 10; ++r) if (active_blk && lam[r] > 0.03 * s[r]) act |= 1u << r;
      }
    } else if (warm_act != RG_ACTIVE_SET_UNKNOWN) {
      // warm start: the verified active set of this block from the previous solve of the same env
      // (consecutive control steps see almost the same problem); wrong guesses are repaired by the rounds
      act = active_blk ? warm_act : 0u;
    } else if (active_blk && t_blk >= H - (n_step == 4 ? kColdGuessLast4 : kColdGuessLast)) {
      // a force in the last step(s) of the horizon barely moves any tracked state, so the regulariser
      // drives it to zero: fz >= fz_min is active there in practically every problem (bit 9)
      act = 1u << 9;
    }
    bool polished = false, fact_valid = false;   // the factor in shared memory is the interior point's, if any
    unsigned act_fact = 0;
    double prev_nchg = 1e300;   // unused, but deleting it moves ptxas's register assignment in the h = 20 lean model kernel
    double up[3] = {0.0, 0.0, 0.0};
    // 3, 6, 12 rounds: later attempts start from a sharper guess; a dead interior point gets the full budget
    const int round_budget = cold ? cold_rounds : (ipm_dead || handed_over) ? (max_polish << 2) : (max_polish << attempt);
#pragma unroll 1
    for (int round = 0; round < round_budget; ++round) {
      ++polish_rounds;
      // --- per block: orthonormal basis of the active normals (<= 3), null-space basis Z, u0.
      // The basis sits in named registers (no local-memory frame: DRAM traffic = the algorithmic bytes) and only while
      // it is used here: the multiplier test rebuilds it.  Against small local arrays indexed by the run-time row count:
      // h = 5 27.2 -> 28.8 M, h = 20 5.72 -> 5.85 M solves/s at 65536 envs (profiles/r02_basis_storage.md).
      int na;
      double u0[3], mproj[6];
      {
        BlockBasis B;
        build_basis(act, active_blk, mu, hv_up, lo_b, B);
        na = B.na;
        // particular solution u0 = sum_k c_k e_k with a_i . u0 = b_i  (forward substitution with rr^T; unused slots have
        // zero basis vectors and unit diagonal, so they contribute nothing)
        const double cp0 = na > 0 ? B.bt0 * B.ir00 : 0.0;
        const double cp1 = na > 1 ? (B.bt1 - B.r01 * cp0) * B.ir11 : 0.0;
        const double cp2 = na > 2 ? (B.bt2 - B.r02 * cp0 - B.r12 * cp1) * B.ir22 : 0.0;
#pragma unroll
        for (int d = 0; d < 3; ++d) u0[d] = cp0 * B.e0[d] + cp1 * B.e1[d] + cp2 * B.e2[d];
        // projector onto the free directions  M = I - sum_k e_k e_k^T, packed (xx,yy,zz,xz,yz,xy),
        // scaled by 1 / (2 alpha): this is the "E^-1" of the equality-constrained Newton system
        mproj[0] = 1.0 - (B.e0[0] * B.e0[0] + B.e1[0] * B.e1[0] + B.e2[0] * B.e2[0]);
        mproj[1] = 1.0 - (B.e0[1] * B.e0[1] + B.e1[1] * B.e1[1] + B.e2[1] * B.e2[1]);
        mproj[2] = 1.0 - (B.e0[2] * B.e0[2] + B.e1[2] * B.e1[2] + B.e2[2] * B.e2[2]);
        mproj[3] = -(B.e0[0] * B.e0[2] + B.e1[0] * B.e1[2] + B.e2[0] * B.e2[2]);
        mproj[4] = -(B.e0[1] * B.e0[2] + B.e1[1] * B.e1[2] + B.e2[1] * B.e2[2]);
        mproj[5] = -(B.e0[0] * B.e0[1] + B.e1[0] * B.e1[1] + B.e2[0] * B.e2[1]);
      }
      if (na == 3 || !active_blk) { mproj[0] = mproj[1] = mproj[2] = mproj[3] = mproj[4] = mproj[5] = 0.0; }
      const double inv2a = 1.0 / two_alpha;
#pragma unroll
      for (int i = 0; i < 6; ++i) mproj[i] *= inv2a;
      RG_TOC(20);
      // Only the time steps from the first block whose active set moved since the last factorisation
      // change Psi, and a left-looking Cholesky keeps its leading columns: refactor the tail only
      // (active rows cluster at the end of the horizon: DESIGN.md 3.3).
      int t_fac;                                                          // first time block to refactorise, -1: none
      {
        double dsum = 0.0, dmx = 0.0, tmin = (double)H;
        if (active_blk && act != act_fact) tmin = (double)t_blk;
        if (!fact_valid) tmin = 0.0;
        block_reduce<C::NW, 4>(dsum, dmx, tmin, sm.red);
        t_fac = tmin < (double)H ? (C::RICCATI ? 0 : (((int)tmin) & ~1)) : -1;   // cholesky_rows restarts on a 4-column panel
      }
      RG_TIC();
      if (t_fac >= 0) factor_psi<H>(sm, ws, blk, mproj, t_fac);
      else if (tid == 0) sm.flag = 0;
      act_fact = act;
      fact_valid = true;
      __syncthreads();
      if (sm.flag) {
        if (!cold) { status |= RG_STATUS_NUMERIC; ipm_dead = true; }   // a failed cold start just hands over
        break;
      }

      // Pass -1 evaluates gr = P u + q at the particular solution, pass 0 is the solve, passes 1-2 steps of iterative
      // refinement (one call site of apply_p serves all of them).  The active set is checked after
      // each solve: when it moves after pass 0 the refinement would be wasted (the next round starts over),
      // and it is skipped as well when pass 0 already left a projected gradient at rounding level.
      // A verdict on the set is only taken from a solve that is accurate enough to give it (projected
      // gradient <= 1e-9 |q|): with many active rows at h = 20 a single refinement step can leave 1e-9,
      // above the multiplier-sign threshold, and one weakly active row then flips in and out for ever.
#pragma unroll
      for (int d = 0; d < 3; ++d) up[d] = u0[d];
      double gr[3] = {0.0, 0.0, 0.0};
      if constexpr (!C::GRAD_IN_PASS_LOOP) {
        double pu0[3];
        apply_p<H>(sm, ws, blk, up, pu0);
#pragma unroll
        for (int d = 0; d < 3; ++d) gr[d] = pu0[d] + q[d];
      }
      unsigned act_new = act;
      double nchg = 0.0, ncone = 0.0, pgm = 0.0;
      bool accept = false;
#pragma unroll 1
      for (int pass = C::GRAD_IN_PASS_LOOP ? -1 : 0; pass < 3; ++pass) {
        double pu[3];
        if (pass >= 0) {
          double ng[3], bprime[3], dx[3];
#pragma unroll
          for (int d = 0; d < 3; ++d) ng[d] = -gr[d];
          RG_TOC(21);
          woodbury_solve<H>(sm, blk, mproj, ng, bprime);
          RG_TOC(22);
          sym3_mul(mproj, bprime, dx);
#pragma unroll
          for (int d = 0; d < 3; ++d) up[d] += dx[d];
        }
        apply_p<H>(sm, ws, blk, up, pu);
        RG_TOC(23);
#pragma unroll
        for (int d = 0; d < 3; ++d) gr[d] = pu[d] + q[d];
        if (pass < 0) continue;

        // --- verify: primal feasibility of the rows left out, multiplier signs of the rows held
        act_new = act;
        if (active_blk) {
          double c5[5];
          g_mul(up, mu, c5);
          const double ftol = 1e-9 * fzmax;
          // Only the MOST violated row of the block comes in per round: both cone rows of a direction (or a cone
          // row and a bound) violated together over-constrain the block when added at once, the sign test throws
          // one out again and the iteration cycles.  One row per block per round settles 99 % of the pace batch
          // within 14 rounds against 76 % for "add all" (tools/experiments/pdas_variants.py), at the same mean
          // number of rounds on trot.
          double worst = -ftol;
          int rworst = -1;
#pragma unroll
          for (int r = 0; r < 10; ++r) {
            const double slack = r < 5 ? hv_up[r] - c5[r] : c5[r - 5] - lo_b[r - 5];
            if (!((act >> r) & 1u) && slack < worst) { worst = slack; rworst = r; }
          }
          if (rworst >= 0) {
            act_new |= 1u << rworst;
            if ((dropped_rows >> rworst) & 1u) sticky_rows |= 1u << rworst;
          }
          int rmin = -1;
          // the basis is rebuilt from the bit mask (a few dozen instructions) instead of being kept live across the
          // factorisation and the sweeps: 21 doubles fewer in flight over the heavy calls
          BlockBasis B;
          { unsigned act_again = act; build_basis(act_again, active_blk, mu, hv_up, lo_b, B); }
          // multipliers: sum_i y_i a_i = -gr on span(e)  ->  back substitution with the upper triangular rr
          const int row0 = B.row0, row1 = B.row1, row2 = B.row2;
          const double g0 = -(gr[0] * B.e0[0] + gr[1] * B.e0[1] + gr[2] * B.e0[2]);
          const double g1 = -(gr[0] * B.e1[0] + gr[1] * B.e1[1] + gr[2] * B.e1[2]);
          const double g2 = -(gr[0] * B.e2[0] + gr[1] * B.e2[1] + gr[2] * B.e2[2]);
          const double y2 = g2 * B.ir22;
          const double y1 = (g1 - B.r12 * y2) * B.ir11;
          const double y0 = (g0 - B.r01 * y1 - B.r02 * y2) * B.ir00;
          double ymin = 1e300;
#pragma unroll
          for (int i = 0; i < 3; ++i) {
            const int row = i == 0 ? row0 : (i == 1 ? row1 : row2);
            const double yi = i == 0 ? y0 : (i == 1 ? y1 : y2);
            if (i < na) {
              // upper-bound rows need y >= 0, lower-bound rows y <= 0
              const double ysgn = row < 5 ? yi : -yi;
              const double drop_tol = ((sticky_rows >> row) & 1u) ? kStickyTol : 1e-10;
              if (ysgn < -drop_tol * qscale) { act_new &= ~(1u << row); dropped_rows |= 1u << row; }
              if (ysgn < ymin) { ymin = ysgn; rmin = row; }
            }
          }
          // a block that already holds three rows is a vertex: a violated fourth row can only come in if one
          // leaves, and the basis builder keeps the first three in bit order -- without this swap the newcomer
          // is dropped again next round and the same round repeats for ever.  The weakest multiplier leaves.
          if (na == 3 && (act_new & ~act) != 0u && (act_new & act) == act) act_new &= ~(1u << rmin);
        }
        // stationarity on the free subspace is what the solve is supposed to deliver; check it anyway so
        // that a wrong factorisation can never be reported as a verified optimum:  |Z Z^T (P u + q)|_inf
        double pg[3];
        sym3_mul(mproj, gr, pg);
        pgm = active_blk ? two_alpha * fmax(fabs(pg[0]), fmax(fabs(pg[1]), fabs(pg[2]))) : 0.0;
        // one reduction carries both counts: rows that moved, and how many of those are friction-cone rows
        // (bits 0-3 / 5-8; bits 4 / 9 are the fz bounds)
        nchg = (double)(__popc(act_new ^ act) + 4096 * __popc((act_new ^ act) & 0x1EFu));
        double dmn = 0.0;
        block_reduce<C::NW, 3>(nchg, pgm, dmn, sm.red);
        ncone = floor(nchg * (1.0 / 4096.0));
        nchg -= 4096.0 * ncone;
        RG_TOC(24);
        const bool trusted = pgm <= 1e-9 * qscale || pass == 2;
        if (nchg > 0.0) { if (trusted) break; else continue; }
        if (pgm <= (pass == 0 ? kSkipRefineTol : pass == 1 ? 1e-10 : 1e-7) * qscale) { accept = true; break; }
      }
#if defined(RG_DEBUG_TRACE) && !defined(RG_DEBUG_TIMELINE_ONLY)
      {
        double cnt = (double)__popc(act_new), dmx2 = 0.0, dmn2 = 0.0;
        block_reduce<C::NW>(cnt, dmx2, dmn2, sm.red);
        RG_TRACE(4 * trace_n + 0, cold ? -2.0 : -1.0); RG_TRACE(4 * trace_n + 1, nchg); RG_TRACE(4 * trace_n + 2, cnt); RG_TRACE(4 * trace_n + 3, pgm / qscale);
        ++trace_n;
      }
#endif
      if (accept) { polished = true; break; }
      // the cold start hands over to the interior point when the unconstrained minimiser violates too
      // many friction-cone rows (fz-bound rows settle in a round or two, cone rows make it cycle)
      if (cold && ((round == 0 && ncone > cold_max_viol) || (round + 1 >= cold_rounds && nchg > kColdLastRoundNchg))) break;
      prev_nchg = nchg;
      act = act_new;
    }
    if (polished) {
      act_out = act;
      status |= cold ? (RG_STATUS_POLISHED | RG_STATUS_ACTIVE_SET_ONLY) : RG_STATUS_POLISHED;
#pragma unroll
      for (int d = 0; d < 3; ++d) u_out[d] = up[d];
      double cnt = (double)__popc(act), dmx = 0.0, dmn = 0.0;
      block_reduce<C::NW, 1>(cnt, dmx, dmn, sm.red);
      n_active_out = (int)cnt;
      done = true;
      break;
    }
    if (ipm_dead) break;
    if constexpr (LEAN) break;
    if (cold) {
      // The cold start gave up: move the interior point's start from the safe point towards the last
      // active-set iterate, as far as strict feasibility allows (ratio test), keeping r_p = 0.
      double dir[3] = {up[0] - u[0], up[1] - u[1], up[2] - u[2]}, c5d[5];
      g_mul(dir, mu, c5d);
      double dsum = 0.0, dmx = 0.0, thmax = 1.0;
      if (active_blk) {
#pragma unroll
        for (int r = 0; r < 5; ++r) {
          if (c5d[r] > 0.0) thmax = fmin(thmax, s[r] / c5d[r]);
          if (c5d[r] < 0.0) thmax = fmin(thmax, s[5 + r] / -c5d[r]);
        }
        if (!(thmax == thmax)) thmax = 0.0;
      }
      block_reduce<C::NW, 4>(dsum, dmx, thmax, sm.red);
      const double theta = kIpmWarm * thmax;
      if constexpr (!LEAN) {
        if (active_blk && theta > 0.0) {
#pragma unroll
          for (int d = 0; d < 3; ++d) u[d] += theta * dir[d];
          double c5[5];
          g_mul(u, mu, c5);
#pragma unroll
          for (int r = 0; r < 5; ++r) { s[r] = hv_up[r] - c5[r]; s[5 + r] = c5[r] - lo_b[r]; }
        }
      }
      continue;
    }
    tol = fmax(tol * 1e-2, 1e-9);   // float64 interior-point iterates are trustworthy down to ~1e-9 here
  }
  if constexpr (LEAN) {
    if (!done) {
      // not verified by the rounds alone: the full solver takes this env from the fallback queue
      if (tid == 0) {
        const int slot = atomicAdd(&scratch->queue_tail, 1);
        scratch->queue[slot] = env;
      }
      return;
    }
  }
  if (!done) {
#pragma unroll
    for (int d = 0; d < 3; ++d) u_out[d] = u_best[d];
  }

  RG_TOC(7);
#ifdef RG_DEBUG_TRACE
  if (g_trace && (int)blockIdx.x == g_trace_env && threadIdx.x == 0) g_trace[900 + 9] += (double)(clock64() - rg_tstart_);
  if (g_trace && g_trace_env == -2 && tid == 0) {
    unsigned long long ns;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
    g_trace[1024 + 4 * env + 1] = (double)ns;
  }
#endif
  // ---------------------------------------------------------------- outputs (negated solution)
  if (is_blk) {
    const float fx = active_blk ? (float)(-u_out[0]) : 0.f;
    const float fy = active_blk ? (float)(-u_out[1]) : 0.f;
    const float fz = active_blk ? (float)(-u_out[2]) : 0.f;
    if (t_blk == 0) {
      float* o = g_forces + 12 * (size_t)env + 3 * leg;
      o[0] = fx; o[1] = fy; o[2] = fz;
    }
    if (g_hforces) {
      float* o = g_hforces + 12 * H * (size_t)env + 12 * t_blk + 3 * leg;
      o[0] = fx; o[1] = fy; o[2] = fz;
    }
    if (g_hforces64) {
      double* o = g_hforces64 + 12 * H * (size_t)env + 12 * t_blk + 3 * leg;
      o[0] = active_blk ? -u_out[0] : 0.0; o[1] = active_blk ? -u_out[1] : 0.0; o[2] = active_blk ? -u_out[2] : 0.0;
    }
  }
  if (g_active && is_blk) g_active[(size_t)env * C::NB + tid] = (uint16_t)((done && active_blk) ? act_out : RG_ACTIVE_SET_UNKNOWN);
  if (g_info && tid == 0) {
    int32_t* o = g_info + 4 * (size_t)env;
    o[RG_INFO_IPM_ITERS] = iters;
    o[RG_INFO_POLISH_ROUNDS] = polish_rounds;
    o[RG_INFO_STATUS] = status;
    o[RG_INFO_NUM_ACTIVE] = n_active_out;
  }
}

// Grid of the lean kernel and of the single-kernel path: one CTA per env (blockIdx.x = env).
template <int H, bool LEAN, bool ENV_MODEL, bool PLAN = false, bool FEET = false>
__device__ __forceinline__ void solve_grid(const RgMpcDev* __restrict__ ws, RgMpcScratch* __restrict__ scratch, int n_env,
                                           const rg_mpc_io& io, const rg_mpc_env_model& model,
                                           const uint8_t* __restrict__ plan = nullptr,
                                           const float* __restrict__ feet = nullptr) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem<H>& sm = *reinterpret_cast<Smem<H>*>(smem_raw);
  const int env = blockIdx.x;
  RG_GRID_LAUNCH_DEPENDENTS();   // see launch_kernels: the fallback grid (lean) or the step epilogue (complete kernel) may be scheduled behind us
  RG_GRID_WAIT();                // launched programmatically behind the step prologue in rg_control_step; a no-op otherwise
  if (env >= n_env) return;
  solve_env<H, LEAN, ENV_MODEL, PLAN, FEET>(sm, ws, scratch, env, false, io, model, plan, feet);
}

// Second kernel of the two-kernel solve: the complete solver on the envs the lean kernel queued.  Persistent CTAs
// stride over the list (it is empty for trot / walk batches: the launch then costs a few microseconds); the cold
// start is skipped -- the lean kernel has just spent its budget on exactly those rounds.  The last CTA to finish
// re-arms the queue counters for the next solve.
template <int H, bool ENV_MODEL, bool PLAN = false, bool FEET = false>
__device__ __forceinline__ void fallback_grid(const RgMpcDev* __restrict__ ws, RgMpcScratch* __restrict__ scratch, int n_env,
                                              const rg_mpc_io& io, const rg_mpc_env_model& model,
                                              const uint8_t* __restrict__ plan = nullptr,
                                              const float* __restrict__ feet = nullptr) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem<H>& sm = *reinterpret_cast<Smem<H>*>(smem_raw);
  RG_GRID_LAUNCH_DEPENDENTS();   // the step epilogue may be scheduled behind this grid
  RG_GRID_WAIT();                // launched programmatically: the lean grid must have completed
  const int count = min(scratch->queue_tail, min(scratch->capacity, n_env));
  for (int q = blockIdx.x; q < count; q += gridDim.x) {
    const int env = scratch->queue[q];
    if (env >= 0 && env < n_env)
      solve_env<H, false, ENV_MODEL, PLAN, FEET>(sm, ws, scratch, env, true, io, model, plan, feet);
    __syncthreads();   // shared memory is reused by the next env of this CTA
  }
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(&scratch->done_ctas, 1) == (int)gridDim.x - 1) {   // every CTA has read queue_tail and finished
      scratch->queue_tail = 0;
      scratch->done_ctas = 0;
    }
  }
}

// The model-free kernels keep the parameter list they were tuned with (an extra kernel parameter renumbers the PTX
// virtual registers, and ptxas then schedules the h = 10 lean kernel differently); the *_model_kernel twins take the
// per-env model (rg_mpc_env_model, at least one array non-NULL).

template <int H, bool LEAN>
__global__ void __launch_bounds__(Cfg<H>::NT, Cfg<H>::MIN_BLOCKS)
mpc_solve_kernel(const RgMpcDev* __restrict__ ws, RgMpcScratch* __restrict__ scratch, int n_env, const rg_mpc_io io) {
  solve_grid<H, LEAN, false>(ws, scratch, n_env, io, rg_mpc_env_model{nullptr, nullptr, nullptr});
}

template <int H, bool LEAN>
__global__ void __launch_bounds__(Cfg<H>::NT, Cfg<H>::MIN_BLOCKS)
mpc_solve_model_kernel(const RgMpcDev* __restrict__ ws, RgMpcScratch* __restrict__ scratch, int n_env, const rg_mpc_io io,
                       const rg_mpc_env_model model) {
  solve_grid<H, LEAN, true>(ws, scratch, n_env, io, model);
}

template <int H>
__global__ void __launch_bounds__(Cfg<H>::NT, Cfg<H>::MIN_BLOCKS)
mpc_fallback_kernel(const RgMpcDev* __restrict__ ws, RgMpcScratch* __restrict__ scratch, int n_env, const rg_mpc_io io) {
  fallback_grid<H, false>(ws, scratch, n_env, io, rg_mpc_env_model{nullptr, nullptr, nullptr});
}

template <int H>
__global__ void __launch_bounds__(Cfg<H>::NT, Cfg<H>::MIN_BLOCKS)
mpc_fallback_model_kernel(const RgMpcDev* __restrict__ ws, RgMpcScratch* __restrict__ scratch, int n_env, const rg_mpc_io io,
                          const rg_mpc_env_model model) {
  fallback_grid<H, true>(ws, scratch, n_env, io, model);
}

// Contact-schedule twins (rg_mpc_build_solve_schedule): always with the per-env model, whose NULL arrays stand for the
// workspace's values, so one instantiation per (H, LEAN) serves a schedule with or without a model.
template <int H, bool LEAN>
__global__ void __launch_bounds__(Cfg<H>::NT, Cfg<H>::MIN_BLOCKS)
mpc_solve_plan_kernel(const RgMpcDev* __restrict__ ws, RgMpcScratch* __restrict__ scratch, int n_env, const rg_mpc_io io,
                      const rg_mpc_env_model model, const uint8_t* __restrict__ plan) {
  solve_grid<H, LEAN, true, true>(ws, scratch, n_env, io, model, plan);
}

template <int H>
__global__ void __launch_bounds__(Cfg<H>::NT, Cfg<H>::MIN_BLOCKS)
mpc_fallback_plan_kernel(const RgMpcDev* __restrict__ ws, RgMpcScratch* __restrict__ scratch, int n_env, const rg_mpc_io io,
                         const rg_mpc_env_model model, const uint8_t* __restrict__ plan) {
  fallback_grid<H, true, true>(ws, scratch, n_env, io, model, plan);
}

// Foothold-plan twins (rg_mpc_build_solve_footholds): with the schedule and the per-env model, as the schedule twins.
template <int H, bool LEAN>
__global__ void __launch_bounds__(Cfg<H>::NT, Cfg<H>::MIN_BLOCKS)
mpc_solve_feet_kernel(const RgMpcDev* __restrict__ ws, RgMpcScratch* __restrict__ scratch, int n_env, const rg_mpc_io io,
                      const rg_mpc_env_model model, const uint8_t* __restrict__ plan, const float* __restrict__ feet) {
  solve_grid<H, LEAN, true, true, true>(ws, scratch, n_env, io, model, plan, feet);
}

template <int H>
__global__ void __launch_bounds__(Cfg<H>::NT, Cfg<H>::MIN_BLOCKS)
mpc_fallback_feet_kernel(const RgMpcDev* __restrict__ ws, RgMpcScratch* __restrict__ scratch, int n_env, const rg_mpc_io io,
                         const rg_mpc_env_model model, const uint8_t* __restrict__ plan, const float* __restrict__ feet) {
  fallback_grid<H, true, true, true>(ws, scratch, n_env, io, model, plan, feet);
}

// Dynamic shared memory above 48 KB (h = 20) and the carveout are per-device function attributes: set them once
// per (kernel, device), under a lock -- a process may drive several GPUs from several threads.
int configure_kernel(const void* kernel, size_t smem, int min_blocks, const char* what) {
  static std::mutex mutex;
  static std::map<const void*, unsigned long long> configured;   // kernel -> bit d set: done for device d
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return rg_check_cuda(e, "cudaGetDevice");
  std::lock_guard<std::mutex> lock(mutex);
  unsigned long long& mask = configured[kernel];
  if (dev < 64 && ((mask >> dev) & 1ull)) return RG_OK;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return rg_check_cuda(e, what);
  // the default carveout leaves room for only ~5 CTAs: ask for what MIN_BLOCKS resident CTAs need and no
  // more, so that the rest of the 228 KB stays L1 (local-memory traffic and the parameter block live there)
  const int need_kb = (int)((min_blocks * (smem + 1024) + 1023) / 1024);
  int carveout = (need_kb * 100 + 227) / 228 + 1;
  if (carveout > 100) carveout = 100;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, carveout);
  if (e != cudaSuccess) return rg_check_cuda(e, what);
  if (dev < 64) mask |= 1ull << dev;
  return RG_OK;
}

// SM count of the current device (cached per device: this sits on the launch path)
int sm_count() {
  static std::mutex mutex;
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  std::lock_guard<std::mutex> lock(mutex);
  if (cached[dev] == 0) {
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cached[dev] = sms > 0 ? sms : 148;
  }
  return cached[dev];
}

template <bool B, class A, class C>
constexpr auto pick(A a, C c) { if constexpr (B) return c; else return a; }

template <int H, bool ENV_MODEL, bool PLAN = false, bool FEET = false>
int launch_kernels(const RgMpcDev* ws, int n_env, const rg_mpc_io& io, int two_kernel, cudaStream_t stream, int chained,
                   const rg_mpc_env_model& model, const uint8_t* plan = nullptr, const float* feet = nullptr) {
  static_assert(!PLAN || ENV_MODEL, "the schedule kernels are instantiated with the per-env model only");
  static_assert(!FEET || PLAN, "the foothold kernels are instantiated with the schedule only");
  const auto lean_kernel = pick<FEET>(pick<PLAN>(pick<ENV_MODEL>(mpc_solve_kernel<H, true>, mpc_solve_model_kernel<H, true>),
                                                 mpc_solve_plan_kernel<H, true>),
                                      mpc_solve_feet_kernel<H, true>);
  const auto full_kernel = pick<FEET>(pick<PLAN>(pick<ENV_MODEL>(mpc_solve_kernel<H, false>, mpc_solve_model_kernel<H, false>),
                                                 mpc_solve_plan_kernel<H, false>),
                                      mpc_solve_feet_kernel<H, false>);
  const auto fallback_kernel = pick<FEET>(pick<PLAN>(pick<ENV_MODEL>(mpc_fallback_kernel<H>, mpc_fallback_model_kernel<H>),
                                                     mpc_fallback_plan_kernel<H>),
                                          mpc_fallback_feet_kernel<H>);
  const size_t smem = sizeof(Smem<H>);
  RgMpcScratch* scratch = (RgMpcScratch*)((char*)ws + RG_MPC_SCRATCH_OFFSET);
  auto launch = [&](auto kernel, int grid, bool programmatic) {
    if constexpr (FEET)
      return rg_launch(kernel, dim3((unsigned)grid), dim3((unsigned)Cfg<H>::NT), smem, stream, programmatic, ws, scratch, n_env, io, model, plan, feet);
    else if constexpr (PLAN)
      return rg_launch(kernel, dim3((unsigned)grid), dim3((unsigned)Cfg<H>::NT), smem, stream, programmatic, ws, scratch, n_env, io, model, plan);
    else if constexpr (ENV_MODEL)
      return rg_launch(kernel, dim3((unsigned)grid), dim3((unsigned)Cfg<H>::NT), smem, stream, programmatic, ws, scratch, n_env, io, model);
    else
      return rg_launch(kernel, dim3((unsigned)grid), dim3((unsigned)Cfg<H>::NT), smem, stream, programmatic, ws, scratch, n_env, io);
  };
  int rc;
  const int slots = sm_count() * Cfg<H>::MIN_BLOCKS;     // CTAs resident at once
  // A batch that fits one wave gains nothing from the split (every env has an SM slot of its own from the start):
  // one launch of the complete kernel instead of two -- this is the small-N latency path.
  if (two_kernel && n_env > slots) {
    // lean active-set kernel on every env, then the complete solver on whatever it queued
    rc = configure_kernel((const void*)lean_kernel, smem, Cfg<H>::MIN_BLOCKS, "cudaFuncSetAttribute(mpc_solve_kernel lean)");
    if (rc != RG_OK) return rc;
    rc = configure_kernel((const void*)fallback_kernel, smem, Cfg<H>::MIN_BLOCKS, "cudaFuncSetAttribute(mpc_fallback_kernel)");
    if (rc != RG_OK) return rc;
    rc = rg_check_cuda(launch(lean_kernel, n_env, chained), "mpc_solve_kernel (lean) launch");
    rg_count_launch();
    if (rc != RG_OK) return rc;
    const int grid = n_env < slots ? n_env : slots;       // as many CTAs as fit at once: an empty queue costs one wave of exits
    // Programmatic dependent launch: every lean CTA signals at its start, so once the last one HAS STARTED the fallback
    // grid may take the slots the draining lean grid leaves free; its CTAs block in griddepcontrol.wait until the lean
    // grid has completed (queue visible).  The launch latency of the second kernel hides behind the first one's tail.
    rc = rg_check_cuda(launch(fallback_kernel, grid, true), "mpc_fallback_kernel launch");
    rg_count_launch();
    return rc;
  }
  rc = configure_kernel((const void*)full_kernel, smem, Cfg<H>::MIN_BLOCKS, "cudaFuncSetAttribute(mpc_solve_kernel)");
  if (rc != RG_OK) return rc;
  rc = rg_check_cuda(launch(full_kernel, n_env, chained), "mpc_solve_kernel launch");
  rg_count_launch();
  return rc;
}

// model: NULL selects the model-free kernels; plan: non-NULL selects the schedule kernels (NULL model = the workspace's);
// feet (only with a plan): non-NULL selects the foothold kernels
template <int H>
int launch_h(const RgMpcDev* ws, int n_env, const rg_mpc_io& io, int two_kernel, cudaStream_t stream, int chained,
             const rg_mpc_env_model* model, const uint8_t* plan, const float* feet) {
  if (plan && feet)
    return launch_kernels<H, true, true, true>(ws, n_env, io, two_kernel, stream, chained,
                                               model ? *model : rg_mpc_env_model{nullptr, nullptr, nullptr}, plan, feet);
  if (plan)
    return launch_kernels<H, true, true>(ws, n_env, io, two_kernel, stream, chained,
                                         model ? *model : rg_mpc_env_model{nullptr, nullptr, nullptr}, plan);
  if (model) return launch_kernels<H, true>(ws, n_env, io, two_kernel, stream, chained, *model);
  return launch_kernels<H, false>(ws, n_env, io, two_kernel, stream, chained, rg_mpc_env_model{nullptr, nullptr, nullptr});
}



// ---- debug / self-test hook (not part of the public header): factor a dense SPD matrix given in
// row-major N6 x N6 and solve one right-hand side with the kernel's own Cholesky / sweep routines.
template <int H>
__global__ void __launch_bounds__(Cfg<H>::NT) chol_selftest_kernel(const double* __restrict__ a_dense,
                                                                   const double* __restrict__ rhs, double* __restrict__ x_out,
                                                                   double* __restrict__ l_out) {
  constexpr int N6 = Cfg<H>::N6;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  using SM = Smem<H, false>;
  SM& sm = *reinterpret_cast<SM*>(smem_raw);
  const int tid = threadIdx.x;
  if (tid < N6) {
    for (int k = 0; k <= tid; ++k) sm.psi[prow(tid) + k] = a_dense[tid * N6 + k];
  }
  __syncthreads();
  cholesky_rows<H>(sm, 0);
  if (tid < N6) sm.avec[tid] = rhs[tid];   // after the factorisation: avec / kvec are its scratch
  __syncthreads();
  if (tid < 32) tri_solve_warp0<H>(sm);
  __syncthreads();
  if (tid < N6) {
    x_out[tid] = sm.avec[tid];
    for (int k = 0; k < tid; ++k) l_out[tid * N6 + k] = sm.psi[prow(tid) + k];
    l_out[tid * N6 + tid] = 1.0 / sm.rdiag[tid];
  }
}

template <int H>
int chol_selftest_launch(const double* a, const double* b, double* x, double* l, cudaStream_t st) {
  const size_t smem = sizeof(Smem<H, false>);
  cudaError_t e = cudaFuncSetAttribute(chol_selftest_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return rg_check_cuda(e, "cudaFuncSetAttribute(chol_selftest_kernel)");
  chol_selftest_kernel<H><<<1, Cfg<H>::NT, smem, st>>>(a, b, x, l);
  return rg_check_cuda(cudaGetLastError(), "chol_selftest_kernel launch");
}

// The kernel's own Riccati routines on a caller-supplied system: k1[6], k2ang[9], k2lin[3] = blocks of the stage
// cost; d[h][21] = packed lower triangles of the D_t; b[6h] -> v[6h] with (K^-1 + blkdiag D_t) v = b.
template <int H>
__global__ void __launch_bounds__(32) riccati_selftest_kernel(const double* __restrict__ k1, const double* __restrict__ k2ang,
                                                              const double* __restrict__ k2lin, const double* __restrict__ d,
                                                              const double* __restrict__ b, double* __restrict__ v_out,
                                                              int* __restrict__ flag_out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  using SM = Smem<H, true>;
  SM& sm = *reinterpret_cast<SM*>(smem_raw);
  const int tid = threadIdx.x;
  if (tid < 6) sm.k1[tid] = k1[tid];
  if (tid < 9) sm.k2ang[tid] = k2ang[tid];
  if (tid < 3) sm.k2lin[tid] = k2lin[tid];
  for (int i = tid; i < 21 * H; i += blockDim.x) sm.nblk[i / 21][i % 21] = d[i];
  for (int i = tid; i < 6 * H; i += blockDim.x) sm.avec[i] = b[i];
  if (tid == 0) sm.solver_warp = 0;
  __syncwarp();
  riccati_factor<H>(sm);
  __syncwarp();
  riccati_solve<H>(sm);
  __syncwarp();
  for (int i = tid; i < 6 * H; i += blockDim.x) v_out[i] = sm.avec[i];
  if (tid == 0) *flag_out = sm.flag;
}

template <int H>
int riccati_selftest_launch(const double* k1, const double* k2ang, const double* k2lin, const double* d, const double* b,
                            double* v, int* flag, cudaStream_t st) {
  const size_t smem = sizeof(Smem<H, true>);
  cudaError_t e = cudaFuncSetAttribute(riccati_selftest_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return rg_check_cuda(e, "cudaFuncSetAttribute(riccati_selftest_kernel)");
  riccati_selftest_kernel<H><<<1, 32, smem, st>>>(k1, k2ang, k2lin, d, b, v, flag);
  return rg_check_cuda(cudaGetLastError(), "riccati_selftest_kernel launch");
}

}  // namespace

extern "C" int rg_debug_chol_solve(int horizon, const double* a_dense, const double* rhs, double* x_out, double* l_out, void* stream) {
  switch (horizon) {
    case 5: return chol_selftest_launch<5>(a_dense, rhs, x_out, l_out, (cudaStream_t)stream);
    case 10: return chol_selftest_launch<10>(a_dense, rhs, x_out, l_out, (cudaStream_t)stream);
    case 20: return chol_selftest_launch<20>(a_dense, rhs, x_out, l_out, (cudaStream_t)stream);
    default: rg_set_error("unsupported horizon %d", horizon); return RG_ERR_UNSUPPORTED;
  }
}

extern "C" int rg_debug_riccati_solve(int horizon, const double* k1, const double* k2ang, const double* k2lin, const double* d,
                                      const double* b, double* v_out, int* flag_out, void* stream) {
  switch (horizon) {
    case 5: return riccati_selftest_launch<5>(k1, k2ang, k2lin, d, b, v_out, flag_out, (cudaStream_t)stream);
    case 10: return riccati_selftest_launch<10>(k1, k2ang, k2lin, d, b, v_out, flag_out, (cudaStream_t)stream);
    case 20: return riccati_selftest_launch<20>(k1, k2ang, k2lin, d, b, v_out, flag_out, (cudaStream_t)stream);
    default: rg_set_error("unsupported horizon %d", horizon); return RG_ERR_UNSUPPORTED;
  }
}

int rg_launch_mpc(const RgMpcDev* ws, int horizon, int n_env, const rg_mpc_io& io, int two_kernel, cudaStream_t stream, int chained,
                  const rg_mpc_env_model* model, const uint8_t* plan, const float* feet) {
  switch (horizon) {
    case 5: return launch_h<5>(ws, n_env, io, two_kernel, stream, chained, model, plan, feet);
    case 10: return launch_h<10>(ws, n_env, io, two_kernel, stream, chained, model, plan, feet);
    case 20: return launch_h<20>(ws, n_env, io, two_kernel, stream, chained, model, plan, feet);
    default:
      rg_set_error("unsupported horizon %d (kernels are built for 5, 10, 20)", horizon);
      return RG_ERR_UNSUPPORTED;
  }
}
