// batchp.cu -- persistent batch engine: ONE CTA owns one QP instance for its whole solve (BASELINE config 4).
//
// The lock-step engine (batch.cu) advances all instances together, one launch per step and one host poll per
// iteration; every instance then pays for the slowest one and for ~30 launches per iteration.  Here a single kernel
// launch solves the whole batch: CTAs pull instance indices from an atomic work queue, run the complete QPALM loop of
// src/qpalm.c:484-711 for that instance (residuals, termination, outer updates, active set, Newton system, exact
// line search) with block-level barriers between the steps, and take the next instance when done.  There is no host
// synchronisation inside a solve and no instance waits for another.
//
// Memory plan (B200): the shared A' (n x m), A (m x n) and D Q D (n x n) are read by every CTA and stay in the 126 MB L2; the
// per-instance H / L (n x n lower, column-major) and vectors are touched by one CTA only.  At 512 instances the factors
// (2 x 230 KB each) do not fit the L2 and stream from HBM, which is why every pass over them is written as a batch of
// requests (cp.async, eight loads in flight, rows requested one block ahead) rather than load -> use.  Shared memory per CTA
// (72 KB at 3 CTAs / SM, 55 KB at 4) holds one panel of the factor (Cholesky, triangular solves), the SYRK's double-buffered rows of A' -- or, during an
// update sweep, the rows of W, the chain warp's ring of window blocks and the row owners' staging ring --, the line search's
// two merge-sort buffers of (key, position) pairs (its nL <= 2m <= 2048 breakpoints s > 0) and the staged GEMV operand.
//
// The Newton system (Q + A_J' Sigma_J A_J + I/gamma) d = -dphi  (src/newton.c:96-118, solver_interface.c:319-519):
//   H is kept per instance and updated incrementally (+ entering / - leaving / +- sigma changes) or rebuilt from c Q by an in-CTA
//   tile-stationary SYRK (cta_syrk), L <- chol(H + beta I) by an in-CTA right-looking blocked Cholesky (each panel as a dataflow: a chain warp
//   on the diagonal, every other thread the owner of one panel row, per-column mbarriers); SYRK and trailing updates run on the FP64 tensor pipe (mma.sync m8n8k4, 16 x 16
//   tiles per warp); then two blocked triangular solves.  When the active set changes by at most min(0.1 (n + m),
//   max_rank_update) rows -- and at most 40, see p_control -- and the factor is current, the factor is UPDATED in place instead
//   (cta_updown_sweep: <= 8 ranks per sweep, entering rows before leaving rows; a chain warp on the diagonal, every other thread
//   the owner of one row, per-column mbarriers), where the reference takes cholmod_updown (newton.c:98-108).  All arithmetic is
//   fp64 FMA / DMMA.
#include "batch.cuh"
#include "chol32.cuh"
#include <math.h>
#include <string.h>
#ifdef QB_BP_DEBUG   // device-side checks of the engine's invariants (-DQB_BP_DEBUG through QB_EXTRA_FLAGS)
#include <assert.h>
#endif

using namespace qb;

// Build-time shape of a CTA; this file is compiled twice (build.sh), and each shape once more with -DQB_BP_PROBE, which
// replaces the solver kernel by the test probes of its building blocks (see kbp_probe_newton):
//   default            8 warps, 32-column panel: 80 registers x 256 threads, 72 KB -> 3 CTAs / SM (444
//                      slots on a B200).  Best per-wave throughput: 444 instances in 57.9 ms (7675 solves/s), 4096 instances
//                      in 488 ms (8396 solves/s) at the end of round 2.
//   -DQB_BP_VARIANT4   8 warps, 24-column panel, registers capped at 64: 55 KB -> 4 CTAs / SM
//                      (592 slots).  Both sort buffers (40 KB) fit the union region of either shape.  Slower per
//                      instance (64 registers: several loops are shaped around that, see p_gemv_rows) but the
//                      BASELINE sweep of 512 instances per GPU fits in ONE wave: 78.8 ms against 90.3 ms with the 68-instance
//                      tail of the default shape.  batch.cu picks it when 3 * SMs < nb <= 4 * SMs.
// Other shapes measured in round 1 (512 instances): 192 threads / PW 24 / 4 per SM 138.6 ms; 192 / PW 16 / 4 per SM
// 147.7 ms; 256 / PW 16 / 64 regs / 4 per SM 133.0 ms; 192 threads / PW 32 / 3 per SM 192.5 ms (fewer threads per CTA
// cost more than the extra occupancy buys); 4-per-SM shape with 224 threads (72 registers) 142.8 ms, with 288 threads
// (56 registers) 145.9 ms.  (The update sweep of round 2 maps thread t to row t of L: NT >= n.)
#ifdef QB_BP_VARIANT4
#define QB_BP_NAMESPACE bp4
#define QB_BP_SUPPORTED batchp4_supported
#define QB_BP_SOLVE batchp4_solve
#define QB_BP_PROBE_NEWTON batchp4_probe_newton
#define QB_BP_PROBE_SORT batchp4_probe_sort
#ifndef QB_BP_NT
#define QB_BP_NT 256
#endif
#ifndef QB_BP_PW
#define QB_BP_PW 24
#endif
#define QB_BP_MINB 4
#else
#define QB_BP_NAMESPACE bp
#define QB_BP_SUPPORTED batchp_supported
#define QB_BP_SOLVE batchp_solve
#define QB_BP_PROBE_NEWTON batchp_probe_newton
#define QB_BP_PROBE_SORT batchp_probe_sort
#endif
#ifdef QB_BP_PROBE   // the probe objects carry their own copy of the device code: keep its (host-stub) symbols apart
#undef QB_BP_NAMESPACE
#ifdef QB_BP_VARIANT4
#define QB_BP_NAMESPACE bp4_probe
#else
#define QB_BP_NAMESPACE bp_probe
#endif
#endif
#ifndef QB_BP_NT
#define QB_BP_NT 256
#endif
#ifndef QB_BP_PW
#define QB_BP_PW 32
#endif
namespace qb {
namespace QB_BP_NAMESPACE {

constexpr int NT = QB_BP_NT, NW = NT / 32;
constexpr int PW = QB_BP_PW;      // panel width (at most 32: the chain warp of the Cholesky holds a panel's diagonal rows)
constexpr int NMAX = 240;         // largest n of this engine (panel = PW x LDP doubles of shared memory)
static_assert(PW <= 32 && PW % 4 == 0, "one chain warp per panel; whole DMMA k-steps");
constexpr int LDP = NMAX + 1;     // odd leading dimension: conflict-free row and column access
static_assert(NMAX <= NT, "the update sweep maps thread t to row t of the factor");
constexpr int SORT_MAX = 2048;    // largest 2m
static_assert(SORT_MAX <= 8 * NT && SORT_MAX <= 65536, "the sort's register runs (8 per thread) cover SORT_MAX; positions fit 16 bits");
constexpr int VS_LEN = (QB_BP_PW == 32) ? 1024 : 960;   // staged GEMV operand (max(n, m) doubles)
// the line search's two ping-pong buffers of SORT_MAX (u64 key, u16 position) pairs (ls_keys / ls_pos)
constexpr size_t kSortBytes = (size_t)SORT_MAX * 2 * (sizeof(unsigned long long) + sizeof(unsigned short));
constexpr size_t kPanelBytes = sizeof(double) * PW * LDP;
constexpr size_t kUnionBytes = kSortBytes > kPanelBytes ? kSortBytes : kPanelBytes;
constexpr size_t kSmemBytes = kUnionBytes + sizeof(double) * (VS_LEN + NMAX + 16 + 2 * PW);

#define BSC(b, slot) P.scal[(size_t)(b) * S_COUNT + (slot)]

struct Args {
  int nb, n, m, ld;
  BSet st;
  const double *At, *Am, *Qs, *D, *Dinv, *E, *Einv;   // Am: A as m x n column-major (A d row-parallel), At: A' (n x m)
  const double *q_raw, *bmin_raw, *bmax_raw;
  double *x_out, *y_out;
  double *q, *bmin, *bmax, *x, *y, *Ax, *Qx, *Aty, *x_prev, *x0, *sigma, *sigma_inv, *sqrt_sigma, *Axys, *z, *pri_res, *pri_res_in,
      *yh, *Atyh, *df, *dphi, *d, *Qd, *Ad;
  int *active, *active_old, *active_cand, *activeH, *list_pos, *list_neg;
  double *sigmaH, *w_pos, *w_neg;
  double *H, *L, *rdiag;
  long long sLL, sR;
  double *ls_da, *ls_db;
  double *scal;
  BCtl *ctl;
  int *queue;
  long long *prof;   // optional [nb][16] per-phase clock64 totals (QPALM_B200_BATCH_PROF=1)
  int nwarm;                         // instances b < nwarm start from the rows of x_ws / y_ws (either may be null: that part cold)
  const double *x_ws, *y_ws;         // unscaled, [nb][n] / [nb][m]
};

struct Flags { int outer, sigma, inner, refac, factor, fq, boost, done, updown; };

struct Smem {
  unsigned char *u;      // union region: sort buffers / panel
  double *panel;         // PW x LDP
  double *vs;            // staged vector (VS_LEN)
  double *v;             // Newton rhs / solution (NMAX + 16)
  double *rd;            // 1 / l_jj of the current panel (PW), spare (PW)
};
// the line search's (key, position) buffers 0 and 1 in the union region (kSortBytes)
__device__ __forceinline__ unsigned long long *ls_keys(const Smem &S, int buf) {
  return reinterpret_cast<unsigned long long *>(S.u) + (size_t)buf * SORT_MAX;
}
__device__ __forceinline__ unsigned short *ls_pos(const Smem &S, int buf) {
  return reinterpret_cast<unsigned short *>(S.u + 2 * SORT_MAX * sizeof(unsigned long long)) + (size_t)buf * SORT_MAX;
}

// ------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------
#define RED_OUT(op, val, slot) { const double r_ = block_red<op>(val, scratch); if (threadIdx.x == 0) BSC(b, slot) = r_; }

// K block reductions behind ONE pair of barriers (block_red pays two barriers per value: p_res_m alone had 22).  Stage 1 is
// block_red's warp butterfly; stage 2 replays, in one thread per value, the tree that block_red's second butterfly forms over
// the per-warp partials (lanes >= NW hold the identity there), so every result is bit-identical to block_red's.
constexpr int RED_MULTI_MAX = 12;
__device__ __forceinline__ double red_dyn(int op, double a, double b) { return op == RED_SUM ? a + b : (op == RED_MAX ? fmax(a, b) : fmin(a, b)); }
template <int K>
__device__ __forceinline__ void block_red_multi(const Args &P, int b, const double (&val)[K], const int (&op)[K], const int (&slot)[K], double *part_buf) {
  static_assert(K <= RED_MULTI_MAX && NW <= 8 && RED_MULTI_MAX * 8 <= VS_LEN, "partials live in the staged-vector buffer (free between phases)");
  double (*part)[8] = reinterpret_cast<double (*)[8]>(part_buf);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();   // the previous user of part[] is done
#pragma unroll
  for (int k = 0; k < K; k++) {
    double x = val[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x = red_dyn(op[k], x, __shfl_xor_sync(0xffffffffu, x, o));
    if (lane == 0) part[k][wid] = x;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < K; k++) {
    if (threadIdx.x == (k % NW) * 32 + k / NW) {
      double a[8];
#pragma unroll
      for (int w = 0; w < 8; w++) a[w] = (w < NW) ? part[k][w] : (op[k] == RED_SUM ? 0.0 : (op[k] == RED_MAX ? -1.0e300 : 1.0e300));
#pragma unroll
      for (int o = 4; o > 0; o >>= 1)
#pragma unroll
        for (int i = 0; i < o; i++) a[i] = red_dyn(op[k], a[i], a[i + o]);
      BSC(b, slot[k]) = a[0];
    }
  }
}

__device__ __noinline__ void p_init(const Args &P, int b, double *scratch) {
  __shared__ double cc_s, sig_s;
  const int n = P.n, m = P.m, tid = threadIdx.x;
  const BSet &st = P.st;
  const size_t on = (size_t)b * n, om = (size_t)b * m;
  double mx = 0.0;
  for (int i = tid; i < n; i += NT) {   // q <- c * (D .* q), c = 1 / max(1, |D q|inf)   (scaling.c:82-90, Qx = 0 at setup)
    double v = P.q_raw[on + i];
    if (st.scaling) v = P.D[i] * v;
    P.q[on + i] = v;
    mx = fmax(mx, fabs(v));
  }
  mx = block_red<RED_MAX>(mx, scratch);
  if (tid == 0) cc_s = st.scaling ? 1 / fmax(1.0, mx) : 1.0;
  __syncthreads();
  const double cc = cc_s;
  for (int i = tid; i < n; i += NT) {
    if (st.scaling) P.q[on + i] *= cc;
    P.x[on + i] = 0; P.Qx[on + i] = 0; P.Aty[on + i] = 0; P.x_prev[on + i] = 0; P.x0[on + i] = 0; P.Qd[on + i] = 0; P.d[on + i] = 0;
  }
  double dist2 = 0.0;
  for (int i = tid; i < m; i += NT) {
    double lo = P.bmin_raw[om + i], hi = P.bmax_raw[om + i];
    if (st.scaling) { lo = P.E[i] * lo; hi = P.E[i] * hi; }
    P.bmin[om + i] = lo; P.bmax[om + i] = hi;
    P.y[om + i] = 0; P.Ax[om + i] = 0; P.Ad[om + i] = 0; P.pri_res_in[om + i] = 0;
    P.active[om + i] = 0; P.active_old[om + i] = 0; P.activeH[om + i] = 0;
    const double t = 0.0 - fmax(lo, fmin(0.0, hi));
    dist2 += t * t;
  }
  dist2 = block_red<RED_SUM>(dist2, scratch);
  if (tid == 0) {
    double s = st.sigma_init * 1.0 / fmax(1.0, 0.5 * dist2);   // f = 0 at x = 0 (iteration.c:50-58)
    s = fmax(1e-4, fmin(s, 1e4));
    sig_s = s;
    BCtl c;
    memset(&c, 0, sizeof(c));
    c.reset_newton = 1; c.gamma = st.gamma_init; c.gamma_prev = st.gamma_init; c.eps_abs_in = st.eps_abs_in; c.eps_rel_in = st.eps_rel_in;
    c.c = cc; c.cinv = 1.0 / cc; c.status = QPALM_UNSOLVED;
    P.ctl[b] = c;
    for (int k = 0; k < S_COUNT; k++) BSC(b, k) = 0.0;
  }
  __syncthreads();
  const double s = sig_s;
  for (int i = tid; i < m; i += NT) { P.sigma[om + i] = s; P.sigma_inv[om + i] = 1.0 / s; P.sqrt_sigma[om + i] = sqrt(s); }
}

// compute_residuals (iteration.c:24-48) + candidate active set (newton.c:122-149) + m-side termination reductions
__device__ __noinline__ void p_res_m(const Args &P, int b, double *part) {
  const int m = P.m, scaling = P.st.scaling;
  const size_t om = (size_t)b * m;
  double r_pri = 0, r_raw = 0, r_ax = 0, r_z = 0, r_edy = 0, oob = 0, adx_max = -1.0e300, adx_min = 1.0e300;
  double n_act = 0, n_ent = 0, n_lea = 0;
  for (int i = threadIdx.x; i < m; i += NT) {
    const double ax = P.Ax[om + i], yi = P.y[om + i], lo = P.bmin[om + i], hi = P.bmax[om + i];
    double t = yi * P.sigma_inv[om + i];
    const double axys = ax + t;
    const double zi = fmax(lo, fmin(axys, hi));
    const double pr = ax - zi;
    t = pr * P.sigma[om + i];
    const double yhi = yi + t;
    P.Axys[om + i] = axys; P.z[om + i] = zi; P.pri_res[om + i] = pr; P.yh[om + i] = yhi;
    const int act = (axys <= lo) || (axys >= hi);
    const int old = P.active_old[om + i];
    P.active_cand[om + i] = act;
    n_act += act; n_ent += (act && !old); n_lea += (!act && old);
    const double ei = scaling ? P.E[i] : 1.0, einv = scaling ? P.Einv[i] : 1.0;
    r_pri = fmax(r_pri, fabs(einv * pr)); r_raw = fmax(r_raw, fabs(pr));
    r_ax = fmax(r_ax, fabs(einv * ax)); r_z = fmax(r_z, fabs(einv * zi));
    const double dy = yhi - yi;
    r_edy = fmax(r_edy, fabs(ei * dy));
    const bool hi_fin = hi < ei * kInf, lo_fin = lo > -ei * kInf;
    oob += hi_fin ? hi * fmax(dy, 0.0) : 0.0;
    oob += lo_fin ? lo * fmin(dy, 0.0) : 0.0;
    const double adx = einv * P.Ad[om + i];
    if (hi_fin) adx_max = fmax(adx_max, adx);
    if (lo_fin) adx_min = fmin(adx_min, adx);
  }
  const double vals[11] = {r_pri, r_raw, r_ax, r_z, r_edy, oob, adx_max, adx_min, n_act, n_ent, n_lea};
  const int ops[11] = {RED_MAX, RED_MAX, RED_MAX, RED_MAX, RED_MAX, RED_SUM, RED_MAX, RED_MIN, RED_SUM, RED_SUM, RED_SUM};
  const int slots[11] = {S_PRI_RES, S_PRI_RES_RAW, S_NORM_AX, S_NORM_Z, S_NORM_EDY, S_OOB, S_ADX_MAX, S_ADX_MIN, S_NB_ACTIVE, S_NB_ENTER, S_NB_LEAVE};
  block_red_multi<11>(P, b, vals, ops, slots, part);
}

// out[i] = scale * sum_k M[i + ld*k] v[k], i < nrows (row sums of a shared column-major matrix: A'yh, Q d and, with the
// m x n copy of A, A d).  Each thread owns up to 4 rows (i, i + NT, ...) and walks the columns with 4-way unrolling, so
// 16 independent L2 requests are in flight per thread; per-row summation order is fixed (reproducible).
template <int RP, int KU>
__device__ __forceinline__ void gemv_rows_body(int nrows, int ncols, int ld, const double *__restrict__ M, double *out, double scale,
                                               const double *vs) {
  const int tid = threadIdx.x;
  for (int i0 = tid; i0 < nrows; i0 += RP * NT) {
    int ri[RP];
#pragma unroll
    for (int a = 0; a < RP; a++) { ri[a] = i0 + a * NT; if (ri[a] >= nrows) ri[a] = nrows - 1; }
    double acc[RP][KU];
#pragma unroll
    for (int a = 0; a < RP; a++)
#pragma unroll
      for (int u = 0; u < KU; u++) acc[a][u] = 0.0;
    int k = 0;
    for (; k + KU - 1 < ncols; k += KU) {
#pragma unroll
      for (int u = 0; u < KU; u++) {
        const double vk = vs[k + u];
        const double *col = M + (size_t)(k + u) * ld;
#pragma unroll
        for (int a = 0; a < RP; a++) acc[a][u] = fma(col[ri[a]], vk, acc[a][u]);
      }
    }
    for (; k < ncols; k++) {
      const double vk = vs[k];
      const double *col = M + (size_t)k * ld;
#pragma unroll
      for (int a = 0; a < RP; a++) acc[a][0] = fma(col[ri[a]], vk, acc[a][0]);
    }
#pragma unroll
    for (int a = 0; a < RP; a++) {
      double t = 0.0;
#pragma unroll
      for (int u = KU - 1; u >= 0; u--) t += acc[a][u];
      if (i0 + a * NT < nrows) out[i0 + a * NT] = t * scale;
    }
  }
}
// The same product for an EVEN number of rows <= NT with an even leading dimension (A' yh and Q d: n rows).  A thread owns a PAIR
// of rows (one 16-byte load per column) and one of G = NT / (nrows / 2) interleaved column groups, so all NT threads have eight
// 16-byte requests in flight (the one-row-per-thread form had 240 threads x 8 x 8 bytes: the kernel's hottest line, waiting on
// the L2, profiles/r02g_ncu_source_kbp_solve.txt).  Four accumulators per row, the groups' partial sums are added in group order:
// fixed summation order, reproducible.  `part` holds G x nrows doubles of shared memory.
__device__ __forceinline__ void gemv_rowpairs_body(int nrows, int ncols, int ld, const double *__restrict__ M, double *out, double scale,
                                                   const double *vs, double *part) {
  const int tid = threadIdx.x, np = nrows >> 1, G = NT / np;
  const int g = tid / np, p = tid - g * np;
  if (g < G) {
    double2 acc[4];
#pragma unroll
    for (int u = 0; u < 4; u++) acc[u] = make_double2(0.0, 0.0);
    const double *Mp = M + 2 * p;
    int k0 = g * 8;
    for (; k0 + 7 < ncols; k0 += G * 8) {
      double2 a[8];
#pragma unroll
      for (int u = 0; u < 8; u++) a[u] = *reinterpret_cast<const double2 *>(Mp + (size_t)(k0 + u) * ld);
#pragma unroll
      for (int u = 0; u < 8; u++) {
        const double vk = vs[k0 + u];
        acc[u & 3].x = fma(a[u].x, vk, acc[u & 3].x);
        acc[u & 3].y = fma(a[u].y, vk, acc[u & 3].y);
      }
    }
    for (int k = k0; k < ncols && k < k0 + 8; k++) {   // this group's ragged last block
      const double2 a = *reinterpret_cast<const double2 *>(Mp + (size_t)k * ld);
      const double vk = vs[k];
      acc[0].x = fma(a.x, vk, acc[0].x);
      acc[0].y = fma(a.y, vk, acc[0].y);
    }
    part[g * nrows + 2 * p] = (acc[3].x + acc[2].x) + (acc[1].x + acc[0].x);
    part[g * nrows + 2 * p + 1] = (acc[3].y + acc[2].y) + (acc[1].y + acc[0].y);
  }
  __syncthreads();
  for (int i = tid; i < nrows; i += NT) {
    double t = 0.0;
    for (int gg = G - 1; gg >= 0; gg--) t += part[gg * nrows + i];
    out[i] = t * scale;
  }
}
__device__ __forceinline__ void p_gemv_rows(int nrows, int ncols, int ld, const double *__restrict__ M, const double *__restrict__ v,
                                            double *out, double scale, const Smem &S) {
  for (int k = threadIdx.x; k < ncols; k += NT) S.vs[k] = v[k];
  __syncthreads();
  if (!(nrows & 1) && !(ld & 1) && nrows >= 2 && (nrows >> 1) <= NT)
    gemv_rowpairs_body(nrows, ncols, ld, M, out, scale, S.vs, S.panel);               // row pairs x column groups (A' yh, Q d)
  else if (nrows <= NT) gemv_rows_body<1, 8>(nrows, ncols, ld, M, out, scale, S.vs);    // one row per thread, 8 columns in flight
#ifdef QB_BP_VARIANT4
  else gemv_rows_body<4, 2>(nrows, ncols, ld, M, out, scale, S.vs);               // 64 registers: 4 x 4 accumulators + 16 loads in flight spill in the loop
#else
  else gemv_rows_body<4, 4>(nrows, ncols, ld, M, out, scale, S.vs);               // 4 rows x 4 columns in flight
#endif
}
// out[k] = sum_i M[i + ld*k] v[i], k < ncols (column dots: A d with A' as M); one warp per column
__device__ __forceinline__ void p_gemv_cols(int len, int ncols, int ld, const double *__restrict__ M, const double *__restrict__ v, double *out,
                            const Smem &S) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int k = tid; k < len; k += NT) S.vs[k] = v[k];
  __syncthreads();
  // four columns per warp step: their loads are independent, so 4 x len/32 L2 requests are in flight per lane
  for (int col0 = warp * 4; col0 < ncols; col0 += NW * 4) {
    double acc[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const int col = (col0 + u < ncols) ? col0 + u : ncols - 1;
      const double *c = M + (size_t)col * ld;
      double a0 = 0, a1 = 0;
      int i = lane;
      for (; i + 32 < len; i += 64) { a0 = fma(c[i], S.vs[i], a0); a1 = fma(c[i + 32], S.vs[i + 32], a1); }
      for (; i < len; i += 32) a0 = fma(c[i], S.vs[i], a0);
      acc[u] = a0 + a1;
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const double r = warp_sum(acc[u]);
      if (lane == 0 && col0 + u < ncols) out[col0 + u] = r;
    }
  }
}

// warm start of instance b after p_init's cold start (qpalm_warm_start, qpalm.c:322-399, then initialize_sigma,
// iteration.c:50-84), in the engine's scaled storage: x = Dinv x_ws, y = c Einv y_ws, Qd = c (D Q D) x, Qx = Qd (+ x / gamma_init),
// Ad = Ax = A x, sigma from f = x'Qx / 2 + q'x and the bound distance of Ax.  Aty, d, the active sets and the control state
// keep their cold values, as a fresh setup leaves them.  Without x, Qx = Ax = 0 and the cold sigma stands.
__device__ __noinline__ void p_warm(const Args &P, int b, double *scratch, const Smem &S) {
  __shared__ double sig_s;
  const int n = P.n, m = P.m, tid = threadIdx.x;
  const BSet &st = P.st;
  const size_t on = (size_t)b * n, om = (size_t)b * m;
  const double cc = P.ctl[b].c;
  if (P.y_ws)
    for (int i = tid; i < m; i += NT) {
      double v = P.y_ws[om + i];
      if (st.scaling) { v = v * P.Einv[i]; v = v * cc; }
      P.y[om + i] = v;
    }
  if (!P.x_ws) return;
  for (int i = tid; i < n; i += NT) {
    double v = P.x_ws[on + i];
    if (st.scaling) v = v * P.Dinv[i];
    P.x[on + i] = v; P.x0[on + i] = v; P.x_prev[on + i] = v;
  }
  __syncthreads();
  p_gemv_rows(n, n, n, P.Qs, P.x + on, P.Qd + on, cc, S);
  __syncthreads();
  p_gemv_rows(m, n, m, P.Am, P.x + on, P.Ad + om, 1.0, S);
  __syncthreads();
  const double inv_g = 1 / st.gamma_init;
  double xqx = 0.0, qtx = 0.0, dist2 = 0.0;
  for (int i = tid; i < n; i += NT) {
    const double xi = P.x[on + i];
    double qx = P.Qd[on + i];
    if (st.proximal) qx = qx + inv_g * xi;
    P.Qx[on + i] = qx;
    xqx += xi * qx; qtx += P.q[on + i] * xi;
  }
  for (int i = tid; i < m; i += NT) {
    const double ax = P.Ad[om + i];
    P.Ax[om + i] = ax;
    const double t = ax - fmax(P.bmin[om + i], fmin(ax, P.bmax[om + i]));
    dist2 += t * t;
  }
  xqx = block_red<RED_SUM>(xqx, scratch);
  qtx = block_red<RED_SUM>(qtx, scratch);
  dist2 = block_red<RED_SUM>(dist2, scratch);
  if (tid == 0) {
    const double f = 0.5 * xqx + qtx;
    sig_s = fmax(1e-4, fmin(st.sigma_init * fmax(1.0, fabs(f)) / fmax(1.0, 0.5 * dist2), 1e4));
  }
  __syncthreads();
  const double s = sig_s;
  for (int i = tid; i < m; i += NT) { P.sigma[om + i] = s; P.sigma_inv[om + i] = 1.0 / s; P.sqrt_sigma[om + i] = sqrt(s); }
}

__device__ __noinline__ void p_res_n(const Args &P, int b, double *part) {
  const int n = P.n;
  const BSet &st = P.st;
  const size_t on = (size_t)b * n;
  const double gamma = P.ctl[b].gamma, neg_inv_gamma = -1 / gamma;
  const double neg_tau_over_gamma = -BSC(b, S_TAU) * (1 / gamma);
  double r_dua = 0, r_dua2 = 0, r_qx = 0, r_q = 0, r_atyh = 0, r_atdy = 0, r_ddx = 0, dxdx = 0, dxqdx = 0, qdx = 0;
  for (int j = threadIdx.x; j < n; j += NT) {
    const double qx = P.Qx[on + j], qj = P.q[on + j], xj = P.x[on + j], at = P.Atyh[on + j];
    double dfj = qx + qj;
    if (st.proximal) dfj = dfj + neg_inv_gamma * P.x0[on + j];
    const double dp = dfj + at;
    P.df[on + j] = dfj; P.dphi[on + j] = dp;
    const double dinv = st.scaling ? P.Dinv[j] : 1.0;
    if (st.proximal) {
      const double xx0 = xj - P.x0[on + j];
      const double t = dp + neg_inv_gamma * xx0;
      r_dua = fmax(r_dua, fabs(dinv * t));
    } else r_dua = fmax(r_dua, fabs(dinv * dp));
    r_dua2 = fmax(r_dua2, fabs(dinv * dp));
    r_qx = fmax(r_qx, fabs(dinv * qx)); r_q = fmax(r_q, fabs(dinv * qj)); r_atyh = fmax(r_atyh, fabs(dinv * at));
    r_atdy = fmax(r_atdy, fabs(dinv * (at - P.Aty[on + j])));
    const double dx = xj - P.x_prev[on + j];
    const double ddx = st.scaling ? P.D[j] * dx : dx;
    r_ddx = fmax(r_ddx, fabs(ddx));
    dxdx += ddx * ddx;
    if (st.proximal) { const double t2 = P.Qd[on + j] + neg_tau_over_gamma * P.d[on + j]; dxqdx += dx * t2; }
    else dxqdx += P.Qd[on + j] * dx;
    qdx += qj * dx;
  }
  const double vals[10] = {r_dua, r_dua2, r_qx, r_q, r_atyh, r_atdy, r_ddx, dxdx, dxqdx, qdx};
  const int ops[10] = {RED_MAX, RED_MAX, RED_MAX, RED_MAX, RED_MAX, RED_MAX, RED_MAX, RED_SUM, RED_SUM, RED_SUM};
  const int slots[10] = {S_DUA_RES, S_DUA2_RES, S_NORM_QX, S_NORM_Q, S_NORM_ATYH, S_NORM_ATDY, S_NORM_DDX, S_DXDX, S_DXQDX, S_QDX};
  block_red_multi<10>(P, b, vals, ops, slots, part);
}

// the control flow of qpalm_solve for one iteration (src/qpalm.c:484-711), executed by one thread
__device__ __noinline__ void p_control(const Args &P, int b, Flags &f) {
  const BSet &st = P.st;
  const int n = P.n, m = P.m;
  f.outer = f.sigma = f.inner = f.refac = f.factor = f.fq = f.boost = f.done = f.updown = 0;
  BCtl c = P.ctl[b];
  const double *h = P.scal + (size_t)b * S_COUNT;
  const double cinv = st.scaling ? c.cinv : 1.0;
  c.pri_res_norm = h[S_PRI_RES];
  c.dua_res_norm = h[S_DUA_RES] * cinv;
  c.dua2_res_norm = h[S_DUA2_RES] * cinv;
  const double nrm_axz = st.scaling ? h[S_NORM_AX] : fmax(h[S_NORM_AX], h[S_NORM_Z]);   // sic, termination.c:99
  c.eps_pri = st.eps_abs + st.eps_rel * nrm_axz;
  double max_norm = fmax(h[S_NORM_QX], fmax(h[S_NORM_Q], h[S_NORM_ATYH]));
  if (st.scaling) max_norm *= cinv;
  c.eps_dua = st.eps_abs + st.eps_rel * max_norm;
  c.eps_dua_in = c.eps_abs_in + c.eps_rel_in * max_norm;
  int term = 0;
  if ((c.pri_res_norm < c.eps_pri) && (c.dua_res_norm < c.eps_dua)) term = QPALM_SOLVED;
  else {
    const double eps_pinf = st.eps_prim_inf * h[S_NORM_EDY];
    if ((eps_pinf != 0) && (h[S_NORM_ATDY] <= eps_pinf) && (h[S_OOB] <= -eps_pinf)) term = QPALM_PRIMAL_INFEASIBLE;
    else {
      const double eps_dinf = st.eps_dual_inf * h[S_NORM_DDX];
      if (eps_dinf != 0) {
        const bool blocked = (m > 0) && ((h[S_ADX_MAX] >= eps_dinf) || (h[S_ADX_MIN] <= -eps_dinf));
        if (!blocked) {
          const double cc = st.scaling ? c.c : 1.0, e2 = st.eps_dual_inf * st.eps_dual_inf;
          if ((h[S_DXQDX] <= -cc * e2 * h[S_DXDX]) || ((h[S_DXQDX] <= cc * e2 * h[S_DXDX]) && (h[S_QDX] <= -cc * eps_dinf)))
            term = QPALM_DUAL_INFEASIBLE;
        }
      }
    }
  }
  if (term) { c.status = term; c.done = 1; P.ctl[b] = c; f.done = 1; return; }
  const int na = (m > 0) ? (int)h[S_NB_ACTIVE] : 0, ne = (m > 0) ? (int)h[S_NB_ENTER] : 0, nl = (m > 0) ? (int)h[S_NB_LEAVE] : 0;
  if ((c.dua2_res_norm <= c.eps_dua_in) || (c.no_change == 3)) {   // qpalm.c:515
    c.no_change = 0;
    f.outer = 1;
    if (c.iter_out > 0 && c.pri_res_norm > c.eps_pri) f.sigma = 1;
    c.eps_abs_in = fmax(st.eps_abs, st.rho * c.eps_abs_in);
    c.eps_rel_in = fmax(st.eps_rel, st.rho * c.eps_rel_in);
    c.gamma_prev = c.gamma;
    if (st.proximal) {
      const bool try_boost = !c.gamma_maxed && c.iter_out > 0 && c.nb_enter == 0 && c.nb_leave == 0 && c.pri_res_norm < c.eps_pri;
      if (try_boost) f.boost = 1;
      else if (c.gamma < st.gamma_max) { c.gamma = fmin(c.gamma * st.gamma_upd, st.gamma_max); c.reset_newton = 1; }
    }
    c.iter_out++; c.prev_iter = c.iter;
  } else if (c.iter == c.prev_iter + st.inner_max_iter) {   // qpalm.c:647-660
    c.no_change = 0;
    f.outer = 2;
    if (c.iter_out > 0 && c.pri_res_norm > c.eps_pri) f.sigma = 1;
    c.gamma_prev = c.gamma;
    if (st.proximal && c.gamma < st.gamma_max) { c.gamma = fmin(c.gamma * st.gamma_upd, st.gamma_max); c.reset_newton = 1; }
    c.iter_out++; c.prev_iter = c.iter;
  } else {   // inner step
    if (c.nb_enter + c.nb_leave) c.no_change = 0; else c.no_change++;
    if ((c.iter % st.reset_newton_iter) == 0) c.reset_newton = 1;
    c.nb_active = na; c.nb_enter = ne; c.nb_leave = nl;
    f.inner = 1;
    c.beta = st.proximal ? 1.0 / c.gamma : 0.0;
    const double rank_limit = fmin(st.max_rank_update_fraction * (double)(n + m), (double)st.max_rank_update);
    c.scratch = 0;
    if ((c.reset_newton && na) || (double)(ne + nl) > rank_limit) { f.refac = 1; f.factor = 1; c.scratch = (c.reset_newton && !st.batch_h_incremental) || !c.H_valid; }
    else if (na) {   // newton.c:103-108: rank update of the factor (entering rows, then leaving rows)
      if (ne + nl > 0) {
        // The reference updates the factor here whatever the rank (<= min(0.1 (n + m), 160) rows).  A sweep handles 8 ranks, so
        // beyond ~5 sweeps the incremental SYRK + refactorisation is the cheaper way to the SAME matrix: 512-instance sweep
        // 91.5 ms without the cap, 88.0 ms at 40 (88.8 / 88.8 / 88.2 / 90.6 ms at 24 / 32 / 48 / 56), iteration counts unchanged.
        if (st.batch_updown && ne + nl <= st.batch_updown_max_rank) f.updown = 1;
        else { f.refac = 1; f.factor = 1; c.scratch = !c.H_valid; }
      }
    }
    else { f.fq = 1; f.factor = 1; }
    c.reset_newton = 0;
    c.n_inner++;
    if (f.factor) { c.n_refac++; c.refac_J += na; }
  }
  P.ctl[b] = c;
}

// update_sigma (iteration.c:86-145); every sigma change leads to a refactorisation (same matrix as the reference's
// rank update of solver_interface.c:443-503)
__device__ __noinline__ void p_update_sigma(const Args &P, int b, double *scratch) {
  const int m = P.m;
  const BSet &st = P.st;
  const size_t om = (size_t)b * m;
  const double nrm = BSC(b, S_PRI_RES_RAW);
  double changed = 0;
  for (int k = threadIdx.x; k < m; k += NT) {
    const double pr = fabs(P.pri_res[om + k]);
    if ((pr > st.theta * fabs(P.pri_res_in[om + k])) && P.active[om + k]) {
      double mult = fmax(1.0, st.delta * pr / (nrm + 1e-6));
      const double sg = P.sigma[om + k], stmp = mult * sg;
      if (stmp <= st.sigma_max) {
        changed += (sg != stmp);
        P.sigma[om + k] = stmp; P.sigma_inv[om + k] = 1.0 / stmp;
        mult = sqrt(mult);
        P.sqrt_sigma[om + k] = mult * P.sqrt_sigma[om + k];
      } else {
        changed += (sg != st.sigma_max);
        P.sigma[om + k] = st.sigma_max; P.sigma_inv[om + k] = 1.0 / st.sigma_max; P.sqrt_sigma[om + k] = st.sqrt_sigma_max;
      }
    }
  }
  changed = block_red<RED_SUM>(changed, scratch);
  if (threadIdx.x == 0) {
    if ((st.proximal && P.ctl[b].gamma_prev < st.gamma_max) || changed > 0) P.ctl[b].reset_newton = 1;
  }
}

// y <- yh, Aty <- Atyh, Qx += (1/gamma - 1/gamma_prev) x, x0 <- x, pri_res_in <- pri_res (qpalm.c:525-526, 629, 635, 655, 658)
__device__ void p_outer(const Args &P, int b, int kind) {
  const int n = P.n, m = P.m;
  const size_t on = (size_t)b * n, om = (size_t)b * m;
  const double g = P.ctl[b].gamma, gp = P.ctl[b].gamma_prev;
  const double dg = (g != gp) ? (1 / g - 1 / gp) : 0.0;
  for (int i = threadIdx.x; i < m; i += NT) {
    if (kind == 1) P.y[om + i] = P.yh[om + i];
    P.pri_res_in[om + i] = P.pri_res[om + i];
  }
  for (int j = threadIdx.x; j < n; j += NT) {
    if (kind == 1) P.Aty[on + j] = P.Atyh[on + j];
    if (P.st.proximal) {
      if (dg != 0.0) P.Qx[on + j] = P.Qx[on + j] + dg * P.x[on + j];
      P.x0[on + j] = P.x[on + j];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// dense building blocks on an n x n lower matrix in global memory (L2 resident), panels in shared memory
// ------------------------------------------------------------------------------------------------
// dst(i, j) = [first ? sscale * src(i, j) + (i == j) * diag_add : dst(i, j)] + sign * sum_{c < w} U[c][i - u0] U[c][j - u0]
// for r0 <= j <= i < n.  U is PW x LDP in shared memory.  Warp task = 128 rows x 4 columns, 4 x 4 register block per lane.
// The accumulators START from the old values: all 16 global loads of a task are issued up front and their latency is
// paid once per task (a read-modify-write after the loop serialises 16 dependent L2 round trips: measured 6x slower).
// FP64 tensor-core tile of the in-CTA rank-w updates: d += a (8 x 4) * b (4 x 8), mma.sync m8n8k4 (DMMA)
__device__ __forceinline__ void bp_dmma884(double &d0, double &d1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// dst(i, j) = base(i, j) + sign * sum_{c < w} U[c][i] U[c][j]   for r0 <= j <= i < n   (the trailing update of the in-CTA
// Cholesky), base = first ? sscale * src + diag_add I : dst.  U = shared panel, column c at U + c * LDP - u0.
// Round 2: the products run on the FP64 tensor pipe.  Each warp takes 16 x 16 tiles of the lower triangle (2 x 2 DMMA tiles,
// round-robin over the warps); per 4 columns of U it loads two A and two B fragments from shared memory and issues four
// mma.sync.m8n8k4 -- a quarter of the shared-memory wavefronts and a sixth of the instructions of the 4 x 4 scalar register
// tile this replaces (which ran the FP64 pipe at 18 %).  The sign rides on the final add.
__device__ __forceinline__ void cta_rank_update_lower(double *dst, int ldd, const double *src, int lds, double sscale, double diag_add, bool first,
                                      int r0, int n, const double *U, int u0, int w, double sign) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int rem = n - r0;
  if (rem <= 0) return;
  const int T = (rem + 15) >> 4, ntiles = T * (T + 1) / 2;
  const int fr = lane >> 2, fk = lane & 3;
  const int wpad = (w + 3) & ~3;
  for (int q = warp; q < ntiles; q += NW) {
    int ib = (int)((sqrtf(8.0f * (float)q + 1.0f) - 1.0f) * 0.5f);
    while (ib * (ib + 1) / 2 > q) ib--;
    while ((ib + 1) * (ib + 2) / 2 <= q) ib++;
    const int jb = q - ib * (ib + 1) / 2;
    const int i0 = r0 + 16 * ib, j0 = r0 + 16 * jb;
    int ra[2], rb[2];   // fragment rows (clamped: rows beyond n read a valid address and are never stored)
#pragma unroll
    for (int t = 0; t < 2; t++) {
      ra[t] = i0 + 8 * t + fr; if (ra[t] >= n) ra[t] = n - 1;
      rb[t] = j0 + 8 * t + fr; if (rb[t] >= n) rb[t] = n - 1;
    }
    // the old values of the tile are requested BEFORE the product loop, so their L2 / DRAM latency hides under it (a
    // read-modify-write after the loop left every warp on the long scoreboard: 15 % of the kernel's stall samples in
    // profiles/r02f_ncu_source_kbp_solve.txt); the arithmetic is unchanged (base + sign * sum)
    double acc[2][2][2], base[2][2][2];
#pragma unroll
    for (int a = 0; a < 2; a++)
#pragma unroll
      for (int e = 0; e < 2; e++)
#pragma unroll
        for (int h = 0; h < 2; h++) {
          acc[a][e][h] = 0.0;
          const int i = i0 + 8 * a + fr, j = j0 + 8 * e + 2 * fk + h;
          double bv = 0.0;
          if (i < n && j < n && i >= j) {
            if (first) { bv = sscale * src[(size_t)i + (size_t)lds * j]; if (i == j) bv += diag_add; }
            else bv = dst[(size_t)i + (size_t)ldd * j];
          }
          base[a][e][h] = bv;
        }
    // fragment addresses once per tile; the callers zero the panel columns [w, wpad), so the product loop has no predicate and no
    // branch (the first version selected `c < w ? load : 0` per fragment: ~60 integer / branch instructions per four DMMAs)
    // 32-bit shared-window addresses (four registers instead of four 64-bit generic pointers: at 64 registers per thread the
    // pointers were spilled inside this loop)
    const unsigned ub = (unsigned)__cvta_generic_to_shared(U + fk * LDP - u0);
    const unsigned sa0 = ub + 8u * (unsigned)ra[0], sa1 = ub + 8u * (unsigned)ra[1], sb0 = ub + 8u * (unsigned)rb[0], sb1 = ub + 8u * (unsigned)rb[1];
#pragma unroll 3
    for (int kc = 0; kc < wpad; kc += 4) {
      const unsigned o = (unsigned)(kc * LDP * 8);
      double fa0, fa1, fb0, fb1;
      asm volatile("ld.shared.f64 %0, [%1];" : "=d"(fa0) : "r"(sa0 + o));
      asm volatile("ld.shared.f64 %0, [%1];" : "=d"(fa1) : "r"(sa1 + o));
      asm volatile("ld.shared.f64 %0, [%1];" : "=d"(fb0) : "r"(sb0 + o));
      asm volatile("ld.shared.f64 %0, [%1];" : "=d"(fb1) : "r"(sb1 + o));
      bp_dmma884(acc[0][0][0], acc[0][0][1], fa0, fb0);
      bp_dmma884(acc[0][1][0], acc[0][1][1], fa0, fb1);
      bp_dmma884(acc[1][0][0], acc[1][0][1], fa1, fb0);
      bp_dmma884(acc[1][1][0], acc[1][1][1], fa1, fb1);
    }
#pragma unroll
    for (int a = 0; a < 2; a++)
#pragma unroll
      for (int e = 0; e < 2; e++)
#pragma unroll
        for (int h = 0; h < 2; h++) {
          const int i = i0 + 8 * a + fr, j = j0 + 8 * e + 2 * fk + h;
          if (i < n && j < n && i >= j) dst[(size_t)i + (size_t)ldd * j] = fma(sign, acc[a][e][h], base[a][e][h]);
        }
  }
}

// cp.async (LDGSTS) 8-byte copy global -> shared.  A panel load requests ALL its elements before anything waits and holds
// no registers; the former `Pn[..] = L[..]` loop kept one or two loads in flight per thread and sat on the long scoreboard
// (the per-instance factors do not fit the L2: 15 % of the kernel's stall samples, profiles/r02f_ncu_source_kbp_solve.txt).
__device__ __forceinline__ void bp_cp_async8(double *smem_dst, const double *gsrc) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void bp_cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void bp_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bp_cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
// Pn[t][r] <- L(k0 + r, k0 + t) for t <= r < rows, t < w; zeros above the diagonal of the w x w block.  Rows fastest (coalesced).
// The caller's __syncthreads() publishes the panel.
__device__ __forceinline__ void panel_load_async(double *Pn, const double *L, int ld, int k0, int w, int rows) {
  for (int t = 0; t < w; t++) {
    const double *col = L + (size_t)k0 + (size_t)ld * (k0 + t);
    for (int r = threadIdx.x; r < rows; r += NT) {
      if (r >= t) bp_cp_async8(&Pn[t * LDP + r], col + r);
      else Pn[t * LDP + r] = 0.0;
    }
  }
  bp_cp_async_wait_all();
}

// Tile-stationary SYRK of the Newton matrix:
//   dst(i, j) = base(i, j) + sum_{e < npos} wpos[e]^2 a_e(i) a_e(j) - sum_{e < nneg} wneg[e]^2 a'_e(i) a'_e(j)   for j <= i < n,
// a_e = A'[:, lpos[e]], a'_e = A'[:, lneg[e]]; base = 0, dst itself, or sscale * src (lds): the zeroed Gershgorin matrix of
// p_boost, the incremental H record, the rebuild from c Q.  Both lists form ONE stream of signed weights s w^2, applied to the
// A fragment in registers.  The 16 x 16 tiles of the lower triangle are taken in passes over a group of 4 x 2 tiles (one per
// warp, its DMMA accumulators in registers) while the whole list streams past in stages of SY_C entries: each tile of dst is
// read once and written once, which matters because at 512 instances the per-instance H streams from HBM.  A stage
// holds only the rows of A' its group needs -- 64 rows for a diagonal group, 96 for an off-diagonal one -- gathered with
// 16-byte cp.async copies of whole 16-row segments (A' is L2-resident) into a double buffer: one barrier per stage.
constexpr int SY_BI = 4, SY_BJ = 2;               // a tile group: 4 i blocks x 2 j blocks of 16 rows, one tile per warp
constexpr int SY_LD = (SY_BI + SY_BJ) * 16 + 4;   // 100 rows per staged column: the fragment loads of a half warp hit 16 banks
constexpr int SY_C = (QB_BP_PW == 32) ? 36 : 24;  // list entries per stage (two stages + the list indices fill the union region)
static_assert(NW == SY_BI * SY_BJ, "one tile per warp");
static_assert(2 * SY_C * SY_LD * sizeof(double) + VS_LEN * sizeof(int) <= kUnionBytes, "two stages + the list indices must fit the union region");
enum { SY_ZERO = 0, SY_DST = 1, SY_SRC = 2 };

__device__ __forceinline__ void bp_cp_async16(double *smem_dst, const double *gsrc) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ double sy_lds(unsigned a) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
  return v;
}

// The job of one cta_syrk call, in shared memory: the loops reload what they need after each barrier, so that little more
// than the tile's accumulators stays in registers across a stage.  With the arguments in registers, or with one flat loop over
// (group, stage), ptxas kept the accumulators in local memory around the product loop at 64 and at 80 registers alike.
struct SyJob {
  double *dst; const double *src, *At; long long *pf; double sscale;
  int ld, lds, n, base, cnt, nst, vec16;
};

// stage `st` of group (gi, gj) into buf: columns c < SY_C = list entries st SY_C + c (entries past the list read column 0 of A'
// and carry weight 0), rows = the group's j blocks at 16 sl (sl < SY_BJ), its i blocks at 16 (SY_BJ + sl).  Rows >= n are not
// copied: they only reach tile entries that are never stored.
__device__ __forceinline__ void sy_gather(double *buf, const SyJob &J, const int *lidx, int st, int gi, int gj) {
  const bool diag = SY_BJ * gj >= SY_BI * gi;
  const int per = diag ? SY_BI * 8 : (SY_BI + SY_BJ) * 8;   // 16-byte copies per staged column
  const int n = J.n, cnt = J.cnt;
  const double *At = J.At;
  for (int q = threadIdx.x; q < SY_C * per; q += NT) {
    const int c = diag ? q / (SY_BI * 8) : q / ((SY_BI + SY_BJ) * 8), r = q - c * per;
    const int sl = (diag ? SY_BJ : 0) + (r >> 3), h = r & 7;
    const int row = 16 * (sl < SY_BJ ? SY_BJ * gj + sl : SY_BI * gi + sl - SY_BJ) + 2 * h;
    if (row < n) {
      const int e = st * SY_C + c;
      const double *g = At + (size_t)n * (size_t)(e < cnt ? lidx[e] : 0) + row;
      double *d = buf + c * SY_LD + 16 * sl + 2 * h;
      if (J.vec16) bp_cp_async16(d, g);
      else { bp_cp_async8(d, g); if (row + 1 < n) bp_cp_async8(d + 1, g + 1); }
    }
  }
  bp_cp_async_commit();
}

__device__ __forceinline__ void cta_syrk(double *dst, int ld, int n, int base, const double *src, int lds, double sscale,
                                      const double *__restrict__ At, const int *lpos, const double *wpos, int npos, const int *lneg,
                                      const double *wneg, int nneg, const Smem &S, long long *pf) {
  __shared__ SyJob J;
  const int tid = threadIdx.x;
  const int cnt = npos + nneg, nst = (cnt + SY_C - 1) / SY_C;
  if (nst == 0) {   // empty list: dst = base
    if (base != SY_DST)
      for (int idx = tid; idx < n * n; idx += NT) {
        const int j = idx / n, i = idx - j * n;
        if (i >= j) dst[(size_t)i + (size_t)ld * j] = (base == SY_SRC) ? sscale * src[(size_t)i + (size_t)lds * j] : 0.0;
      }
    __syncthreads();
    return;
  }
  double *buf0 = S.panel;
  int *lidx = reinterpret_cast<int *>(S.panel + 2 * SY_C * SY_LD);
  double *sw = S.vs;   // signed weights, padded with zeros to nst SY_C entries (runs on into S.v, free during the SYRK)
  for (int e = tid; e < nst * SY_C; e += NT) {
    double v = 0.0;
    if (e < cnt) {
      const bool p = e < npos;
      const double w = p ? wpos[e] : wneg[e - npos];
      lidx[e] = p ? lpos[e] : lneg[e - npos];
      v = p ? w * w : -(w * w);
    }
    sw[e] = v;
  }
  if (tid == 0) {
    J.dst = dst; J.src = src; J.At = At; J.pf = pf; J.sscale = sscale;
    J.ld = ld; J.lds = lds; J.n = n; J.base = base; J.cnt = cnt; J.nst = nst;
    J.vec16 = !(n & 1) && !(reinterpret_cast<size_t>(At) & 15);
  }
  __syncthreads();
  const int NGI = (((n + 15) >> 4) + SY_BI - 1) / SY_BI, ngp = (SY_BI / SY_BJ) * NGI * (NGI + 1) / 2;
  sy_gather(buf0, J, lidx, 0, 0, 0);
  int gi = 0, gj = 0;
  for (int gp = 0; gp < ngp; gp++) {
    const int warp = threadIdx.x >> 5;
    double acc[2][2][2];   // [a][e][h]: entry (16 ib + 8 a + fr, 16 jb + 8 e + 2 fk + h) of the warp's tile (ib, jb)
#pragma unroll
    for (int a = 0; a < 2; a++)
#pragma unroll
      for (int e = 0; e < 2; e++) { acc[a][e][0] = 0.0; acc[a][e][1] = 0.0; }
    const int nst_ = J.nst;
    for (int st = 0; st < nst_; st++) {
      const long long tw = clock64();
      bp_cp_async_wait_group<0>();
      __syncthreads();   // this stage is visible; every warp is done with the other buffer
      if (J.pf) { const long long t_ = clock64(); if (threadIdx.x == NT - 1) atomicAdd(reinterpret_cast<unsigned long long *>(J.pf + 15), (unsigned long long)(t_ - tw)); }
      const int g = gp * nst_ + st;
      if (st + 1 < nst_) sy_gather(buf0 + ((g + 1) & 1) * SY_C * SY_LD, J, lidx, st + 1, gi, gj);
      else if (gp + 1 < ngp) {
        const bool wrap = SY_BJ * (gj + 1) >= SY_BI * (gi + 1);
        sy_gather(buf0 + ((g + 1) & 1) * SY_C * SY_LD, J, lidx, 0, wrap ? gi + 1 : gi, wrap ? 0 : gj + 1);
      }
      const int lane = threadIdx.x & 31, fr = lane >> 2, fk = lane & 3;
      if (st + 1 == nst_ && lane < 16 && J.base != SY_ZERO) {   // the tile's base column segments (128 bytes each) into the L2 under the last stage
        const int i = 16 * (SY_BI * gi + (warp >> 1)), j = 16 * (SY_BJ * gj + (warp & 1)) + lane;
        if (i < J.n && j < J.n)
          asm volatile("prefetch.global.L2 [%0];" ::"l"(J.base == SY_DST ? J.dst + (size_t)i + (size_t)J.ld * j : J.src + (size_t)i + (size_t)J.lds * j));
      }
      const bool diag = SY_BJ * gj >= SY_BI * gi;
      const unsigned ub = (unsigned)__cvta_generic_to_shared(buf0 + (g & 1) * SY_C * SY_LD + fk * SY_LD);
      const unsigned aa = ub + 8u * (unsigned)(16 * (SY_BJ + (warp >> 1)) + fr);
      const unsigned ab = ub + 8u * (unsigned)(16 * (diag ? SY_BJ + SY_BJ * gj - SY_BI * gi + (warp & 1) : (warp & 1)) + fr);
      const unsigned wk = (unsigned)__cvta_generic_to_shared(S.vs + st * SY_C + fk);
#pragma unroll 3
      for (int kc = 0; kc < SY_C; kc += 4) {
        const unsigned o = (unsigned)(kc * SY_LD * 8);
        const double s_ = sy_lds(wk + 8u * kc);
        const double fa0 = sy_lds(aa + o) * s_, fa1 = sy_lds(aa + o + 64) * s_;
        const double fb0 = sy_lds(ab + o), fb1 = sy_lds(ab + o + 64);
        bp_dmma884(acc[0][0][0], acc[0][0][1], fa0, fb0);
        bp_dmma884(acc[0][1][0], acc[0][1][1], fa0, fb1);
        bp_dmma884(acc[1][0][0], acc[1][0][1], fa1, fb0);
        bp_dmma884(acc[1][1][0], acc[1][1][1], fa1, fb1);
      }
    }
    {   // H(tile) <- base + the stream's sum: each tile of dst is read once and written once
      const int lane = threadIdx.x & 31, fr = lane >> 2, fk = lane & 3, n_ = J.n, base_ = J.base;
      const int ib = SY_BI * gi + (warp >> 1), jb = SY_BJ * gj + (warp & 1);
#pragma unroll
      for (int a = 0; a < 2; a++)
#pragma unroll
        for (int e = 0; e < 2; e++)
#pragma unroll
          for (int h = 0; h < 2; h++) {
            const int i = 16 * ib + 8 * a + fr, j = 16 * jb + 8 * e + 2 * fk + h;
            if (i < n_ && j <= i) {
              double *d = J.dst + (size_t)i + (size_t)J.ld * j;
              const double v = (base_ == SY_DST) ? *d : ((base_ == SY_SRC) ? J.sscale * J.src[(size_t)i + (size_t)J.lds * j] : 0.0);
              *d = v + acc[a][e][h];
            }
          }
    }
    if (SY_BJ * (gj + 1) >= SY_BI * (gi + 1)) { gi++; gj = 0; } else gj++;
  }
  __syncthreads();   // the stages and weights are free for the caller
}

// ------------------------------------------------------------------------------------------------
// rank-k update / downdate of the instance's factor inside the CTA -- the cholmod_updown replacement of the batch engine
// (ldlupdate_entering_constraints / ldldowndate_leaving_constraints, src/solver_interface.c:407-441; recurrence of
// Modify/t_cholmod_updown_numkr.c:289-376 restated for L L').  <= KU ranks per sweep, entering rows (+) before leaving (-).
//
// Per column j with pivot d = l_jj^2 and, per rank r, the carried alpha_r and the current w_r[j]:
//     d_{r+1} = d_r + s_r w_r[j]^2 / alpha_r          gamma_r = -s_r w_r[j] / (alpha_r d_{r+1})        alpha_r <- alpha_r d_{r+1} / d_r
// and for the rows below:  t = l_ij / l_jj;  { w_r[i] -= w_r[j] t;  t -= gamma_r w_r[i] } over r;  l_ij = t sqrt(d_k).
// The chain over the ranks of one column only ever ADDS (s_r w^2 / alpha_r are known up front), so lane r of warp 0 owns
// rank r, the d_r come out of one warp prefix sum and each lane pays a single division: the serial cost per column does
// not grow with the rank.  The sweep walks 16-column panels staged in shared memory: warp 0 runs the recurrence on the
// 16 x 16 diagonal block (its rows of W in registers) and leaves the column coefficients in shared memory, then every thread
// transforms one row below the block.
// ------------------------------------------------------------------------------------------------
constexpr int KU = 8, UW = 16, WIN = 32, PBL = 33;   // ranks per sweep, columns per block, rows of the chain warp's window, block row pitch
constexpr int NRING = 3;                              // window-block buffers: in use by the chain / being requested / being written back
constexpr int LVW = 8;                                // row owners: columns of their row's entries in flight (shared-memory staging ring)
constexpr int NBAR = PW > UW ? PW : UW;               // per-column mbarriers: one per column of a Cholesky panel (the sweep and the solves use UW)
static_assert((KU * LDP + NRING * UW * PBL + LVW * LDP) * sizeof(double) <= kUnionBytes,
              "W block + the ring of window-block buffers + the row owners' staging ring must fit the union region");

struct UdCoef {   // in S.vs: the coefficients of one 16-column block, written column by column by the chain warp
  double winv[UW], d0[UW], dfin[2][UW];   // old pivots (1 / l_jj, l_jj^2) of the whole block, written at its start; dfin by block parity: the previous block's new pivots are still needed while it is written back
  __align__(16) double wj[UW][KU];
  __align__(16) double gam[UW][KU];
  __align__(16) double wpiv[KU];   // the pivot row's W as it stands before its column (published by that row's lane one column earlier)
  __align__(16) double cbuf[KU];   // per-rank pivot increments s_r w_r^2 / alpha_r of the current column
};
static_assert(sizeof(UdCoef) <= sizeof(double) * VS_LEN, "update coefficients must fit the staged-vector buffer");

__device__ __forceinline__ void ud_mbar_init(unsigned long long *bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count));
}
// arrive by lane 0 only, as a PREDICATED instruction (a branch would split the chain warp, see the note in the column loop)
__device__ __forceinline__ void ud_mbar_arrive_lane0(unsigned long long *bar, int lane) {
  asm volatile("{\n.reg .pred p;\nsetp.eq.s32 p, %1, 0;\n@p mbarrier.arrive.shared::cta.b64 _, [%0];\n}\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(lane) : "memory");
}
__device__ __forceinline__ void ud_mbar_wait(unsigned long long *bar, unsigned parity) {
  const unsigned a = (unsigned)__cvta_generic_to_shared(bar);
#ifdef QB_UD_TESTWAIT
  asm volatile("{\n.reg .pred p;\nWAIT_%=:\nmbarrier.test_wait.parity.shared::cta.b64 p, [%0], %1;\n@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}\n" ::"r"(a), "r"(parity) : "memory");
#else
  asm volatile("{\n.reg .pred p;\nWAIT_%=:\nmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}\n" ::"r"(a), "r"(parity) : "memory");
#endif
}

// chain warp: request the 32 x 16 window block at (k0, k0) -- lane = row k0 + lane, columns c <= lane -- into Pb[c * PBL + lane]
__device__ __forceinline__ void ud_block_prefetch(double *Pb, const double *L, int ld, int k0, int n, int lane) {
  const int row = k0 + lane;
#pragma unroll
  for (int c = 0; c < UW; c++) {
    if (row < n && k0 + c < n && c <= lane) bp_cp_async8(&Pb[c * PBL + lane], L + (size_t)row + (size_t)ld * (k0 + c));
    else Pb[c * PBL + lane] = 0.0;
  }
  bp_cp_async_commit();
}

// one sweep: L <- chol(L L' + sum_{r < kpos} w_r w_r' - sum_{kpos <= r < k} w_r w_r'),  w_r = wgt[r] * A'[:, list[r]]
//
// Round-2 shape (profiles/r02f_ncu_source_kbp_solve.txt: the old panel-staged sweep spent 18 % of the kernel with seven warps parked
// on the barrier behind warp 0's recurrence and another 12 % loading / storing panels):
//   * the CHAIN WARP (warp 0) walks the diagonal.  Its 32 lanes are the rows k0 .. k0 + 31 of the current 16-column block (the 16 block
//     rows and 16 look-ahead rows); their L entries sit in a small shared buffer that was requested one block ahead (cp.async), their
//     rows of W in registers.  Per column it forms the (alpha, gamma) coefficients, publishes them and arrives on that column's mbarrier.
//   * every other thread owns ONE row of L for the whole sweep (thread t <-> row t), keeps that row of W in registers and its 16
//     entries of the current block in registers (loaded straight from global memory before the block starts, written straight back):
//     it waits on the column's mbarrier, applies the column, and so trails the chain warp by one column.  The rows-below pass, the
//     panel staging and two of the four barriers per block are gone; what remains per block is the chain itself.
// The arithmetic per row is unchanged (t = l / l_jj; { w_r -= w_r[j] t; t -= gamma_r w_r }; l' = t sqrt(d_k)).
// bars: UW mbarriers (count 1) initialised once per kernel; every block completes exactly one phase of each; phase = blocks so far.
// block-end rendezvous of the two roles (named barrier 1; __syncthreads() is barrier 0 and is used by the code around the sweep)
__device__ __forceinline__ void ud_block_barrier() { asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory"); }

// write the finished window block (rows k0 .. k0 + 31, columns k0 .. k0 + 15; unit-scaled entries in Pn, new pivots squared in dfin)
// back to L: l' = t sqrt(d_k), l_jj' = sqrt(d_k), rdiag = 1 / l_jj'.  Called by `nthr` threads with t = 0 .. nthr - 1.
__device__ __forceinline__ void ud_flush_block(double *L, int ld, int n, double *rdiag_g, int k0, const double *Pn, const double *dfin, int t, int nthr) {
  const int w = (n - k0 < UW) ? n - k0 : UW;
  for (int e = t; e < WIN * UW; e += nthr) {
    const int l = e & (WIN - 1), c = e / WIN;
    if (c < w && k0 + l < n && l >= c) {
      double ln, lninv;
      chol32::sqrt_and_rcp(dfin[c], ln, lninv);   // branch-free (no slow-path call); every user of the new pivot forms it this way
      L[(size_t)(k0 + l) + (size_t)ld * (k0 + c)] = (l == c) ? ln : Pn[c * PBL + l] * ln;
      if (l == c) rdiag_g[k0 + c] = lninv;
    }
  }
}

// role 1 of the sweep: the chain warp (warp 0).  Nothing but the recurrence: its window blocks are requested and written back by
// the row owners (a first version did both here and spent 40 % of every block outside the column loop).
__device__ __forceinline__ void ud_chain_role(int n, int k, int kpos, double *Wm, double *Pb0, UdCoef &cf, int *info, unsigned long long *bars,
                                              long long *pf) {
  const int lane = threadIdx.x & 31;
  long long tq = clock64();
#define PC(k) do { if (pf) { const long long t_ = clock64(); if (lane == 31) atomicAdd(reinterpret_cast<unsigned long long *>(pf + (k)), (unsigned long long)(t_ - tq)); tq = t_; } } while (0)
  double ial = 1.0;                          // lane r < k: 1 / alpha_r
  const double sg = (lane < kpos) ? 1.0 : -1.0;
  bool bad = false;
  int slot = 0, blk = 0;
  for (int k0 = 0; k0 < n; k0 += UW, slot = (slot + 1 == NRING) ? 0 : slot + 1, blk++) {
    const int w = (n - k0 < UW) ? n - k0 : UW;
    double *Pn = Pb0 + slot * (UW * PBL);
    double *dfin_out = cf.dfin[blk & 1];
    const bool rowvalid = k0 + lane < n;
    double wl[KU];
#pragma unroll
    for (int r = 0; r < KU; r++) wl[r] = rowvalid ? Wm[r * LDP + k0 + lane] : 0.0;
    // off the chain: the old pivots are not touched before their own column, so 1 / l_jj and l_jj^2 of all 16 columns are
    // formed up front (lane = column); the new pivots sqrt(d) and the column scaling are left to the write-back
    const double ldiag = (lane < w) ? Pn[lane * PBL + lane] : 1.0;
    double winv_l;   // 1 / l_jj: reciprocal seed + two Newton steps (the IEEE division subroutine has a slow-path call as well)
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(winv_l) : "d"(ldiag));
    winv_l = fma(winv_l, fma(-ldiag, winv_l, 1.0), winv_l);
    winv_l = fma(winv_l, fma(-ldiag, winv_l, 1.0), winv_l);
    const double d0_l = ldiag * ldiag;
    __syncwarp();
    PC(23);
    // Column step.  One dependent chain: pivot row's W (shared memory, left there by that row's lane at the end of the previous
    // step) -> per-rank increments c_r -> their prefix sums d_r (ONE exchange through shared memory and a depth-3 add tree; the first
    // version scanned with three dependent shuffle rounds at ~54 clocks each) -> reciprocal -> gamma_r, alpha_r -> publish ->
    // row update of the window.  There is no shuffle in the loop (the old pivots of the block sit in shared memory), so a lane-dependent
    // branch around a store cannot push later steps onto the slow collective path.
    if (lane == 0) {
#pragma unroll
      for (int r = 0; r < KU; r++) cf.wpiv[r] = wl[r];
    }
    if (lane < UW) { cf.winv[lane] = winv_l; cf.d0[lane] = d0_l; }
    double sgial = sg * ial;
    __syncwarp();
    for (int j = 0; j < w; j++) {
      const double winv = cf.winv[j], d0 = cf.d0[j];
      const double wj = (lane < k) ? cf.wpiv[lane & (KU - 1)] : 0.0;
      const double c = wj * wj * sgial;            // = sg wj^2 ial, same rounding as ((sg wj) wj) ial
      if (lane < KU) cf.cbuf[lane] = c;
      __syncwarp();
      double incl;
      {
        const double2 *cb = reinterpret_cast<const double2 *>(cf.cbuf);
        const double2 c01 = cb[0], c23 = cb[1], c45 = cb[2], c67 = cb[3];
        const int rr = lane & (KU - 1);
        const double m0 = c01.x, m1 = (rr >= 1) ? c01.y : 0.0, m2 = (rr >= 2) ? c23.x : 0.0, m3 = (rr >= 3) ? c23.y : 0.0;
        const double m4 = (rr >= 4) ? c45.x : 0.0, m5 = (rr >= 5) ? c45.y : 0.0, m6 = (rr >= 6) ? c67.x : 0.0, m7 = (rr >= 7) ? c67.y : 0.0;
        incl = ((m0 + m1) + (m2 + m3)) + ((m4 + m5) + (m6 + m7));
      }
      const double dnext = d0 + incl, dprev = d0 + (incl - c);
      if (lane < k && !(dnext > 0.0)) bad = true;
      double q;   // ial / dnext: reciprocal seed + two Newton steps instead of the IEEE division subroutine
      asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(q) : "d"(dnext));
      q = fma(q, fma(-dnext, q, 1.0), q);
      q = fma(q, fma(-dnext, q, 1.0), q);
      q *= ial;
      const double gam = -sg * wj * q;
      ial = dprev * q;
      sgial = sg * ial;
      // publish column j: lanes < KU the rank coefficients, lane k - 1 (which holds d_k) the new pivot squared
      if (lane < KU) { cf.wj[j][lane] = (lane < k) ? wj : 0.0; cf.gam[j][lane] = (lane < k) ? gam : 0.0; }
      if (lane == k - 1) dfin_out[j] = dnext;
      __syncwarp();
      ud_mbar_arrive_lane0(bars + j, lane);   // column j is published: the row owners may apply it
      {
        double t = (rowvalid ? Pn[j * PBL + lane] : 0.0) * winv;
        const double2 *wj2 = reinterpret_cast<const double2 *>(cf.wj[j]), *gm2 = reinterpret_cast<const double2 *>(cf.gam[j]);
#pragma unroll
        for (int r2 = 0; r2 < KU / 2; r2++) {
          const double2 a = wj2[r2], g = gm2[r2];
          wl[2 * r2] = fma(-a.x, t, wl[2 * r2]);
          t = fma(-g.x, wl[2 * r2], t);
          wl[2 * r2 + 1] = fma(-a.y, t, wl[2 * r2 + 1]);
          t = fma(-g.y, wl[2 * r2 + 1], t);
        }
        if (lane > j && rowvalid) Pn[j * PBL + lane] = t;   // unit-scaled; the write-back multiplies by the new pivot
        if (lane == j + 1) {   // the next pivot row: leave its W for the next step
#pragma unroll
          for (int r = 0; r < KU; r++) cf.wpiv[r] = wl[r];
        }
      }
      __syncwarp();
    }
    PC(25);
    for (int j = w; j < UW; j++) ud_mbar_arrive_lane0(bars + j, lane);   // ragged last block: every barrier completes one phase per block
    if (lane >= UW && rowvalid) {   // the look-ahead rows are block rows of the next window: hand their W over
#pragma unroll
      for (int r = 0; r < KU; r++) Wm[r * LDP + k0 + lane] = wl[r];
    }
    __syncwarp();
    PC(26);
    ud_block_barrier();
    PC(27);
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) *info = 1;
#undef PC
}

// role 2 of the sweep: a row owner (threads >= WIN; thread t <-> row t).  Besides its own row it helps the chain warp: the previous
// window block is written back by all row owners, the next one is requested by warp 1.
__device__ __forceinline__ void ud_row_role(double *L, int ld, int n, double *rdiag_g, double *Wm, double *Pb0, double *Ls, const UdCoef &cf,
                                            unsigned long long *bars, unsigned phase) {
  const int row = threadIdx.x, lane = threadIdx.x & 31;
  const bool requester = (threadIdx.x >> 5) == 1;
  double wv[KU];
#pragma unroll
  for (int r = 0; r < KU; r++) wv[r] = (row < n) ? Wm[r * LDP + row] : 0.0;
  int slot = 0, blk = 0;
  // This row's entries of the block travel through a private staging ring in shared memory: Ls[c % LVW][row] is written by this
  // thread's own cp.async and read by this thread only, so no barrier is involved and no registers are held (16 entries in
  // registers spill at 64 registers per thread, and a spilled entry costs an L2 round trip per column).  Entry c + LVW (of this or
  // the next block) is requested as soon as entry c has been consumed, i.e. LVW columns ahead of its use.
  if (row >= WIN && row < n) {
#pragma unroll
    for (int c = 0; c < LVW; c++) {
      if (c < n) bp_cp_async8(&Ls[c * LDP + row], L + (size_t)row + (size_t)ld * c);
      bp_cp_async_commit();
    }
  }
  for (int k0 = 0; k0 < n; k0 += UW, slot = (slot + 1 == NRING) ? 0 : slot + 1, blk++) {
    const int w = (n - k0 < UW) ? n - k0 : UW;
    const unsigned par = phase & 1u;
    phase++;
    const int slot_next = (slot + 1 == NRING) ? 0 : slot + 1, slot_prev = (slot == 0) ? NRING - 1 : slot - 1;
    const bool below = row >= k0 + WIN && row < n, below_next = row >= k0 + UW + WIN && row < n;
    double *Lr = L + (size_t)row + (size_t)ld * k0;
    const double *dfin = cf.dfin[blk & 1];
    if (requester && k0 + UW < n) ud_block_prefetch(Pb0 + slot_next * (UW * PBL), L, ld, k0 + UW, n, lane);
    if (k0 > 0) ud_flush_block(L, ld, n, rdiag_g, k0 - UW, Pb0 + slot_prev * (UW * PBL), cf.dfin[(blk - 1) & 1], threadIdx.x - WIN, NT - WIN);
    if (below) {   // below the window: apply the block column by column as it is published
#pragma unroll
      for (int c = 0; c < UW; c++) {
        if (c < w) {
          bp_cp_async_wait_group<LVW - 1>();   // this thread's request for column c has landed (later groups may still be in flight)
          ud_mbar_wait(bars + c, par);
          double t = Ls[(c % LVW) * LDP + row] * cf.winv[c];
          const double2 *wj2 = reinterpret_cast<const double2 *>(cf.wj[c]), *gm2 = reinterpret_cast<const double2 *>(cf.gam[c]);
#pragma unroll
          for (int r2 = 0; r2 < KU / 2; r2++) {
            const double2 a = wj2[r2], g = gm2[r2];
            wv[2 * r2] = fma(-a.x, t, wv[2 * r2]);
            t = fma(-g.x, wv[2 * r2], t);
            wv[2 * r2 + 1] = fma(-a.y, t, wv[2 * r2 + 1]);
            t = fma(-g.y, wv[2 * r2 + 1], t);
          }
          double ln, lninv;
          chol32::sqrt_and_rcp(dfin[c], ln, lninv);
          Lr[(size_t)ld * c] = t * ln;
        }
        // refill the slot just consumed: column c + LVW of this block, or of the next block when this row stays below the window
        const int cn = c + LVW;
        if ((cn < UW || below_next) && k0 + cn < n) bp_cp_async8(&Ls[(c % LVW) * LDP + row], Lr + (size_t)ld * cn);
        bp_cp_async_commit();
      }
      if (row < k0 + WIN + UW) {   // this row enters the chain warp's window with the next block: hand its W over
#pragma unroll
        for (int r = 0; r < KU; r++) Wm[r * LDP + row] = wv[r];
      }
    }
    if (requester) bp_cp_async_wait_group<0>();
    ud_block_barrier();
  }
}

__device__ __noinline__ void cta_updown_sweep(double *L, int ld, int n, double *rdiag_g, const double *__restrict__ At,
                                              const int *__restrict__ list, const double *__restrict__ wgt, int k, int kpos, const Smem &S, int *info,
                                              unsigned long long *bars, unsigned &phase, long long *pf) {
  const int tid = threadIdx.x;
  double *Wm = S.panel, *Pb0 = S.panel + KU * LDP;
  UdCoef &cf = *reinterpret_cast<UdCoef *>(S.vs);
  long long tq = clock64();
#define PQ(k) do { if (pf) { const long long t_ = clock64(); if (tid == NT - 1) atomicAdd(reinterpret_cast<unsigned long long *>(pf + (k)), (unsigned long long)(t_ - tq)); tq = t_; } } while (0)
  for (int idx = tid; idx < KU * n; idx += NT) {   // gather the rows (zero columns beyond k)
    const int r = idx / n, i = idx - r * n;
    Wm[r * LDP + i] = (r < k) ? wgt[r] * At[(size_t)i + (size_t)n * list[r]] : 0.0;
  }
  if (tid < 32) { ud_block_prefetch(Pb0, L, ld, 0, n, tid); bp_cp_async_wait_group<0>(); }
  __syncthreads();
  PQ(22);
  if (tid < 32) ud_chain_role(n, k, kpos, Wm, Pb0, cf, info, bars, pf);
  else ud_row_role(L, ld, n, rdiag_g, Wm, Pb0, Pb0 + NRING * UW * PBL, cf, bars, phase);
  const int nblk = (n + UW - 1) / UW;
  phase += (unsigned)nblk;
  ud_flush_block(L, ld, n, rdiag_g, (nblk - 1) * UW, Pb0 + ((nblk - 1) % NRING) * (UW * PBL), cf.dfin[(nblk - 1) & 1], tid, NT);   // last window block
  __syncthreads();
  PQ(24);
#undef PQ
}

// ------------------------------------------------------------------------------------------------
// v <- (L L')^{-1} v: the two triangular solves of the Newton step, as the dataflow of the update sweep.  v is S.v, L the
// instance's factor in global memory (n x n lower), rdiag_g = 1 / diag(L).  Both directions walk 16-column blocks:
//   * the CHAIN WARP (warp 0) holds the 32-entry window of v at the block (the 16 block entries and 16 look-ahead entries) in
//     registers and the window's entries of L in a shared buffer requested one block ahead (cp.async, warp 1); per column it
//     forms the next solution entry, publishes it in S.v, arrives on that column's mbarrier and applies it to its window;
//   * every other thread owns one entry of v outside the window -- forward: row t (thread t), backward: column t - 32 --, keeps it
//     in a register, streams its entries of the block's L through a private cp.async ring (LVW ahead of use, as the sweep's row
//     owners) and applies each column as soon as its mbarrier completes;
//   * at a block's end the entries that enter the next window are handed to the chain through S.v (named barrier 1).
// The panel-staged form it replaces paid, per 24 / 32-column panel, a full load of the panel, a wait and three barriers with
// seven warps parked behind one warp's chain (13 us per panel at 512 instances, profiles/r03a_batch_phase_clocks_parent_solve_split.txt).
// Rounding: every entry is updated by one fma per column in column order (forward: ascending j, z_j = v_j / l_jj as v_j * rdiag;
// backward: descending i, d_j likewise), whoever holds it, so the result does not depend on the CTA shape.  This is the only
// forward substitution of the engine: the factorisation no longer runs one while its panels are resident.
// ------------------------------------------------------------------------------------------------
constexpr int SV_SLOT = UW * PBL + UW;   // one window block: 16 x 32 entries of L at [c * PBL + lane] and the block's 16 1 / l_jj
constexpr int SV_NWIN = 3;               // window blocks: in use by the chain / requested one and two blocks ahead
constexpr int SV_G = 4;                  // owners: columns applied per mbarrier wait
static_assert((SV_NWIN * SV_SLOT * sizeof(double)) % 16 == 0 && (SV_NWIN * SV_SLOT + UW * NT) * sizeof(double) <= kUnionBytes,
              "the window blocks + the owners' staging ring of the triangular solves must fit the union region");

// The owners poll with test_wait.  A thread suspended in try_wait (ud_mbar_wait) resumed too late for a chain step of ~180 clocks:
// at 512 instances the chain then spent 2.6 us per block end waiting for the owners' last columns (4.9 of the solve's 8.4 ms per
// instance); polling took the launch from 78.4 to 76.1 ms.  The sweep keeps try_wait: its owners have eight ranks of work per column.
__device__ __forceinline__ void sv_mbar_wait_spin(unsigned long long *bar, unsigned parity) {
  const unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile("{\n.reg .pred p;\nWAIT_%=:\nmbarrier.test_wait.parity.shared::cta.b64 p, [%0], %1;\n@!p bra WAIT_%=;\n}\n" ::"r"(a), "r"(parity) : "memory");
}

// 16-byte cp.async that bypasses L1 (.cg has no 8-byte form)
__device__ __forceinline__ void bp_cp_async16_cg(void *smem_dst, const double *gsrc) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}

// request window block k0: forward rows k0 + lane, columns k0 + c (c <= lane); backward rows k0 + c, columns k0 - 16 + lane
// (lower triangle only, zeros elsewhere); 1 / l_jj of columns k0 .. k0 + 15 behind them.  Called by the chain warp.
template <bool fwd>
__device__ __forceinline__ void sv_block_prefetch(double *Pb, const double *L, int ld, const double *rdiag_g, int k0, int n, int lane) {
#pragma unroll
  for (int c = 0; c < UW; c++) {
    const int row = fwd ? k0 + lane : k0 + c, col = fwd ? k0 + c : k0 - UW + lane;
    if (row < n && col >= 0 && col <= row) bp_cp_async8(&Pb[c * PBL + lane], L + (size_t)row + (size_t)ld * col);
    else Pb[c * PBL + lane] = 0.0;
  }
  if (lane < UW && k0 + lane < n) bp_cp_async8(&Pb[UW * PBL + lane], rdiag_g + k0 + lane);
  bp_cp_async_commit();
}

// chain warp.  fwd: lane = row k0 + lane; block columns ascending.  bwd: lane = column k0 - 16 + lane; block rows descending.
// It requests its own window blocks, two ahead, so a block's L is in flight for two blocks' worth of chain.
// Slots pf[0] / pf[1]: the column loops / the block-end rendezvous and window waits (clock of lane 31).
template <bool fwd>
__device__ __forceinline__ void sv_chain_role(const double *L, int ld, int n, const double *rdiag_g, double *v, double *Pb0, unsigned long long *bars,
                                              long long *pf) {
  const int lane = threadIdx.x & 31;
  long long tq = clock64();
#define PC(k) do { if (pf) { const long long t_ = clock64(); if (lane == 31) atomicAdd(reinterpret_cast<unsigned long long *>(pf + (k)), (unsigned long long)(t_ - tq)); tq = t_; } } while (0)
  const int nblk = (n + UW - 1) / UW;
  auto blk_k0 = [&](int blk) { return fwd ? blk * UW : (nblk - 1 - blk) * UW; };
#pragma unroll 1
  for (int blk = 0; blk < 2; blk++) {
    if (blk < nblk) sv_block_prefetch<fwd>(Pb0 + blk * SV_SLOT, L, ld, rdiag_g, blk_k0(blk), n, lane);
    else bp_cp_async_commit();
  }
  for (int blk = 0; blk < nblk; blk++) {
    const int k0 = blk_k0(blk), w = (n - k0 < UW) ? n - k0 : UW;
    if (blk + 2 < nblk) sv_block_prefetch<fwd>(Pb0 + ((blk + 2) % SV_NWIN) * SV_SLOT, L, ld, rdiag_g, blk_k0(blk + 2), n, lane);
    else bp_cp_async_commit();   // an empty group: "all but the two newest groups" stays "this block's window"
    bp_cp_async_wait_group<2>();
    __syncwarp();
    PC(1);
    const double *Pb = Pb0 + (blk % SV_NWIN) * SV_SLOT, *rd = Pb + UW * PBL;
    const int e = fwd ? k0 + lane : k0 - UW + lane;   // this lane's entry of v
    const bool valid = e >= 0 && e < n;
    double x = valid ? v[e] : 0.0;
    for (int jj = 0; jj < w; jj++) {
      const int j = fwd ? jj : w - 1 - jj, src = fwd ? j : UW + j;   // column (fwd) / row (bwd) k0 + j, held by lane src
      const double a = Pb[j * PBL + lane], r = rd[j];
      const double z = __shfl_sync(0xffffffffu, x, src) * r;
      if (lane == 0) v[k0 + j] = z;
      ud_mbar_arrive_lane0(bars + j, lane);   // entry k0 + j is final: the owners may apply it
      const bool after = fwd ? lane > src : lane < src;
      x = (lane == src) ? z : (after ? fma(-a, z, x) : x);
    }
    PC(0);
    for (int j = w; j < UW; j++) ud_mbar_arrive_lane0(bars + j, lane);   // ragged block: every barrier completes one phase per block
    if ((fwd ? lane >= UW : lane < UW) && valid) v[e] = x;              // the look-ahead entries: the next block's window
    ud_block_barrier();
  }
  PC(1);
#undef PC
}

// an owner (threads >= 32).  fwd: row t = thread t, below the window (t >= k0 + 32); bwd: column t - 32, left of the window
// (t - 32 < k0 - 16).  Its entries of L arrive through a private ring in shared memory, a whole block (16 entries) ahead of use:
// fwd 16 slots of 8 bytes, L(e, col), one per column (neighbouring threads read neighbouring rows: whole sectors per warp);
// bwd 8 slots of 16 bytes, L(r, e) L(r + 1, e) with r even, one per two rows (a column segment, read in whole 16-byte pieces
// past L1: the 8-byte form would allocate an L1 line per thread that the co-resident CTAs need for their own working sets).
template <bool fwd>
__device__ __forceinline__ void sv_owner_role(const double *L, int ld, int n, double *v, double2 *R, unsigned long long *bars, unsigned phase) {
  const int t = threadIdx.x, e = fwd ? t : t - WIN;
  const int nblk = (n + UW - 1) / UW, last = (nblk - 1) * UW;
  double *R8 = reinterpret_cast<double *>(R);
  double x = (e < n) ? v[e] : 0.0;
  if (fwd ? (e >= WIN && e < n) : (e < last - UW)) {
#pragma unroll
    for (int q = 0; q < (fwd ? UW : UW / 2); q++) {   // fwd: columns 0 .. 15; bwd: rows last + 14 - 2 q, + 1
      if (fwd) { if (q < n) bp_cp_async8(&R8[q * NT + t], L + (size_t)e + (size_t)ld * q); }
      else if (last + UW - 2 - 2 * q < n) bp_cp_async16_cg(&R[q * NT + t], L + (size_t)ld * e + (last + UW - 2 - 2 * q));
      bp_cp_async_commit();
    }
  }
  for (int blk = 0; blk < nblk; blk++) {
    const int k0 = fwd ? blk * UW : last - blk * UW, w = (n - k0 < UW) ? n - k0 : UW;
    const unsigned par = (phase + blk) & 1u;
    const bool own = fwd ? (e >= k0 + WIN && e < n) : (e < k0 - UW);
    const bool own_next = fwd ? (e >= k0 + UW + WIN && e < n) : (e < k0 - 2 * UW);
    if (own) {
#pragma unroll 1
      for (int p = 0; p < UW; p++) {   // rolled: sixteen copies of the wait loops cost instruction-cache misses in every other phase
        const int j = fwd ? p : UW - 1 - p;
        if (j < w) {
          if (fwd) bp_cp_async_wait_group<UW - 1>();   // this slot has landed (the later ones may be in flight)
          else bp_cp_async_wait_group<UW / 2 - 1>();
          // one wait per group of SV_G columns, on the group's last column in chain order (the chain publishes in order): a woken
          // owner then applies SV_G columns, where one wait per column cost more than the chain's step and left the owners a
          // block's worth of wake-ups behind it at every block end
          if (fwd ? (j % SV_G == 0) : (j % SV_G == SV_G - 1 || j == w - 1))
            sv_mbar_wait_spin(bars + (fwd ? min(j | (SV_G - 1), w - 1) : (j & ~(SV_G - 1))), par);
          double l;
          if (fwd) l = R8[p * NT + t];
          else { const double2 l2 = R[(p >> 1) * NT + t]; l = (p & 1) ? l2.x : l2.y; }
          x = fma(-l, v[k0 + j], x);
        }
        // the slot is used up: refill it with the same slot of the next block
        if (fwd) {
          if (own_next && k0 + UW + p < n) bp_cp_async8(&R8[p * NT + t], L + (size_t)e + (size_t)ld * (k0 + UW + p));
          bp_cp_async_commit();
        } else if (p & 1) {
          if (own_next) bp_cp_async16_cg(&R[(p >> 1) * NT + t], L + (size_t)ld * e + (k0 - 1 - p));
          bp_cp_async_commit();
        }
      }
      if (!own_next) v[e] = x;   // this entry enters the chain warp's window with the next block
    }
    ud_block_barrier();
  }
}

// one direction (nblk blocks, mbarrier phases phase .. phase + nblk - 1)
template <bool fwd>
__device__ __forceinline__ void sv_direction(const double *L, int ld, int n, const double *rdiag_g, const Smem &S, unsigned long long *bars,
                                             unsigned phase, long long *pf) {
  double *Pb0 = S.panel;
  double2 *R = reinterpret_cast<double2 *>(S.panel + SV_NWIN * SV_SLOT);
  if (threadIdx.x < 32) sv_chain_role<fwd>(L, ld, n, rdiag_g, S.v, Pb0, bars, pf);
  else sv_owner_role<fwd>(L, ld, n, S.v, R, bars, phase);
  __syncthreads();
}
// bars / phase: the update sweep's per-column mbarriers and their phase count (each direction completes one phase of each barrier
// per block).  pf: the instance's phase-clock row (slots 28 .. 31), or null.
__device__ __noinline__ void cta_chol_solve(const double *L, int ld, int n, const double *rdiag_g, const Smem &S, unsigned long long *bars,
                                            unsigned &phase, long long *pf) {
  const unsigned nblk = (unsigned)((n + UW - 1) / UW), ph = phase;   // phase lives in the caller's frame: read and written once
  sv_direction<true>(L, ld, n, rdiag_g, S, bars, ph, pf ? pf + 28 : nullptr);           // L z = v
  sv_direction<false>(L, ld, n, rdiag_g, S, bars, ph + nblk, pf ? pf + 30 : nullptr);   // L' d = z
  phase = ph + 2 * nblk;
}

// ------------------------------------------------------------------------------------------------
// L <- chol(sscale * src + beta I) (lower, n x n), right-looking with PW-column panels.  rdiag_g[j] = 1 / l_jj.
// A panel (its rows k0 .. n - 1 in S.panel, P[t][r], t = column, r = row - k0) is factorised as the dataflow of the update
// sweep and the triangular solves:
//   * the CHAIN WARP (warp 0) holds rows k0 .. k0 + 31 (lane = row): the w <= 32 diagonal rows and, in the 24-column shape,
//     the first 8 rows below them.  Per column j: the pivot from lane j (one shuffle), l_jj and 1 / l_jj, the column scaled,
//     published in the panel with rd[j], an arrive on column j's mbarrier, then column j applied to the window;
//   * every other thread owns one panel row (thread t <-> row k0 + t; n <= NMAX <= NT): it waits on column j's mbarrier, scales
//     its entry by rd[j] and applies column j to the rest of its row.
// The rows stay in the panel (the odd LDP keeps a warp's accesses to one column conflict-free; 24 or 32 doubles per thread
// in registers spill at 64 / 80 registers).  Each thread then stores its own row of L, so one barrier per panel remains
// before the trailing DMMA update.  The form it replaces factored 16- or 8-column diagonal blocks in warp 0 with the seven
// other warps parked at a barrier, then the rows below, then the columns to the right: about ten barriers per panel.
// Rounding: every entry takes one fma per column in ascending column order, l_ij = a_ij * (1 / l_jj), whoever holds it.
// bars: NBAR mbarriers (count 1); every panel completes one phase of each.  Barriers 0 .. UW - 1 are those of the sweep and
// the solves (phase count `phase`), barriers UW .. NBAR - 1 serve only the factorisation (`phase_hi`).
// ------------------------------------------------------------------------------------------------
// apply column j (its entries l_cj in P[j][c], this row's l_rj = l) to columns j0 <= c < w of row r, r >= c only (rlim = r,
// or -1 for a row outside the panel).  Four columns' loads are issued before their fmas and stores.
__device__ __forceinline__ void potrf_row_apply(double *Pn, int r, int rlim, int j, int j0, int w, double l) {
  int c = j0;
#pragma unroll 1
  for (; c + 4 <= w; c += 4) {
    double lc[4], a[4];
#pragma unroll
    for (int u = 0; u < 4; u++) { lc[u] = Pn[j * LDP + c + u]; a[u] = Pn[(c + u) * LDP + r]; }
#pragma unroll
    for (int u = 0; u < 4; u++) if (rlim >= c + u) Pn[(c + u) * LDP + r] = fma(-l, lc[u], a[u]);
  }
#pragma unroll 1
  for (; c < w; c++) if (rlim >= c) Pn[c * LDP + r] = fma(-l, Pn[j * LDP + c], Pn[c * LDP + r]);
}

// One panel after its load: factor, store its rows of L and 1 / l_jj, zero the pad columns [w, w + 3 & ~3) of every row for the
// DMMA product loop.  par_lo / par_hi: the parity of this panel's phase of barriers < UW / >= UW.  The caller's
// __syncthreads() ends the panel.  Phase clocks: 17 chain column loop, 18 chain store + wait (lane 31); 19 owners' column loop,
// 20 owners' store + wait (thread 32, the first owner).
__device__ __noinline__ void potrf_panel(double *Pn, double *rd, double *L, int ld, double *rdiag_g, int k0, int w, int rows,
                                         unsigned long long *bars, unsigned par_lo, unsigned par_hi, int *info, long long *pf) {
  const int tid = threadIdx.x;
  long long tq = clock64();
#define PQ(k, rec) do { if (pf) { const long long t_ = clock64(); if (rec) atomicAdd(reinterpret_cast<unsigned long long *>(pf + (k)), (unsigned long long)(t_ - tq)); tq = t_; } } while (0)
  if (tid < WIN) {   // chain warp: no lane-dependent branch around the shuffles, __syncwarp and arrives (predicated stores only)
    const int lane = tid;
    const bool live = lane < rows;
    const int rlim = live ? lane : -1;
    double cur = live ? Pn[lane] : 0.0;   // this row's entry of the current column, final
    double pv = __shfl_sync(0xffffffffu, cur, 0);
    bool bad = false;
#pragma unroll 1
    for (int j = 0; j < w; j++) {
      double ljj, inv;
      chol32::sqrt_and_rcp(pv, ljj, inv);
      if (!(pv > 0.0)) bad = true;   // pv is the same in every lane
      const double l = (lane == j) ? ljj : cur * inv;
      // the next pivot first: lane j + 1 needs only its own l_{j+1,j}, so the chain per column is one shuffle, sqrt / rcp, one
      // multiply and one fma (the published column and the rest of the window follow)
      const int j1 = (j + 1 < w) ? j + 1 : j;
      const double a1 = Pn[j1 * LDP + lane];
      pv = __shfl_sync(0xffffffffu, fma(-l, l, a1), (j + 1) & 31);
      if (rlim >= j) Pn[j * LDP + lane] = l;
      if (lane == j) rd[j] = inv;
      __syncwarp();
      ud_mbar_arrive_lane0(bars + j, lane);   // column j is published: the row owners may apply it
      cur = fma(-l, Pn[j * LDP + j1], a1);    // column j + 1 of this row (lane j + 1: the pivot just shuffled)
      potrf_row_apply(Pn, lane, rlim, j, j + 2, w, l);
    }
    for (int j = w; j < NBAR; j++) ud_mbar_arrive_lane0(bars + j, lane);   // ragged last panel: every barrier completes one phase
    if (bad && lane == 0) *info = 1;
    PQ(17, lane == 31);
    if (live) {
      for (int c = 0; c < w; c++) if (c <= lane) L[(size_t)(k0 + lane) + (size_t)ld * (k0 + c)] = Pn[c * LDP + lane];
      for (int c = w; c < ((w + 3) & ~3); c++) Pn[c * LDP + lane] = 0.0;
    }
    if (lane < w) rdiag_g[k0 + lane] = rd[lane];   // rd[lane] was written by this lane
  } else if (tid < rows) {   // row owner (row tid >= 32 > w: every column of the panel applies)
    const int r = tid;
#pragma unroll 1
    for (int j = 0; j < w; j++) {
      ud_mbar_wait(bars + j, j < UW ? par_lo : par_hi);
      const double l = Pn[j * LDP + r] * rd[j];
      Pn[j * LDP + r] = l;
      potrf_row_apply(Pn, r, r, j, j + 1, w, l);
    }
    PQ(19, tid == WIN);
    for (int c = 0; c < w; c++) L[(size_t)(k0 + r) + (size_t)ld * (k0 + c)] = Pn[c * LDP + r];
    for (int c = w; c < ((w + 3) & ~3); c++) Pn[c * LDP + r] = 0.0;
  }
  __syncthreads();
  PQ(tid == 31 ? 18 : 20, tid == 31 || tid == WIN);
#undef PQ
}

__device__ __forceinline__ void cta_potrf(double *L, int ld, const double *src, int lds, double sscale, double beta, int n, double *rdiag_g,
                          const Smem &S, int *info, unsigned long long *bars, unsigned &phase, unsigned &phase_hi, long long *pf) {
  const int tid = threadIdx.x;
  double *Pn = S.panel;
  const unsigned ph = phase, phh = phase_hi;   // read and written once (they live in the caller's frame)
  long long tq = clock64();
// Phase clocks: one predicated atomic, NO divergent region.  (An `if (tid == 0) { load; add; store }` body leaves lane 0 split
// from the rest of warp 0 under independent thread scheduling; every __shfl_sync of the following single-warp phases then
// takes the WARPSYNC.COLLECTIVE slow path -- measured 131k instead of 13.6k clocks per 16 x 16 diagonal block, which made
// the profile of round 1 blame the wrong phase.)
#define PQ(k) do { if (pf) { const long long t_ = clock64(); if (tid == NT - 1) atomicAdd(reinterpret_cast<unsigned long long *>(pf + (k)), (unsigned long long)(t_ - tq)); tq = t_; } } while (0)
  unsigned p = 0;
  for (int k0 = 0; k0 < n; k0 += PW, p++) {
    const int w = (n - k0 < PW) ? n - k0 : PW, rows = n - k0;
    const bool first = (k0 == 0);
    if (first) {
      for (int idx = tid; idx < w * rows; idx += NT) {   // panel load, rows fastest (coalesced)
        const int t = idx / rows, r = idx - t * rows;
        double v = 0.0;
        if (r >= t) { v = sscale * src[(size_t)r + (size_t)lds * t]; if (r == t) v += beta; }
        Pn[t * LDP + r] = v;
      }
    } else panel_load_async(Pn, L, ld, k0, w, rows);
    __syncthreads();
    PQ(16);
    potrf_panel(Pn, S.rd, L, ld, rdiag_g, k0, w, rows, bars, (ph + p) & 1u, (phh + p) & 1u, info, pf);
    if (pf) tq = clock64();
    cta_rank_update_lower(L, ld, src, lds, sscale, beta, first, k0 + w, n, Pn, k0, w, -1.0);
    __syncthreads();
    PQ(21);
  }
  phase = ph + p;
  phase_hi = phh + p;
#undef PQ
}

// ordered lists of the entering (candidate active, not in the factor) and leaving rows, entering first, weights sqrt(sigma):
// list_pos[0 .. ne + nl), w_pos likewise (set_entering_leaving_constraints, newton.c:134-149).  Returns counts through ctl.npos / nneg.
__device__ __noinline__ void p_updown_lists(const Args &P, int b) {
  __shared__ int warp_cnt0[NW], warp_cnt1[NW];
  __shared__ int base0, base1;
  const int m = P.m, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t om = (size_t)b * m;
  if (tid == 0) { base0 = 0; base1 = 0; }
  __syncthreads();
  for (int start = 0; start < m; start += NT) {
    const int i = start + tid;
    bool p0 = false, p1 = false;
    if (i < m) {
      const int a = P.active_cand[om + i], o = P.active_old[om + i];
      p0 = a && !o; p1 = !a && o;
    }
    const unsigned b0 = __ballot_sync(0xffffffffu, p0), b1 = __ballot_sync(0xffffffffu, p1);
    if (lane == 0) { warp_cnt0[warp] = __popc(b0); warp_cnt1[warp] = __popc(b1); }
    __syncthreads();
    int off0 = base0, off1 = base1;
    for (int w = 0; w < warp; w++) { off0 += warp_cnt0[w]; off1 += warp_cnt1[w]; }
    const unsigned lt = (1u << lane) - 1u;
    if (p0) P.list_pos[om + off0 + __popc(b0 & lt)] = i;
    if (p1) P.list_neg[om + off1 + __popc(b1 & lt)] = i;
    __syncthreads();
    if (tid == 0) { int t0 = 0, t1 = 0; for (int w = 0; w < NW; w++) { t0 += warp_cnt0[w]; t1 += warp_cnt1[w]; } base0 += t0; base1 += t1; }
    __syncthreads();
  }
  const int ne = base0, nl = base1;
  __syncthreads();
  for (int q = tid; q < nl; q += NT) P.list_pos[om + ne + q] = P.list_neg[om + q];   // append the leaving rows
  __syncthreads();
  for (int q = tid; q < ne + nl; q += NT) P.w_pos[om + q] = P.sqrt_sigma[om + P.list_pos[om + q]];
  if (tid == 0) { BCtl &c = P.ctl[b]; c.npos = ne; c.nneg = nl; }
}

// ------------------------------------------------------------------------------------------------
// active-set commit + ordered H-difference lists (batch.cu kb_lists, one CTA)
// ------------------------------------------------------------------------------------------------
__device__ __noinline__ void p_lists(const Args &P, int b, int refac) {
  __shared__ int warp_cnt0[NW], warp_cnt1[NW];
  __shared__ int base0, base1, redo;
  const int m = P.m, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t om = (size_t)b * m;
  for (int i = tid; i < m; i += NT) P.active[om + i] = P.active_cand[om + i];
  if (!refac) return;
  int scratch_mode = P.ctl[b].scratch;
  const int nb_active = P.ctl[b].nb_active;
  for (int attempt = 0; attempt < 2; attempt++) {
    __syncthreads();
    if (tid == 0) { base0 = 0; base1 = 0; redo = 0; }
    __syncthreads();
    for (int start = 0; start < m; start += NT) {
      const int i = start + tid;
      bool p0 = false, p1 = false;
      double s0 = 0.0, s1 = 0.0;
      if (i < m) {
        const int a = P.active[om + i];
        const double wn = a ? P.sigma[om + i] : 0.0;
        const double wh = (scratch_mode || !P.activeH[om + i]) ? 0.0 : P.sigmaH[om + i];
        const double dw = wn - wh;
        if (dw > 0.0) { p0 = true; s0 = (wh == 0.0) ? P.sqrt_sigma[om + i] : sqrt(dw); }
        else if (dw < 0.0) { p1 = true; s1 = sqrt(-dw); }
      }
      const unsigned b0 = __ballot_sync(0xffffffffu, p0), b1 = __ballot_sync(0xffffffffu, p1);
      if (lane == 0) { warp_cnt0[warp] = __popc(b0); warp_cnt1[warp] = __popc(b1); }
      __syncthreads();
      int off0 = base0, off1 = base1;
      for (int w = 0; w < warp; w++) { off0 += warp_cnt0[w]; off1 += warp_cnt1[w]; }
      const unsigned lt = (1u << lane) - 1u;
      if (p0) { const int pos = off0 + __popc(b0 & lt); P.list_pos[om + pos] = i; P.w_pos[om + pos] = s0; }
      if (p1) { const int pos = off1 + __popc(b1 & lt); P.list_neg[om + pos] = i; P.w_neg[om + pos] = s1; }
      __syncthreads();
      if (tid == 0) { int t0 = 0, t1 = 0; for (int w = 0; w < NW; w++) { t0 += warp_cnt0[w]; t1 += warp_cnt1[w]; } base0 += t0; base1 += t1; }
      __syncthreads();
    }
    if (tid == 0 && !scratch_mode && base0 + base1 > nb_active) redo = 1;   // cheaper to rebuild from Q
    __syncthreads();
    if (!redo) break;
    scratch_mode = 1;
  }
  for (int i = tid; i < m; i += NT) { P.activeH[om + i] = P.active[om + i]; P.sigmaH[om + i] = P.sigma[om + i]; }
  if (tid == 0) {
    BCtl &c = P.ctl[b];
    c.npos = base0; c.nneg = base1; c.H_valid = 1; c.scratch = scratch_mode;
    c.syrk_entries += base0 + base1; c.n_scratch += scratch_mode;
  }
}

// ordered list of the active rows with weights sqrt(sigma) (boost_gamma's A_J' Sigma_J A_J)
__device__ __noinline__ void p_active_list(const Args &P, int b) {
  __shared__ int warp_cnt[NW];
  __shared__ int base;
  const int m = P.m, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t om = (size_t)b * m;
  if (tid == 0) base = 0;
  __syncthreads();
  for (int start = 0; start < m; start += NT) {
    const int i = start + tid;
    const bool p = (i < m) && P.active[om + i];
    const unsigned bl = __ballot_sync(0xffffffffu, p);
    if (lane == 0) warp_cnt[warp] = __popc(bl);
    __syncthreads();
    int off = base;
    for (int w = 0; w < warp; w++) off += warp_cnt[w];
    if (p) { const int pos = off + __popc(bl & ((1u << lane) - 1u)); P.list_pos[om + pos] = i; P.w_pos[om + pos] = P.sqrt_sigma[om + i]; }
    __syncthreads();
    if (tid == 0) { int t = 0; for (int w = 0; w < NW; w++) t += warp_cnt[w]; base += t; }
    __syncthreads();
  }
  if (tid == 0) P.ctl[b].npos = base;
}

// boost_gamma path of the outer update (qpalm.c:613-627, iteration.c:159-211).  Returns with gamma / reset_newton set.
__device__ __noinline__ void p_boost(const Args &P, int b, double *scratch, const Smem &S) {
  __shared__ int need_gersh;
  const int n = P.n, m = P.m, tid = threadIdx.x;
  const BSet &st = P.st;
  const size_t om = (size_t)b * m, on = (size_t)b * n;
  double na = 0, ne = 0, nl = 0;
  for (int i = tid; i < m; i += NT) {
    const double t = P.y[om + i] / P.sigma[om + i];
    const double a = P.Ax[om + i] + t;
    P.Axys[om + i] = a;
    const int act = (a <= P.bmin[om + i]) || (a >= P.bmax[om + i]);
    P.active[om + i] = act;
    na += act; ne += act && !P.active_old[om + i]; nl += !act && P.active_old[om + i];
  }
  na = block_red<RED_SUM>(na, scratch); ne = block_red<RED_SUM>(ne, scratch); nl = block_red<RED_SUM>(nl, scratch);
  if (tid == 0) {
    BCtl &c = P.ctl[b];
    c.nb_active = (int)na; c.nb_enter = (int)ne; c.nb_leave = (int)nl; c.boost = 0;
    need_gersh = 0;
    if (ne == 0 && nl == 0) {
      c.boost = 1;
      if (na == 0) { c.gamma = 1e12; c.reset_newton = 1; }   // iteration.c:198-200
      else { c.scratch = 1; c.npos = 0; c.nneg = 0; need_gersh = 1; }
    } else if (c.gamma < st.gamma_max) { c.gamma = fmin(c.gamma * st.gamma_upd, st.gamma_max); c.reset_newton = 1; }
  }
  __syncthreads();
  if (need_gersh) {
    p_active_list(P, b);
    __syncthreads();
    double *Lb = P.L + (size_t)b * P.sLL;
    const int ld = P.ld;
    cta_syrk(Lb, ld, n, SY_ZERO, nullptr, 0, 0.0, P.At, P.list_pos + om, P.w_pos + om, P.ctl[b].npos, nullptr, nullptr, 0, S, nullptr);
    double ub = -1.0e300;
    for (int i = tid; i < n; i += NT) {   // Gershgorin: |row i| of the symmetric matrix
      double acc = 0.0;
      for (int j = 0; j <= i; j++) acc += fabs(Lb[(size_t)i + (size_t)j * ld]);
      for (int j = i + 1; j < n; j++) acc += fabs(Lb[(size_t)j + (size_t)i * ld]);
      ub = fmax(ub, acc);
    }
    ub = block_red<RED_MAX>(ub, scratch);
    if (tid == 0) {
      BCtl &c = P.ctl[b];
      c.gamma = fmax(st.gamma_max, 1e14 / ub);
      c.gamma_maxed = 1;
      c.reset_newton = 1;
    }
    __syncthreads();
  }
  // Qx / Qd shifts for a changed gamma (iteration.c:205-209); the Qd shift belongs to boost_gamma only
  const double g = P.ctl[b].gamma, gp = P.ctl[b].gamma_prev;
  if (g != gp) {
    const double tau = BSC(b, S_TAU);
    const int boosted = P.ctl[b].boost;
    for (int j = tid; j < n; j += NT) {
      P.Qx[on + j] = P.Qx[on + j] + (1.0 / g - 1.0 / gp) * P.x[on + j];
      if (boosted) P.Qd[on + j] = P.Qd[on + j] + (tau / g - tau / gp) * P.d[on + j];
    }
    __syncthreads();
    if (tid == 0) P.ctl[b].reset_newton = 1;
  }
}

// ------------------------------------------------------------------------------------------------
// line search (linesearch.c:14-120)
// ------------------------------------------------------------------------------------------------
// The breakpoints s > 0 (+inf included) go to buffer 0 of the sort as (bit pattern of s, index) pairs, compacted: a warp
// takes its slots with one shared atomic, so their order varies from run to run, which the sort's total order makes
// irrelevant.  The others (s <= 0 or NaN) are never walked by p_ls_select and are not stored.  Their count is S_NL.
__device__ __noinline__ void p_ls_build(const Args &P, int b, double *part, const Smem &S) {
  __shared__ unsigned n_brk;
  const int n = P.n, m = P.m, lane = threadIdx.x & 31;
  const size_t on = (size_t)b * n, om = (size_t)b * m, o2 = (size_t)b * 2 * m;
  unsigned long long *bk = ls_keys(S, 0);
  unsigned short *bp = ls_pos(S, 0);
  if (threadIdx.x == 0) n_brk = 0;
  const double inv_gamma = 1 / P.ctl[b].gamma;
  double eta = 0, beta = 0;
  for (int j = threadIdx.x; j < n; j += NT) {
    double qd = P.Qd[on + j];
    const double dj = P.d[on + j];
    if (P.st.proximal) { qd = qd + inv_gamma * dj; P.Qd[on + j] = qd; }
    eta += dj * qd; beta += dj * P.df[on + j];
  }
  __syncthreads();   // n_brk = 0 before the first slot is taken
  double a_part = 0, b_part = 0, n_l = 0;
  for (int i0 = 0; i0 < m; i0 += NT) {   // whole warps per step: the ballots below
    const int i = i0 + threadIdx.x;
    bool inL[2] = {false, false};
    double sv[2] = {0.0, 0.0};
    if (i < m) {
      const double ss = P.sqrt_sigma[om + i], sg = P.sigma[om + i], ax = P.Ax[om + i], yi = P.y[om + i];
      const double t = ss * P.Ad[om + i];
      double dl[2], al[2];
      dl[1] = t; dl[0] = t * -1;
      double u = ax - P.bmin[om + i]; u = sg * u; u = yi + u; al[0] = u / ss;
      u = P.bmax[om + i] - ax; u = sg * u; u = u - yi; al[1] = u / ss;
#pragma unroll
      for (int hh = 0; hh < 2; hh++) {
        const int idx = i + hh * m;
        const double s = al[hh] / dl[hh];
        const bool inP = dl[hh] > 0;
        inL[hh] = s > 0; sv[hh] = s;
        const double d2 = dl[hh] * dl[hh], dalp = dl[hh] * al[hh];
        P.ls_da[o2 + idx] = inP ? d2 : -d2;
        P.ls_db[o2 + idx] = inP ? -dalp : dalp;
        if ((int)inL[hh] + (int)inP == 1) { a_part += d2; b_part += dalp; }
        n_l += inL[hh];
      }
    }
    const unsigned b0 = __ballot_sync(0xffffffffu, inL[0]), b1 = __ballot_sync(0xffffffffu, inL[1]);
    unsigned at = 0;
    if (lane == 0 && (b0 | b1)) at = atomicAdd(&n_brk, (unsigned)(__popc(b0) + __popc(b1)));
    at = __shfl_sync(0xffffffffu, at, 0);
    const unsigned lt = (1u << lane) - 1u;
    if (inL[0]) { const unsigned k = at + __popc(b0 & lt); bk[k] = (unsigned long long)__double_as_longlong(sv[0]); bp[k] = (unsigned short)i; }
    if (inL[1]) { const unsigned k = at + __popc(b0) + __popc(b1 & lt); bk[k] = (unsigned long long)__double_as_longlong(sv[1]); bp[k] = (unsigned short)(i + m); }
  }
  const double vals[5] = {eta, beta, a_part, b_part, n_l};
  const int ops[5] = {RED_SUM, RED_SUM, RED_SUM, RED_SUM, RED_SUM};
  const int slots[5] = {S_ETA, S_BETA, S_LS_A, S_LS_B, S_NL};
  block_red_multi<5>(P, b, vals, ops, slots, part);
#ifdef QB_BP_DEBUG
  __syncthreads();
  if (threadIdx.x == 0) assert(n_brk == (unsigned)BSC(b, S_NL));
#endif
}

// (ka, pa) < (kb, pb) lexicographically.  The positions of one sort are distinct, so this is a total order and every sort by
// it returns the permutation of a stable sort by key.  Keys compare as unsigned integers: for positive doubles and +inf that
// is the order of the values.
__device__ __forceinline__ bool kp_less(unsigned long long ka, unsigned pa, unsigned long long kb, unsigned pb) {
  return (ka < kb) | ((ka == kb) & (pa < pb));   // no short circuit: predicates, not branches, in the network and the merges
}

// Sorts the N <= SORT_MAX (key, position) pairs of buffer 0 by kp_less; the result is in buffer 0.  Thread t sorts pairs
// [8 t, 8 t + 8) in registers (a 19-comparator network), then each merge level doubles the run length: thread t writes
// outputs [8 t, 8 t + 8) of its pair of runs, starting where a binary search of the merge path puts it.  One barrier per level
// (8 at N = 2048).  The register stage writes to buffer (number of levels & 1), so the last level lands in buffer 0.
__device__ __noinline__ void p_ls_sort(int N, const Smem &S) {
  const int tid = threadIdx.x, o0 = 8 * tid;
  int levels = 0;
  for (int w = 8; w < N; w <<= 1) levels++;
  int buf = levels & 1;
  if (o0 < N) {
    const unsigned long long *ki = ls_keys(S, 0);
    const unsigned short *pi = ls_pos(S, 0);
    unsigned long long k[8];
    unsigned p[8];
#pragma unroll
    for (int u = 0; u < 8; u++) {   // past N: (~0, 0xFFFF) sorts after every pair of the input (positions < SORT_MAX)
      k[u] = o0 + u < N ? ki[o0 + u] : ~0ull;
      p[u] = o0 + u < N ? pi[o0 + u] : 0xFFFFu;
    }
    constexpr int NET[19][2] = {{0, 2}, {1, 3}, {4, 6}, {5, 7}, {0, 4}, {1, 5}, {2, 6}, {3, 7}, {0, 1}, {2, 3},
                                {4, 5}, {6, 7}, {2, 4}, {3, 5}, {1, 4}, {3, 6}, {1, 2}, {3, 4}, {5, 6}};
#pragma unroll
    for (int c = 0; c < 19; c++) {
      const int x = NET[c][0], y = NET[c][1];
      const bool sw = kp_less(k[y], p[y], k[x], p[x]);
      const unsigned long long kx = k[x];
      const unsigned px = p[x];
      k[x] = sw ? k[y] : k[x]; p[x] = sw ? p[y] : p[x];
      k[y] = sw ? kx : k[y]; p[y] = sw ? px : p[y];
    }
    unsigned long long *ko = ls_keys(S, buf);
    unsigned short *po = ls_pos(S, buf);
#pragma unroll
    for (int u = 0; u < 8; u++)
      if (o0 + u < N) { ko[o0 + u] = k[u]; po[o0 + u] = (unsigned short)p[u]; }
  }
  for (int w = 8; w < N; w <<= 1) {
    __syncthreads();
    const unsigned long long *ki = ls_keys(S, buf);
    const unsigned short *pi = ls_pos(S, buf);
    unsigned long long *ko = ls_keys(S, buf ^ 1);
    unsigned short *po = ls_pos(S, buf ^ 1);
    if (o0 < N) {   // runs A = [a0, a0 + na), B = [a0 + w, a0 + w + nb); this thread's outputs start at d in their merge
      const int a0 = o0 & ~(2 * w - 1), b0 = a0 + w, d = o0 - a0;
      const int na = min(w, N - a0), nb = max(0, min(w, N - b0));
      int lo = max(0, d - nb), hi = min(d, na);
      while (lo < hi) {   // the number of A pairs among the first d outputs
        const int mid = (lo + hi) >> 1;
        if (kp_less(ki[a0 + mid], pi[a0 + mid], ki[b0 + d - mid - 1], pi[b0 + d - mid - 1])) lo = mid + 1;
        else hi = mid;
      }
      int ia = lo, ib = d - lo;
      // heads of the two runs; an exhausted run's head (~0, 0x10000) is greater than every pair
      unsigned long long ka = ia < na ? ki[a0 + ia] : ~0ull, kb = ib < nb ? ki[b0 + ib] : ~0ull;
      unsigned pa = ia < na ? pi[a0 + ia] : 0x10000u, pb = ib < nb ? pi[b0 + ib] : 0x10000u;
      const int cnt = min(8, N - o0);
#pragma unroll
      for (int u = 0; u < 8; u++) {
        if (u < cnt) {
          const bool ta = kp_less(ka, pa, kb, pb);
          ko[o0 + u] = ta ? ka : kb; po[o0 + u] = (unsigned short)(ta ? pa : pb);
          if (ta) { ia++; ka = ia < na ? ki[a0 + ia] : ~0ull; pa = ia < na ? pi[a0 + ia] : 0x10000u; }
          else { ib++; kb = ib < nb ? ki[b0 + ib] : ~0ull; pb = ib < nb ? pi[b0 + ib] : 0x10000u; }
        }
      }
    }
    buf ^= 1;
  }
}

// Walks the sorted breakpoints (p_ls_sort's buffer 0; nothing may write the union region in between) in chunks of NT,
// carrying the running (a, b) sums; tau = -b / a at the first breakpoint where a s + b > 0.
__device__ __noinline__ void p_ls_select(const Args &P, int b, const Smem &S) {
  __shared__ double wa[NW], wb[NW];
  __shared__ double carry_a, carry_b;
  __shared__ int found;
  const size_t o2 = (size_t)b * 2 * P.m;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nL = (int)BSC(b, S_NL);
  const unsigned long long *sk = ls_keys(S, 0);
  const unsigned short *sp = ls_pos(S, 0);
  if (tid == 0) {
    carry_a = BSC(b, S_ETA) + BSC(b, S_LS_A); carry_b = BSC(b, S_BETA) - BSC(b, S_LS_B); found = 0x7fffffff;
    P.ctl[b].ls_breakpoints += nL;
  }
  __syncthreads();
  for (int start = 0; start < nL; start += NT) {
    const int i = start + tid;
    double ta = 0.0, tb = 0.0, s = 0.0;
    if (i < nL) { const unsigned int idx = sp[i]; ta = P.ls_da[o2 + idx]; tb = P.ls_db[o2 + idx]; s = __longlong_as_double((long long)sk[i]); }
    double ia = ta, ib = tb;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double ua = __shfl_up_sync(0xffffffffu, ia, o), ub = __shfl_up_sync(0xffffffffu, ib, o);
      if (lane >= o) { ia += ua; ib += ub; }
    }
    if (lane == 31) { wa[warp] = ia; wb[warp] = ib; }
    __syncthreads();
    double oa = 0.0, ob = 0.0;
    for (int w = 0; w < warp; w++) { oa += wa[w]; ob += wb[w]; }
    double ea = __shfl_up_sync(0xffffffffu, ia, 1), eb = __shfl_up_sync(0xffffffffu, ib, 1);
    if (lane == 0) { ea = 0.0; eb = 0.0; }
    const double a_i = carry_a + (oa + ea), b_i = carry_b + (ob + eb);
    if (i < nL && (a_i * s + b_i > 0)) atomicMin(&found, i);
    __syncthreads();
    if (found != 0x7fffffff) {
      if (i == found) { BSC(b, S_TAU) = -b_i / a_i; P.ctl[b].ls_walked += i + 1; }
      return;
    }
    if (tid == NT - 1) { carry_a += oa + ia; carry_b += ob + ib; }
    __syncthreads();
  }
  if (tid == 0) { BSC(b, S_TAU) = -carry_b / carry_a; P.ctl[b].ls_walked += nL; }
}

__device__ void p_update_iterate(const Args &P, int b) {
  const int n = P.n, m = P.m;
  const double tau = BSC(b, S_TAU);
  const size_t on = (size_t)b * n, om = (size_t)b * m;
  for (int i = threadIdx.x; i < n; i += NT) {
    const double xi = P.x[on + i];
    P.x_prev[on + i] = xi; P.x[on + i] = xi + tau * P.d[on + i];
    const double qd = P.Qd[on + i] * tau;
    P.Qd[on + i] = qd; P.Qx[on + i] = P.Qx[on + i] + qd;
  }
  for (int i = threadIdx.x; i < m; i += NT) {
    const double ad = P.Ad[om + i] * tau;
    P.Ad[om + i] = ad; P.Ax[om + i] = P.Ax[om + i] + ad;
  }
}

// store_solution (termination.c:242-252) + compute_objective (iteration.c:231-270)
__device__ __noinline__ void p_store(const Args &P, int b, double *scratch) {
  const int n = P.n, m = P.m;
  const BSet &st = P.st;
  const size_t on = (size_t)b * n, om = (size_t)b * m;
  const double cinv = P.ctl[b].cinv, inv_gamma = 1 / P.ctl[b].gamma;
  double obj = 0;
  for (int i = threadIdx.x; i < n; i += NT) {
    const double xi = P.x[on + i];
    P.x_out[on + i] = st.scaling ? xi * P.D[i] : xi;
    if (st.proximal) obj += (0.5 * (P.Qx[on + i] - inv_gamma * xi) + P.q[on + i]) * xi;
    else obj += (0.5 * P.Qx[on + i] + P.q[on + i]) * xi;
  }
  for (int i = threadIdx.x; i < m; i += NT) {
    double v = P.yh[om + i];
    if (st.scaling) { v *= cinv; v = v * P.E[i]; }
    P.y_out[om + i] = v;
  }
  obj = block_red<RED_SUM>(obj, scratch);
  if (threadIdx.x == 0) { if (st.scaling) obj *= cinv; P.ctl[b].objective = obj + st.data_c; }
}

// ------------------------------------------------------------------------------------------------
// the persistent kernel
// ------------------------------------------------------------------------------------------------
#define PH(k) do { if (P.prof) { const long long t_ = clock64(); if (tid == NT - 1) atomicAdd(reinterpret_cast<unsigned long long *>(P.prof + (size_t)b * 32 + (k)), (unsigned long long)(t_ - t_ph)); t_ph = t_; } } while (0)
#ifndef QB_BP_MINB
#define QB_BP_MINB (QB_BP_NT <= 192 ? 4 : 3)
#endif
#ifndef QB_BP_PROBE
__global__ void __launch_bounds__(NT, QB_BP_MINB) kbp_solve(const Args P) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ double scratch[32];
  __shared__ int s_b;
  __shared__ Flags s_f;
  __shared__ int s_info;
  __shared__ __align__(8) unsigned long long s_udbar[NBAR];   // per-column mbarriers of the dataflows (chain warp -> row owners)
  unsigned ud_phase = 0, ud_phase_hi = 0;                      // phases so far of barriers < UW / >= UW (see cta_potrf)
  if (threadIdx.x == 0) {
    for (int j = 0; j < NBAR; j++) ud_mbar_init(s_udbar + j, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  Smem S;
  S.u = smem_raw;
  S.panel = reinterpret_cast<double *>(smem_raw);
  S.vs = reinterpret_cast<double *>(smem_raw + kUnionBytes);
  S.v = S.vs + VS_LEN;
  S.rd = S.v + NMAX + 16;
  const int tid = threadIdx.x, n = P.n, m = P.m, ld = P.ld;
  const BSet &st = P.st;
  for (;;) {
    __syncthreads();
    if (tid == 0) s_b = atomicAdd(P.queue, 1);
    __syncthreads();
    const int b = s_b;
    if (b >= P.nb) return;
    const size_t on = (size_t)b * n, om = (size_t)b * m;
    double *Hb = P.H + (size_t)b * P.sLL, *Lb = P.L + (size_t)b * P.sLL, *rdg = P.rdiag + (size_t)b * P.sR;
    long long t_ph = clock64();
    if (P.prof && tid == 0) for (int k = 0; k < 32; k++) P.prof[(size_t)b * 32 + k] = 0;
    p_init(P, b, scratch);
    __syncthreads();
    if (b < P.nwarm) { p_warm(P, b, scratch, S); __syncthreads(); }
    PH(0);
    for (;;) {
      // ---- residuals + termination scalars ----
      p_res_m(P, b, S.vs);
      __syncthreads();
      PH(1);
      p_gemv_rows(n, m, n, P.At, P.yh + om, P.Atyh + on, 1.0, S);
      __syncthreads();
      PH(2);
      p_res_n(P, b, S.vs);
      __syncthreads();
      if (tid == 0) p_control(P, b, s_f);
      __syncthreads();
      const Flags f = s_f;
      __syncthreads();   // everyone holds a private copy before thread 0 touches s_f again
      PH(3);
      if (f.done) break;
      // ---- outer updates ----
      if (f.sigma) { p_update_sigma(P, b, scratch); __syncthreads(); }
      if (f.outer) { p_outer(P, b, f.outer); __syncthreads(); }
      if (st.proximal && f.boost) { p_boost(P, b, scratch, S); __syncthreads(); }
      PH(4);
      // ---- inner step ----
      if (f.inner) {
        int refac = f.refac, factor = f.factor;
        if (f.updown) {   // rank update of the factor instead of a refactorisation (newton.c:103-108)
          p_updown_lists(P, b);
          if (tid == 0) s_info = 0;
          __syncthreads();
          const int ne = P.ctl[b].npos, nl = P.ctl[b].nneg;
          for (int off = 0; off < ne + nl; off += KU) {
            const int k = (ne + nl - off < KU) ? ne + nl - off : KU;
            const int kpos = (ne - off < 0) ? 0 : ((ne - off < k) ? ne - off : k);
            cta_updown_sweep(Lb, ld, n, rdg, P.At, P.list_pos + om + off, P.w_pos + om + off, k, kpos, S, &s_info,
                             s_udbar, ud_phase, P.prof ? P.prof + (size_t)b * 32 : nullptr);
          }
          __syncthreads();
          if (tid == 0) {
            BCtl &c = P.ctl[b];
            c.n_updown += (ne + nl + KU - 1) / KU; c.updown_ranks += ne + nl;
            if (s_info) { c.n_updown_fail++; c.scratch = !c.H_valid; c.n_refac++; c.refac_J += c.nb_active; }
          }
          if (s_info) { refac = 1; factor = 1; }   // a downdate lost definiteness: rebuild the factor from H
          __syncthreads();
          PH(14);
        }
        p_lists(P, b, refac);
        __syncthreads();
        PH(5);
        if (refac) {
          const BCtl c = P.ctl[b];   // scratch: H <- c Q + the lists, else H += / -= the lists
          cta_syrk(Hb, ld, n, c.scratch ? SY_SRC : SY_DST, P.Qs, n, c.c, P.At, P.list_pos + om, P.w_pos + om, c.npos, P.list_neg + om,
                   P.w_neg + om, c.nneg, S, P.prof ? P.prof + (size_t)b * 32 : nullptr);
        }
        PH(6);
        for (int i = tid; i < n; i += NT) S.v[i] = P.dphi[on + i] * -1;
        __syncthreads();
        if (factor) {
          const double beta = P.ctl[b].beta;
          if (tid == 0) s_info = 0;
          cta_potrf(Lb, ld, f.fq ? P.Qs : Hb, f.fq ? n : ld, f.fq ? P.ctl[b].c : 1.0, beta, n, rdg, S, &s_info,
                    s_udbar, ud_phase, ud_phase_hi, P.prof ? P.prof + (size_t)b * 32 : nullptr);
        }
        PH(7);
        cta_chol_solve(Lb, ld, n, rdg, S, s_udbar, ud_phase, P.prof ? P.prof + (size_t)b * 32 : nullptr);
        for (int i = tid; i < n; i += NT) P.d[on + i] = S.v[i];
        for (int i = tid; i < m; i += NT) P.active_old[om + i] = P.active[om + i];
        __syncthreads();
        PH(8);
        // ---- line search + iterate update ----
        p_gemv_rows(n, n, n, P.Qs, P.d + on, P.Qd + on, P.ctl[b].c, S);
        __syncthreads();
        PH(13);
        p_gemv_rows(m, n, m, P.Am, P.d + on, P.Ad + om, 1.0, S);
        __syncthreads();
        PH(9);
        p_ls_build(P, b, S.vs, S);
        __syncthreads();
        PH(10);
        p_ls_sort((int)BSC(b, S_NL), S);
        __syncthreads();
        PH(11);
        p_ls_select(P, b, S);
        __syncthreads();
        p_update_iterate(P, b);
        __syncthreads();
        PH(12);
      }
      if (tid == 0) {   // end of iteration (qpalm.c:484, 711-735)
        BCtl &c = P.ctl[b];
        c.iter++;
        s_f.done = 0;
        if (c.iter >= st.max_iter) { c.status = QPALM_MAX_ITER_REACHED; c.done = 1; s_f.done = 1; }
      }
      __syncthreads();
      if (s_f.done) break;
    }
    __syncthreads();
    p_store(P, b, scratch);
  }
}

#else   // QB_BP_PROBE
// ------------------------------------------------------------------------------------------------
// test probes: the Newton-step building blocks and the line-search sort on caller data, run the way kbp_solve runs them
// (same CTA shape, launch bounds, shared-memory carving, per-column mbarriers whose phase carries across the sweeps and the
// instances of a CTA, persistent CTAs on an atomic queue), so that a test checks the code the solver executes.
// They are built from this file in objects of their own (build.sh, -DQB_BP_PROBE): with a second caller in the same
// translation unit, the __noinline__ building blocks (cta_updown_sweep, potrf_panel) would no longer see kbp_solve's
// __shared__ mbarrier and info addresses as constants, and kbp_solve would be compiled differently (more spills).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ Smem probe_smem(unsigned char *smem_raw) {
  Smem S;
  S.u = smem_raw;
  S.panel = reinterpret_cast<double *>(smem_raw);
  S.vs = reinterpret_cast<double *>(smem_raw + kUnionBytes);
  S.v = S.vs + VS_LEN;
  S.rd = S.v + NMAX + 16;
  return S;
}

// per instance b (batch.cuh, BpProbeArgs): H <- src, H += / -= the SYRK lists, L <- chol(H + beta I), d_fused <- (L L')^{-1} rhs;
// then the rank update of L by the rows upd[0 .. nup) in sweeps of KU (kbp_solve's update branch) and d_after <- (L L')^{-1} rhs
// with the final L and rdiag; then P.rounds rounds of {+ or - the update rows, solve} and P.rounds rounds of {solve}.  info[b]: bit 0 a sweep lost definiteness, bit 1
// the factorisation met a non-positive pivot.
__global__ void __launch_bounds__(NT, QB_BP_MINB) kbp_probe_newton(const BpProbeArgs P) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_b;
  __shared__ int s_info;
  __shared__ __align__(8) unsigned long long s_udbar[NBAR];
  unsigned ud_phase = 0, ud_phase_hi = 0;
  if (threadIdx.x == 0) {
    for (int j = 0; j < NBAR; j++) ud_mbar_init(s_udbar + j, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const Smem S = probe_smem(smem_raw);
  const int tid = threadIdx.x, n = P.n, m = P.m, ld = P.ld;
  for (;;) {
    __syncthreads();
    if (tid == 0) s_b = atomicAdd(P.queue, 1);
    __syncthreads();
    const int b = s_b;
    if (b >= P.nb) return;
    const size_t on = (size_t)b * n, sLL = (size_t)ld * ld;
    double *Hb = P.H + (size_t)b * sLL, *Lb = P.L + (size_t)b * sLL, *rdg = P.rdiag + (size_t)b * ld;
    const int npos = P.cnt[4 * b], nneg = P.cnt[4 * b + 1], nup = P.cnt[4 * b + 2], kpos = P.cnt[4 * b + 3];
    const int *lst = P.lists + (size_t)b * 3 * m;
    const double *wt = P.wts + (size_t)b * 3 * m;
    const double *src = P.from_q ? P.H0 : P.H0 + (size_t)b * n * n;
    const double sc = P.from_q ? P.sscale : 1.0;
    if (P.from_q)   // kbp_solve's rebuild: H <- sscale Q + the lists
      cta_syrk(Hb, ld, n, SY_SRC, P.H0, n, sc, P.At, lst, wt, npos, lst + m, wt + m, nneg, S, nullptr);
    else {          // the incremental form: H <- H0, then H += / -= the lists in place
      for (int i = tid; i < n; i += NT)
        for (int j = 0; j <= i; j++) Hb[(size_t)i + (size_t)ld * j] = src[(size_t)i + (size_t)n * j];
      __syncthreads();
      cta_syrk(Hb, ld, n, SY_DST, nullptr, 0, 0.0, P.At, lst, wt, npos, lst + m, wt + m, nneg, S, nullptr);
    }
    for (int i = tid; i < n; i += NT) S.v[i] = P.rhs[on + i];
    __syncthreads();
    if (tid == 0) s_info = 0;
    // from_q without lists: the f.fq path, the factor reads the shared source (lds = n) directly; else the refactorisation of H
    const bool fq = P.from_q && npos + nneg == 0;
    cta_potrf(Lb, ld, fq ? P.H0 : Hb, fq ? n : ld, fq ? sc : 1.0, P.beta, n, rdg, S, &s_info, s_udbar, ud_phase, ud_phase_hi, nullptr);
    cta_chol_solve(Lb, ld, n, rdg, S, s_udbar, ud_phase, nullptr);
    for (int i = tid; i < n; i += NT) P.d_fused[on + i] = S.v[i];
    __syncthreads();
    const int finfo = s_info;
    __syncthreads();
    if (tid == 0) s_info = 0;
    __syncthreads();
    for (int off = 0; off < nup; off += KU) {
      const int k = (nup - off < KU) ? nup - off : KU;
      const int kp = (kpos - off < 0) ? 0 : ((kpos - off < k) ? kpos - off : k);
      cta_updown_sweep(Lb, ld, n, rdg, P.At, lst + 2 * m + off, wt + 2 * m + off, k, kp, S, &s_info, s_udbar, ud_phase, nullptr);
    }
    __syncthreads();
    if (tid == 0) P.info[b] = (s_info ? 1 : 0) | (finfo ? 2 : 0);
    for (int i = tid; i < n; i += NT) S.v[i] = P.rhs[on + i];
    __syncthreads();
    cta_chol_solve(Lb, ld, n, rdg, S, s_udbar, ud_phase, nullptr);
    for (int i = tid; i < n; i += NT) P.d_after[on + i] = S.v[i];
    for (int r = 0; r < 2 * P.rounds; r++) {   // rounds x {update sweeps, solve}, then rounds x {solve}
      __syncthreads();
      if (r < P.rounds) {   // the update rows, all entering in even rounds and all leaving in odd ones
        for (int off = 0; off < nup; off += KU) {
          const int k = (nup - off < KU) ? nup - off : KU;
          cta_updown_sweep(Lb, ld, n, rdg, P.At, lst + 2 * m + off, wt + 2 * m + off, k, (r & 1) ? 0 : k, S, &s_info, s_udbar, ud_phase, nullptr);
        }
      }
      for (int i = tid; i < n; i += NT) S.v[i] = P.rhs[on + i] * (double)(r + 1);
      __syncthreads();
      cta_chol_solve(Lb, ld, n, rdg, S, s_udbar, ud_phase, nullptr);
      for (int i = tid; i < n; i += NT) P.d_rounds[((size_t)b * 2 * P.rounds + r) * n + i] = S.v[i];
    }
  }
}

// p_ls_sort on instance b's N (key, val) pairs at keys + b N, vals + b N, loaded the way p_ls_build leaves them (position =
// index in the array): the keys are sorted in place, vals_out + b N receives the vals in the sorted order
__global__ void __launch_bounds__(NT, QB_BP_MINB) kbp_probe_sort(int nb, int N, unsigned long long *keys, const unsigned int *vals,
                                                                 unsigned int *vals_out, int *queue) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_b;
  const Smem S = probe_smem(smem_raw);
  for (;;) {
    __syncthreads();
    if (threadIdx.x == 0) s_b = atomicAdd(queue, 1);
    __syncthreads();
    const int b = s_b;
    if (b >= nb) return;
    unsigned long long *kb = keys + (size_t)b * N;
    for (int i = threadIdx.x; i < N; i += NT) { ls_keys(S, 0)[i] = kb[i]; ls_pos(S, 0)[i] = (unsigned short)i; }
    __syncthreads();
    p_ls_sort(N, S);
    __syncthreads();
    for (int i = threadIdx.x; i < N; i += NT) { kb[i] = ls_keys(S, 0)[i]; vals_out[(size_t)b * N + i] = vals[(size_t)b * N + ls_pos(S, 0)[i]]; }
  }
}

// occupancy x SMs capped at nb: the grid QB_BP_SOLVE gives kbp_solve
static int probe_grid(const void *kernel, int nb, int *grid) {
  QB_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
  int per_sm = 0, dev = 0, sms = 0;
  QB_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, NT, kSmemBytes));
  QB_CUDA_TRY(cudaGetDevice(&dev));
  QB_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  *grid = (per_sm < 1 ? 1 : per_sm) * sms;
  if (*grid > nb) *grid = nb;
  return 0;
}
#endif  // QB_BP_PROBE

}  // namespace QB_BP_NAMESPACE (bp / bp4)

#ifndef QB_BP_PROBE

bool QB_BP_SUPPORTED(int n, int m) {
  return n >= 1 && n <= QB_BP_NAMESPACE::NMAX && m >= 1 && 2 * m <= QB_BP_NAMESPACE::SORT_MAX && m <= QB_BP_NAMESPACE::VS_LEN;
}

int QB_BP_SOLVE(QPALMB200Batch *B, int nb, int nwarm, int wx, int wy) {
  using namespace QB_BP_NAMESPACE;
  Engine *e = B->shared;
  Args P;
  memset(&P, 0, sizeof(P));
  P.nb = nb; P.n = B->n; P.m = B->m; P.ld = B->ld; P.st = B->set;
  P.At = e->At; P.Am = B->Am; P.Qs = B->Qs; P.D = e->D; P.Dinv = e->Dinv; P.E = e->E; P.Einv = e->Einv;
  P.q_raw = B->q_raw; P.bmin_raw = B->bmin_raw; P.bmax_raw = B->bmax_raw; P.x_out = B->x_out; P.y_out = B->y_out;
  P.q = B->q; P.bmin = B->bmin; P.bmax = B->bmax; P.x = B->x; P.y = B->y; P.Ax = B->Ax; P.Qx = B->Qx; P.Aty = B->Aty;
  P.x_prev = B->x_prev; P.x0 = B->x0; P.sigma = B->sigma; P.sigma_inv = B->sigma_inv; P.sqrt_sigma = B->sqrt_sigma;
  P.Axys = B->Axys; P.z = B->z; P.pri_res = B->pri_res; P.pri_res_in = B->pri_res_in; P.yh = B->yh; P.Atyh = B->Atyh;
  P.df = B->df; P.dphi = B->dphi; P.d = B->d; P.Qd = B->Qd; P.Ad = B->Ad;
  P.active = B->active; P.active_old = B->active_old; P.active_cand = B->active_cand; P.activeH = B->activeH;
  P.list_pos = B->list_pos; P.list_neg = B->list_neg; P.sigmaH = B->sigmaH; P.w_pos = B->w_pos; P.w_neg = B->w_neg;
  P.H = B->H; P.L = B->L; P.rdiag = B->invdiag;
  P.sLL = (long long)B->ld * B->npad; P.sR = (long long)B->npad * kPanel;
  P.prof = B->prof;
  P.nwarm = nwarm; P.x_ws = wx ? B->x_ws : nullptr; P.y_ws = wy ? B->y_ws : nullptr;
  P.ls_da = B->ls_da; P.ls_db = B->ls_db; P.scal = B->scal; P.ctl = B->ctl; P.queue = B->queue;
  static int ctas_per_sm = 0, num_sms = 0;
  if (!ctas_per_sm) {
    QB_CUDA_TRY(cudaFuncSetAttribute(kbp_solve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
    QB_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, kbp_solve, NT, kSmemBytes));
    int dev = 0;
    QB_CUDA_TRY(cudaGetDevice(&dev));
    QB_CUDA_TRY(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
    if (ctas_per_sm < 1) ctas_per_sm = 1;
  }
  int grid = ctas_per_sm * num_sms;
  if (grid > nb) grid = nb;
  QB_CUDA_TRY(cudaMemsetAsync(B->queue, 0, sizeof(int), B->stream));
  QB_LAUNCH(kbp_solve, grid, NT, kSmemBytes, B->stream, P);
  QB_CUDA_TRY(cudaGetLastError());
  return 0;
}
#else   // QB_BP_PROBE

int QB_BP_PROBE_NEWTON(const BpProbeArgs &P, cudaStream_t s) {
  using namespace QB_BP_NAMESPACE;
  if (P.nb < 1 || P.n < 1 || P.n > NMAX || P.m < 1) return 1;
  int grid = 0;
  if (int r = probe_grid((const void *)kbp_probe_newton, P.nb, &grid)) return r;
  QB_CUDA_TRY(cudaMemsetAsync(P.queue, 0, sizeof(int), s));
  QB_LAUNCH(kbp_probe_newton, grid, NT, kSmemBytes, s, P);
  QB_CUDA_TRY(cudaGetLastError());
  return 0;
}

int QB_BP_PROBE_SORT(int nb, int N, unsigned long long *keys, const unsigned int *vals, unsigned int *vals_out, int *queue, cudaStream_t s) {
  using namespace QB_BP_NAMESPACE;
  if (nb < 1 || N < 1 || N > SORT_MAX) return 1;
  int grid = 0;
  if (int r = probe_grid((const void *)kbp_probe_sort, nb, &grid)) return r;
  QB_CUDA_TRY(cudaMemsetAsync(queue, 0, sizeof(int), s));
  QB_LAUNCH(kbp_probe_sort, grid, NT, kSmemBytes, s, nb, N, keys, vals, vals_out, queue);
  QB_CUDA_TRY(cudaGetLastError());
  return 0;
}
#endif  // QB_BP_PROBE

}  // namespace qb
