// batch.cu -- batch entry point (include/qpalm_b200.h Part 3): nb QPs that share Q, A and the settings but have
// their own q, bmin, bmax (BASELINE config 4, the chain80w-style MPC sweep).
//
// All instances advance in lock step through the QPALM iteration; every step of the iteration is ONE kernel
// launch over the whole batch (grid.y / grid.x = instance) and the per-instance control flow of qpalm_solve
// (src/qpalm.c:484-711: terminate / outer update / forced outer update / inner step, refactor decision of
// src/newton.c:96-118) runs on the device in k_control, one thread per instance, so the host only launches a fixed
// kernel sequence per iteration and polls one counter.  Per-instance Newton systems are assembled with the batched
// DMMA SYRK and factorised with the batched blocked Cholesky of dense.cu (the shared Q and A stay in L2).
//
// Ruiz scaling: D and E depend on A only and are shared; the cost scaling c = 1/max(1, |D q|inf) (scaling.c:84-89)
// depends on q and is per instance, so the shared scaled Hessian is kept as D Q D and c is applied on the fly.
#include "batch.cuh"
#include <stdlib.h>
#include <math.h>
#include <string.h>

using namespace qb;

namespace {

#define BSC(b, slot) scal[(size_t)(b) * S_COUNT + (slot)]

// ------------------------------------------------------------------------------------------------
// per-instance initialisation: scale the inputs, cold start (qpalm_warm_start(NULL, NULL)), sigma
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
kb_init(int n, int m, BSet st, const double *__restrict__ D, const double *__restrict__ E,
        const double *__restrict__ q_raw, const double *__restrict__ bmin_raw, const double *__restrict__ bmax_raw,
        double *q, double *bmin, double *bmax, double *x, double *y, double *Ax, double *Qx, double *Aty, double *x_prev,
        double *x0, double *sigma, double *sigma_inv, double *sqrt_sigma, double *Qd, double *Ad, double *d, double *pri_res_in,
        int *active, int *active_old, int *activeH, double *scal, BCtl *ctl) {
  __shared__ double scratch[32];
  __shared__ double cc_s;
  const int b = blockIdx.x, tid = threadIdx.x;
  const size_t on = (size_t)b * n, om = (size_t)b * m;
  // q <- c * (D .* q), c = 1 / max(1, |D q|inf)   (scaling.c:82-90, Qx = 0 at setup)
  double mx = 0.0;
  for (int i = tid; i < n; i += blockDim.x) {
    double v = q_raw[on + i];
    if (st.scaling) v = D[i] * v;
    q[on + i] = v;
    mx = fmax(mx, fabs(v));
  }
  mx = block_red<RED_MAX>(mx, scratch);
  if (tid == 0) cc_s = st.scaling ? 1 / fmax(1.0, mx) : 1.0;
  __syncthreads();
  const double cc = cc_s;
  for (int i = tid; i < n; i += blockDim.x) {
    if (st.scaling) q[on + i] *= cc;
    x[on + i] = 0; Qx[on + i] = 0; Aty[on + i] = 0; x_prev[on + i] = 0; x0[on + i] = 0; Qd[on + i] = 0; d[on + i] = 0;
  }
  double dist2 = 0.0;
  for (int i = tid; i < m; i += blockDim.x) {
    double lo = bmin_raw[om + i], hi = bmax_raw[om + i];
    if (st.scaling) { lo = E[i] * lo; hi = E[i] * hi; }
    bmin[om + i] = lo; bmax[om + i] = hi;
    y[om + i] = 0; Ax[om + i] = 0; Ad[om + i] = 0; pri_res_in[om + i] = 0;
    active[om + i] = 0; active_old[om + i] = 0; activeH[om + i] = 0;
    const double t = 0.0 - fmax(lo, fmin(0.0, hi));
    dist2 += t * t;
  }
  dist2 = block_red<RED_SUM>(dist2, scratch);
  __shared__ double sig_s;
  if (tid == 0) {
    double s = st.sigma_init * 1.0 / fmax(1.0, 0.5 * dist2);   // f = 0 at x = 0 (iteration.c:50-58)
    s = fmax(1e-4, fmin(s, 1e4));
    sig_s = s;
    BCtl c;
    memset(&c, 0, sizeof(c));
    c.reset_newton = 1; c.gamma = st.gamma_init; c.gamma_prev = st.gamma_init; c.eps_abs_in = st.eps_abs_in; c.eps_rel_in = st.eps_rel_in;
    c.c = cc; c.cinv = 1.0 / cc; c.status = QPALM_UNSOLVED;
    ctl[b] = c;
    for (int k = 0; k < S_COUNT; k++) BSC(b, k) = 0.0;
  }
  __syncthreads();
  const double s = sig_s;
  for (int i = tid; i < m; i += blockDim.x) { sigma[om + i] = s; sigma_inv[om + i] = 1.0 / s; sqrt_sigma[om + i] = sqrt(s); }
}

// ------------------------------------------------------------------------------------------------
// warm start of instances b < grid after kb_init (qpalm_warm_start, qpalm.c:322-399): x = Dinv x_ws (x0 = x_prev = x),
// y = c Einv y_ws; with x, kb_gemv_rows / kb_gemv_cols then form Qd = c (D Q D) x and Ad = A x, and kb_warm_sigma finishes.
// A null x_ws or y_ws leaves that part cold.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
kb_warm_set(int n, int m, BSet st, const double *__restrict__ Dinv, const double *__restrict__ Einv, const double *__restrict__ x_ws,
            const double *__restrict__ y_ws, const BCtl *__restrict__ ctl, double *x, double *x0, double *x_prev, double *y) {
  const int b = blockIdx.x;
  const size_t on = (size_t)b * n, om = (size_t)b * m;
  if (x_ws)
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      double v = x_ws[on + i];
      if (st.scaling) v = v * Dinv[i];
      x[on + i] = v; x0[on + i] = v; x_prev[on + i] = v;
    }
  if (y_ws) {
    const double cc = ctl[b].c;
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
      double v = y_ws[om + i];
      if (st.scaling) { v = v * Einv[i]; v = v * cc; }
      y[om + i] = v;
    }
  }
}
// Qx = Qd (+ x / gamma_init), Ax = Ad, sigma = clamp(sigma_init max(1, |f|) / max(1, dist2 / 2)) with f = x'Qx / 2 + q'x and
// dist2 = |Ax - clip(Ax)|^2 (initialize_sigma, iteration.c:50-84)
__global__ void __launch_bounds__(256)
kb_warm_sigma(int n, int m, BSet st, const double *__restrict__ x, const double *__restrict__ q, const double *__restrict__ Qd,
              const double *__restrict__ Ad, const double *__restrict__ bmin, const double *__restrict__ bmax, double *Qx, double *Ax,
              double *sigma, double *sigma_inv, double *sqrt_sigma) {
  __shared__ double scratch[32];
  __shared__ double sig_s;
  const int b = blockIdx.x, tid = threadIdx.x;
  const size_t on = (size_t)b * n, om = (size_t)b * m;
  const double inv_g = 1 / st.gamma_init;
  double xqx = 0.0, qtx = 0.0, dist2 = 0.0;
  for (int i = tid; i < n; i += blockDim.x) {
    const double xi = x[on + i];
    double qx = Qd[on + i];
    if (st.proximal) qx = qx + inv_g * xi;
    Qx[on + i] = qx;
    xqx += xi * qx; qtx += q[on + i] * xi;
  }
  for (int i = tid; i < m; i += blockDim.x) {
    const double ax = Ad[om + i];
    Ax[om + i] = ax;
    const double t = ax - fmax(bmin[om + i], fmin(ax, bmax[om + i]));
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
  for (int i = tid; i < m; i += blockDim.x) { sigma[om + i] = s; sigma_inv[om + i] = 1.0 / s; sqrt_sigma[om + i] = sqrt(s); }
}

// ------------------------------------------------------------------------------------------------
// residual step (compute_residuals + candidate active set + termination reductions), one CTA per instance
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
kb_res_m(int m, int scaling, const BCtl *__restrict__ ctl, const double *__restrict__ Ax, const double *__restrict__ y,
         const double *__restrict__ sigma, const double *__restrict__ sigma_inv, const double *__restrict__ bmin,
         const double *__restrict__ bmax, const double *__restrict__ E, const double *__restrict__ Einv,
         const double *__restrict__ Ad, const int *__restrict__ active_old,
         double *Axys, double *z, double *pri_res, double *yh, int *active_cand, double *scal) {
  const int b = blockIdx.x;
  if (ctl[b].done) return;
  __shared__ double scratch[32];
  const size_t om = (size_t)b * m;
  double r_pri = 0, r_raw = 0, r_ax = 0, r_z = 0, r_edy = 0, oob = 0, adx_max = -1.0e300, adx_min = 1.0e300;
  double n_act = 0, n_ent = 0, n_lea = 0;
  for (int i = threadIdx.x; i < m; i += blockDim.x) {
    const double ax = Ax[om + i], yi = y[om + i], lo = bmin[om + i], hi = bmax[om + i];
    double t = yi * sigma_inv[om + i];
    const double axys = ax + t;
    const double zi = fmax(lo, fmin(axys, hi));
    const double pr = ax - zi;
    t = pr * sigma[om + i];
    const double yhi = yi + t;
    Axys[om + i] = axys; z[om + i] = zi; pri_res[om + i] = pr; yh[om + i] = yhi;
    const int act = (axys <= lo) || (axys >= hi);
    const int old = active_old[om + i];
    active_cand[om + i] = act;
    n_act += act; n_ent += (act && !old); n_lea += (!act && old);
    const double ei = scaling ? E[i] : 1.0, einv = scaling ? Einv[i] : 1.0;
    r_pri = fmax(r_pri, fabs(einv * pr)); r_raw = fmax(r_raw, fabs(pr));
    r_ax = fmax(r_ax, fabs(einv * ax)); r_z = fmax(r_z, fabs(einv * zi));
    const double dy = yhi - yi;
    r_edy = fmax(r_edy, fabs(ei * dy));
    const bool hi_fin = hi < ei * kInf, lo_fin = lo > -ei * kInf;
    oob += hi_fin ? hi * fmax(dy, 0.0) : 0.0;
    oob += lo_fin ? lo * fmin(dy, 0.0) : 0.0;
    const double adx = einv * Ad[om + i];
    if (hi_fin) adx_max = fmax(adx_max, adx);
    if (lo_fin) adx_min = fmin(adx_min, adx);
  }
#define RED_OUT(op, v, slot) { const double r_ = block_red<op>(v, scratch); if (threadIdx.x == 0) BSC(b, slot) = r_; }
  RED_OUT(RED_MAX, r_pri, S_PRI_RES) RED_OUT(RED_MAX, r_raw, S_PRI_RES_RAW) RED_OUT(RED_MAX, r_ax, S_NORM_AX)
  RED_OUT(RED_MAX, r_z, S_NORM_Z) RED_OUT(RED_MAX, r_edy, S_NORM_EDY) RED_OUT(RED_SUM, oob, S_OOB)
  RED_OUT(RED_MAX, adx_max, S_ADX_MAX) RED_OUT(RED_MIN, adx_min, S_ADX_MIN) RED_OUT(RED_SUM, n_act, S_NB_ACTIVE)
  RED_OUT(RED_SUM, n_ent, S_NB_ENTER) RED_OUT(RED_SUM, n_lea, S_NB_LEAVE)
}

// out[b][i] = scale_b * sum_k M[i + ld*k] v[b][k]  (row sums of a shared column-major matrix; used for A'yh and Q d)
__global__ void __launch_bounds__(256)
kb_gemv_rows(int nrows, int ncols, int ld, const double *__restrict__ M, const double *__restrict__ v, long long sv,
             double *out, long long so, const BCtl *__restrict__ ctl, const int *__restrict__ mask, int use_c) {
  const int b = blockIdx.y;
  if (ctl[b].done || (mask && !mask[b])) return;
  extern __shared__ double vs[];
  const double *vb = v + (size_t)b * sv;
  for (int k = threadIdx.x; k < ncols; k += blockDim.x) vs[k] = vb[k];
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nrows) return;
  const double *r = M + i;
  double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
  int k = 0;
  for (; k + 3 < ncols; k += 4) {
    a0 = fma(r[(size_t)k * ld], vs[k], a0);
    a1 = fma(r[(size_t)(k + 1) * ld], vs[k + 1], a1);
    a2 = fma(r[(size_t)(k + 2) * ld], vs[k + 2], a2);
    a3 = fma(r[(size_t)(k + 3) * ld], vs[k + 3], a3);
  }
  for (; k < ncols; k++) a0 = fma(r[(size_t)k * ld], vs[k], a0);
  double acc = (a0 + a1) + (a2 + a3);
  if (use_c) acc *= ctl[b].c;
  out[(size_t)b * so + i] = acc;
}
// out[b][k] = sum_i M[i + ld*k] v[b][i]   (column dots; used for A d with At as M)
__global__ void __launch_bounds__(256)
kb_gemv_cols(int len, int ncols, int ld, const double *__restrict__ M, const double *__restrict__ v, long long sv,
             double *out, long long so, const BCtl *__restrict__ ctl, const int *__restrict__ mask) {
  const int b = blockIdx.y;
  if (ctl[b].done || (mask && !mask[b])) return;
  extern __shared__ double vs[];
  const double *vb = v + (size_t)b * sv;
  for (int k = threadIdx.x; k < len; k += blockDim.x) vs[k] = vb[k];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int col = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (col >= ncols) return;
  const double *c = M + (size_t)col * ld;
  double a0 = 0, a1 = 0;
  int i = lane;
  for (; i + 32 < len; i += 64) { a0 = fma(c[i], vs[i], a0); a1 = fma(c[i + 32], vs[i + 32], a1); }
  for (; i < len; i += 32) a0 = fma(c[i], vs[i], a0);
  const double acc = warp_sum(a0 + a1);
  if (lane == 0) out[(size_t)b * so + col] = acc;
}

__global__ void __launch_bounds__(256)
kb_res_n(int n, BSet st, const BCtl *__restrict__ ctl, const double *__restrict__ Qx, const double *__restrict__ q,
         const double *__restrict__ x0, const double *__restrict__ x, const double *__restrict__ x_prev,
         const double *__restrict__ Atyh, const double *__restrict__ Aty, const double *__restrict__ D,
         const double *__restrict__ Dinv, const double *__restrict__ Qd, const double *__restrict__ d,
         double *df, double *dphi, double *scal) {
  const int b = blockIdx.x;
  if (ctl[b].done) return;
  __shared__ double scratch[32];
  const size_t on = (size_t)b * n;
  const double gamma = ctl[b].gamma, neg_inv_gamma = -1 / gamma;
  const double neg_tau_over_gamma = -BSC(b, S_TAU) * (1 / gamma);
  double r_dua = 0, r_dua2 = 0, r_qx = 0, r_q = 0, r_atyh = 0, r_atdy = 0, r_ddx = 0, dxdx = 0, dxqdx = 0, qdx = 0;
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    const double qx = Qx[on + j], qj = q[on + j], xj = x[on + j], at = Atyh[on + j];
    double dfj = qx + qj;
    if (st.proximal) dfj = dfj + neg_inv_gamma * x0[on + j];
    const double dp = dfj + at;
    df[on + j] = dfj; dphi[on + j] = dp;
    const double dinv = st.scaling ? Dinv[j] : 1.0;
    if (st.proximal) {
      const double xx0 = xj - x0[on + j];
      const double t = dp + neg_inv_gamma * xx0;
      r_dua = fmax(r_dua, fabs(dinv * t));
    } else r_dua = fmax(r_dua, fabs(dinv * dp));
    r_dua2 = fmax(r_dua2, fabs(dinv * dp));
    r_qx = fmax(r_qx, fabs(dinv * qx)); r_q = fmax(r_q, fabs(dinv * qj)); r_atyh = fmax(r_atyh, fabs(dinv * at));
    r_atdy = fmax(r_atdy, fabs(dinv * (at - Aty[on + j])));
    const double dx = xj - x_prev[on + j];
    const double ddx = st.scaling ? D[j] * dx : dx;
    r_ddx = fmax(r_ddx, fabs(ddx));
    dxdx += ddx * ddx;
    if (st.proximal) { const double t2 = Qd[on + j] + neg_tau_over_gamma * d[on + j]; dxqdx += dx * t2; }
    else dxqdx += Qd[on + j] * dx;
    qdx += qj * dx;
  }
  RED_OUT(RED_MAX, r_dua, S_DUA_RES) RED_OUT(RED_MAX, r_dua2, S_DUA2_RES) RED_OUT(RED_MAX, r_qx, S_NORM_QX)
  RED_OUT(RED_MAX, r_q, S_NORM_Q) RED_OUT(RED_MAX, r_atyh, S_NORM_ATYH) RED_OUT(RED_MAX, r_atdy, S_NORM_ATDY)
  RED_OUT(RED_MAX, r_ddx, S_NORM_DDX) RED_OUT(RED_SUM, dxdx, S_DXDX) RED_OUT(RED_SUM, dxqdx, S_DXQDX) RED_OUT(RED_SUM, qdx, S_QDX)
}

// ------------------------------------------------------------------------------------------------
// the control flow of qpalm_solve for one iteration, one thread per instance (src/qpalm.c:484-711)
// ------------------------------------------------------------------------------------------------
__global__ void kb_control(int nb, int n, int m, BSet st, BCtl *ctl, const double *__restrict__ scal, int *mask_outer,
                           int *mask_sigma, int *mask_inner, int *mask_refac, int *mask_factor, int *mask_fq, int *mask_boost) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nb) return;
  mask_outer[b] = mask_sigma[b] = mask_inner[b] = mask_refac[b] = mask_factor[b] = mask_fq[b] = mask_boost[b] = 0;
  BCtl c = ctl[b];
  if (c.done) return;
  const double *h = scal + (size_t)b * S_COUNT;
  // calculate_residuals_and_tolerances (termination.c:44-128)
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
  // check_termination (termination.c:19-42)
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
  if (term) { c.status = term; c.done = 1; ctl[b] = c; return; }
  const int na = (m > 0) ? (int)h[S_NB_ACTIVE] : 0, ne = (m > 0) ? (int)h[S_NB_ENTER] : 0, nl = (m > 0) ? (int)h[S_NB_LEAVE] : 0;
  if ((c.dua2_res_norm <= c.eps_dua_in) || (c.no_change == 3)) {   // qpalm.c:515
    c.no_change = 0;
    mask_outer[b] = 1;
    if (c.iter_out > 0 && c.pri_res_norm > c.eps_pri) mask_sigma[b] = 1;
    c.eps_abs_in = fmax(st.eps_abs, st.rho * c.eps_abs_in);
    c.eps_rel_in = fmax(st.eps_rel, st.rho * c.eps_rel_in);
    c.gamma_prev = c.gamma;
    if (st.proximal) {
      const bool try_boost = !c.gamma_maxed && c.iter_out > 0 && c.nb_enter == 0 && c.nb_leave == 0 && c.pri_res_norm < c.eps_pri;
      if (try_boost) mask_boost[b] = 1;   // decided in kb_boost after the dual update (needs the recomputed active set)
      else if (c.gamma < st.gamma_max) { c.gamma = fmin(c.gamma * st.gamma_upd, st.gamma_max); c.reset_newton = 1; }
    }
    c.iter_out++; c.prev_iter = c.iter;
  } else if (c.iter == c.prev_iter + st.inner_max_iter) {   // qpalm.c:647-660
    c.no_change = 0;
    mask_outer[b] = 2;
    if (c.iter_out > 0 && c.pri_res_norm > c.eps_pri) mask_sigma[b] = 1;
    c.gamma_prev = c.gamma;
    if (st.proximal && c.gamma < st.gamma_max) { c.gamma = fmin(c.gamma * st.gamma_upd, st.gamma_max); c.reset_newton = 1; }
    c.iter_out++; c.prev_iter = c.iter;
  } else {   // inner step
    if (c.nb_enter + c.nb_leave) c.no_change = 0; else c.no_change++;
    if ((c.iter % st.reset_newton_iter) == 0) c.reset_newton = 1;
    c.nb_active = na; c.nb_enter = ne; c.nb_leave = nl;
    mask_inner[b] = 1;
    c.beta = st.proximal ? 1.0 / c.gamma : 0.0;
    const double rank_limit = fmin(st.max_rank_update_fraction * (double)(n + m), (double)st.max_rank_update);
    c.scratch = 0;
    if ((c.reset_newton && na) || (double)(ne + nl) > rank_limit) { mask_refac[b] = 1; mask_factor[b] = 1; c.scratch = c.reset_newton || !c.H_valid; }
    else if (na) { if (ne + nl > 0) { mask_refac[b] = 1; mask_factor[b] = 1; c.scratch = !c.H_valid; } }
    else { mask_fq[b] = 1; mask_factor[b] = 1; }
    c.reset_newton = 0;
    c.n_inner++;
    if (mask_factor[b]) { c.n_refac++; c.refac_J += na; }
  }
  ctl[b] = c;
}

// update_sigma (iteration.c:86-145); in the batch every sigma change leads to a refactorisation (same matrix
// as the reference's rank update of solver_interface.c:443-503)
__global__ void __launch_bounds__(256)
kb_update_sigma(int m, BSet st, BCtl *ctl, const int *__restrict__ mask, const double *__restrict__ pri_res,
                const double *__restrict__ pri_res_in, const int *__restrict__ active, double *sigma, double *sigma_inv,
                double *sqrt_sigma, const double *__restrict__ scal) {
  const int b = blockIdx.x;
  if (!mask[b]) return;
  __shared__ double scratch[32];
  const size_t om = (size_t)b * m;
  const double nrm = BSC(b, S_PRI_RES_RAW);
  double changed = 0;
  for (int k = threadIdx.x; k < m; k += blockDim.x) {
    const double pr = fabs(pri_res[om + k]);
    if ((pr > st.theta * fabs(pri_res_in[om + k])) && active[om + k]) {
      double mult = fmax(1.0, st.delta * pr / (nrm + 1e-6));
      const double sg = sigma[om + k], stmp = mult * sg;
      if (stmp <= st.sigma_max) {
        changed += (sg != stmp);
        sigma[om + k] = stmp; sigma_inv[om + k] = 1.0 / stmp;
        mult = sqrt(mult);
        sqrt_sigma[om + k] = mult * sqrt_sigma[om + k];
      } else {
        changed += (sg != st.sigma_max);
        sigma[om + k] = st.sigma_max; sigma_inv[om + k] = 1.0 / st.sigma_max; sqrt_sigma[om + k] = st.sqrt_sigma_max;
      }
    }
  }
  changed = block_red<RED_SUM>(changed, scratch);
  if (threadIdx.x == 0) {
    if ((st.proximal && ctl[b].gamma_prev < st.gamma_max) || changed > 0) ctl[b].reset_newton = 1;
  }
}

// dual update and the rest of the outer iteration: y <- yh, Aty <- Atyh, Qx += (1/gamma - 1/gamma_prev) x,
// x0 <- x, pri_res_in <- pri_res (qpalm.c:525-526, 629, 635, 655, 658)
__global__ void __launch_bounds__(256)
kb_outer(int n, int m, BSet st, const BCtl *__restrict__ ctl, const int *__restrict__ mask, double *y, const double *__restrict__ yh,
         double *Aty, const double *__restrict__ Atyh, double *Qx, const double *__restrict__ x, double *x0, double *pri_res_in,
         const double *__restrict__ pri_res) {
  const int b = blockIdx.x;
  const int kind = mask[b];
  if (!kind) return;
  const size_t on = (size_t)b * n, om = (size_t)b * m;
  const double g = ctl[b].gamma, gp = ctl[b].gamma_prev;
  const double dg = (g != gp) ? (1 / g - 1 / gp) : 0.0;
  for (int i = threadIdx.x; i < m; i += blockDim.x) {
    if (kind == 1) y[om + i] = yh[om + i];
    pri_res_in[om + i] = pri_res[om + i];
  }
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    if (kind == 1) Aty[on + j] = Atyh[on + j];
    if (st.proximal) {
      if (dg != 0.0) Qx[on + j] = Qx[on + j] + dg * x[on + j];
      x0[on + j] = x[on + j];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// inner step: commit the active set and build the H-difference lists (ordered), one CTA per instance
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
kb_lists(int m, BCtl *ctl, const int *__restrict__ mask_inner, const int *__restrict__ mask_refac, const int *__restrict__ cand,
         int *active, const double *__restrict__ sigma, const double *__restrict__ sqrt_sigma, int *activeH, double *sigmaH,
         int *list_pos, int *list_neg, double *w_pos, double *w_neg, int *Kpos, int *Kneg, int *mask_scratch) {
  const int b = blockIdx.x;
  if (!mask_inner[b]) { if (threadIdx.x == 0) { Kpos[b] = 0; Kneg[b] = 0; mask_scratch[b] = 0; } return; }
  __shared__ int warp_cnt0[32], warp_cnt1[32];
  __shared__ int base0, base1, redo;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t om = (size_t)b * m;
  for (int i = tid; i < m; i += blockDim.x) active[om + i] = cand[om + i];
  if (!mask_refac[b]) { if (tid == 0) { Kpos[b] = 0; Kneg[b] = 0; mask_scratch[b] = 0; } return; }
  int scratch_mode = ctl[b].scratch;
  const int nb_active = ctl[b].nb_active;
  for (int attempt = 0; attempt < 2; attempt++) {
    __syncthreads();
    if (tid == 0) { base0 = 0; base1 = 0; redo = 0; }
    __syncthreads();
    for (int start = 0; start < m; start += 1024) {
      const int i = start + tid;
      bool p0 = false, p1 = false;
      double s0 = 0.0, s1 = 0.0;
      if (i < m) {
        const int a = active[om + i];
        const double wn = a ? sigma[om + i] : 0.0;
        const double wh = (scratch_mode || !activeH[om + i]) ? 0.0 : sigmaH[om + i];
        const double dw = wn - wh;
        if (dw > 0.0) { p0 = true; s0 = (wh == 0.0) ? sqrt_sigma[om + i] : sqrt(dw); }
        else if (dw < 0.0) { p1 = true; s1 = sqrt(-dw); }
      }
      const unsigned b0 = __ballot_sync(0xffffffffu, p0), b1 = __ballot_sync(0xffffffffu, p1);
      if (lane == 0) { warp_cnt0[warp] = __popc(b0); warp_cnt1[warp] = __popc(b1); }
      __syncthreads();
      int off0 = base0, off1 = base1;
      for (int w = 0; w < warp; w++) { off0 += warp_cnt0[w]; off1 += warp_cnt1[w]; }
      const unsigned lt = (1u << lane) - 1u;
      if (p0) { const int pos = off0 + __popc(b0 & lt); list_pos[om + pos] = i; w_pos[om + pos] = s0; }
      if (p1) { const int pos = off1 + __popc(b1 & lt); list_neg[om + pos] = i; w_neg[om + pos] = s1; }
      __syncthreads();
      if (tid == 0) { int t0 = 0, t1 = 0; for (int w = 0; w < 32; w++) { t0 += warp_cnt0[w]; t1 += warp_cnt1[w]; } base0 += t0; base1 += t1; }
      __syncthreads();
    }
    if (tid == 0 && !scratch_mode && base0 + base1 > nb_active) redo = 1;   // cheaper to rebuild from Q
    __syncthreads();
    if (!redo) break;
    scratch_mode = 1;
  }
  for (int i = tid; i < m; i += blockDim.x) { activeH[om + i] = active[om + i]; sigmaH[om + i] = sigma[om + i]; }
  if (tid == 0) {
    Kpos[b] = (base0 + 15) / 16 * 16; Kneg[b] = (base1 + 15) / 16 * 16;
    ctl[b].npos = base0; ctl[b].nneg = base1; ctl[b].H_valid = 1; ctl[b].scratch = scratch_mode;
    mask_scratch[b] = scratch_mode;
  }
}

// dst_b(lower) <- c_b * Qs (+ diag_add, pad identity when to_L)
__global__ void kb_init_from_Q(int n, int npad, int ld, const double *__restrict__ Qs, double *dst, long long sd,
                               const BCtl *__restrict__ ctl, const int *__restrict__ mask, int to_L) {
  const int b = blockIdx.z;
  if (!mask[b]) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
  if (i >= npad || i < j) return;
  double v;
  if (i < n && j < n) { v = Qs[(size_t)i + (size_t)j * n] * ctl[b].c; if (to_L && i == j) v += ctl[b].beta; }
  else v = (to_L && i == j) ? 1.0 : 0.0;
  dst[(size_t)b * sd + (size_t)i + (size_t)j * ld] = v;
}
__global__ void kb_copy_H_to_L(int n, int npad, int ld, const double *__restrict__ H, double *L, long long sd,
                               const BCtl *__restrict__ ctl, const int *__restrict__ mask) {
  const int b = blockIdx.z;
  if (!mask[b]) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
  if (i >= npad || i < j) return;
  double v;
  if (i < n && j < n) v = H[(size_t)b * sd + (size_t)i + (size_t)j * ld] + ((i == j) ? ctl[b].beta : 0.0);
  else v = (i == j) ? 1.0 : 0.0;
  L[(size_t)b * sd + (size_t)i + (size_t)j * ld] = v;
}
// W_b[:, c] = scale_b[c] * At[:, list_b[c]] for c < K_b (zero beyond the list)
__global__ void kb_gather(int n, int npad, int m, const double *__restrict__ At, const int *__restrict__ list,
                          const double *__restrict__ scale, const int *__restrict__ Kz, const BCtl *__restrict__ ctl, int use_neg,
                          const int *__restrict__ mask, double *W, int ldw, long long sW) {
  const int b = blockIdx.z, c = blockIdx.y;
  if (!mask[b] || c >= Kz[b]) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npad) return;
  const int cnt = use_neg ? ctl[b].nneg : ctl[b].npos;
  double v = 0.0;
  if (c < cnt && i < n) {
    const int row = list[(size_t)b * m + c];
    v = At[(size_t)i + (size_t)n * row] * scale[(size_t)b * m + c];
  }
  W[(size_t)b * sW + (size_t)i + (size_t)ldw * c] = v;
}
__global__ void kb_neg_to_pad(int n, int npad, const double *__restrict__ dphi, double *vpad, const int *__restrict__ mask) {
  const int b = blockIdx.y;
  if (!mask[b]) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < npad) vpad[(size_t)b * npad + i] = (i < n) ? dphi[(size_t)b * n + i] * -1 : 0.0;
}
__global__ void kb_commit(int n, int npad, int m, const int *__restrict__ mask, const double *__restrict__ vpad, double *d,
                          const int *__restrict__ active, int *active_old) {
  const int b = blockIdx.x;
  if (!mask[b]) return;
  for (int i = threadIdx.x; i < n; i += blockDim.x) d[(size_t)b * n + i] = vpad[(size_t)b * npad + i];
  for (int i = threadIdx.x; i < m; i += blockDim.x) active_old[(size_t)b * m + i] = active[(size_t)b * m + i];
}

// ------------------------------------------------------------------------------------------------
// line search: eta/beta dots + breakpoints, in-CTA stable radix sort, scan/select, iterate update
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
kb_ls_build(int n, int m, BSet st, const BCtl *__restrict__ ctl, const int *__restrict__ mask, const double *__restrict__ d,
            double *Qd, const double *__restrict__ df, const double *__restrict__ Ad, const double *__restrict__ Ax,
            const double *__restrict__ y, const double *__restrict__ sigma, const double *__restrict__ sqrt_sigma,
            const double *__restrict__ bmin, const double *__restrict__ bmax, unsigned long long *key, unsigned int *val,
            double *da, double *db, double *scal) {
  const int b = blockIdx.x;
  if (!mask[b]) return;
  __shared__ double scratch[32];
  const size_t on = (size_t)b * n, om = (size_t)b * m, o2 = (size_t)b * 2 * m;
  const double inv_gamma = 1 / ctl[b].gamma;
  double eta = 0, beta = 0;
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    double qd = Qd[on + j];
    const double dj = d[on + j];
    if (st.proximal) { qd = qd + inv_gamma * dj; Qd[on + j] = qd; }
    eta += dj * qd; beta += dj * df[on + j];
  }
  double a_part = 0, b_part = 0, n_l = 0;
  for (int i = threadIdx.x; i < m; i += blockDim.x) {
    const double ss = sqrt_sigma[om + i], sg = sigma[om + i], ax = Ax[om + i], yi = y[om + i];
    const double t = ss * Ad[om + i];
    double dl[2], al[2];
    dl[1] = t; dl[0] = t * -1;
    double u = ax - bmin[om + i]; u = sg * u; u = yi + u; al[0] = u / ss;
    u = bmax[om + i] - ax; u = sg * u; u = u - yi; al[1] = u / ss;
#pragma unroll
    for (int hh = 0; hh < 2; hh++) {
      const int idx = i + hh * m;
      const double s = al[hh] / dl[hh];
      const bool inL = s > 0, inP = dl[hh] > 0;
      key[o2 + idx] = inL ? (unsigned long long)__double_as_longlong(s) : ~0ull;
      val[o2 + idx] = (unsigned int)idx;
      const double d2 = dl[hh] * dl[hh], dalp = dl[hh] * al[hh];
      da[o2 + idx] = inP ? d2 : -d2;
      db[o2 + idx] = inP ? -dalp : dalp;
      if ((int)inL + (int)inP == 1) { a_part += d2; b_part += dalp; }
      n_l += inL;
    }
  }
  RED_OUT(RED_SUM, eta, S_ETA) RED_OUT(RED_SUM, beta, S_BETA) RED_OUT(RED_SUM, a_part, S_LS_A)
  RED_OUT(RED_SUM, b_part, S_LS_B) RED_OUT(RED_SUM, n_l, S_NL)
}

// stable LSD radix sort of N <= kSortMax (key, val) pairs entirely in shared memory, one CTA per instance
constexpr int kSortMax = 4096, kSortThreads = 512, kSortWarps = kSortThreads / 32;
constexpr size_t kSortSmem = (size_t)kSortMax * 2 * (8 + 4) + sizeof(unsigned) * (kSortWarps * 256 + 256 + 256) + 64;
__global__ void __launch_bounds__(kSortThreads)
kb_sort(int N, const int *__restrict__ mask, unsigned long long *key, unsigned int *val) {
  const int b = blockIdx.x;
  if (!mask[b]) return;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned long long *k0 = reinterpret_cast<unsigned long long *>(smem_raw), *k1 = k0 + kSortMax;
  unsigned int *v0 = reinterpret_cast<unsigned int *>(k1 + kSortMax), *v1 = v0 + kSortMax;
  unsigned int *warp_cnt = v1 + kSortMax;          // [kSortWarps][256]
  unsigned int *running = warp_cnt + kSortWarps * 256;   // [256]
  unsigned int *hist = running + 256;              // [256]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  unsigned long long *kg = key + (size_t)b * N;
  unsigned int *vg = val + (size_t)b * N;
  for (int i = tid; i < N; i += kSortThreads) { k0[i] = kg[i]; v0[i] = vg[i]; }
  __syncthreads();
  unsigned long long *kin = k0, *kout = k1;
  unsigned int *vin = v0, *vout = v1;
  for (int pass = 0; pass < 8; pass++) {
    const int shift = pass * 8;
    if (tid < 256) hist[tid] = 0;
    __syncthreads();
    for (int i = tid; i < N; i += kSortThreads) atomicAdd(&hist[(unsigned)(kin[i] >> shift) & 255u], 1u);
    __syncthreads();
    if (hist[(unsigned)(kin[0] >> shift) & 255u] == (unsigned)N) { __syncthreads(); continue; }   // all keys share this digit
    if (warp == 0) {   // exclusive scan of the 256 bins by one warp (8 bins per lane)
      unsigned int loc[8], sum = 0;
#pragma unroll
      for (int t = 0; t < 8; t++) { loc[t] = hist[lane * 8 + t]; sum += loc[t]; }
      unsigned int inc = sum;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const unsigned int u = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += u; }
      unsigned int run = inc - sum;
#pragma unroll
      for (int t = 0; t < 8; t++) { running[lane * 8 + t] = run; run += loc[t]; }
    }
    __syncthreads();
    for (int start = 0; start < N; start += kSortThreads) {
      for (int i = tid; i < kSortWarps * 256; i += kSortThreads) warp_cnt[i] = 0;
      __syncthreads();
      const int e = start + tid;
      const bool valid = e < N;
      unsigned long long k = 0; unsigned int v = 0; unsigned int dg = 0x10000u + lane;
      if (valid) { k = kin[e]; v = vin[e]; dg = (unsigned)(k >> shift) & 255u; }
      const unsigned peers = __match_any_sync(0xffffffffu, dg);
      const int rank = __popc(peers & ((1u << lane) - 1u));
      if (valid && rank == 0) warp_cnt[warp * 256 + dg] = __popc(peers);
      __syncthreads();
      if (valid) {
        unsigned int off = running[dg];
        for (int w = 0; w < warp; w++) off += warp_cnt[w * 256 + dg];
        kout[off + rank] = k; vout[off + rank] = v;
      }
      __syncthreads();
      if (tid < 256) {
        unsigned int t = 0;
#pragma unroll
        for (int w = 0; w < kSortWarps; w++) t += warp_cnt[w * 256 + tid];
        running[tid] += t;
      }
      __syncthreads();
    }
    unsigned long long *tk = kin; kin = kout; kout = tk;
    unsigned int *tv = vin; vin = vout; vout = tv;
  }
  __syncthreads();
  for (int i = tid; i < N; i += kSortThreads) { kg[i] = kin[i]; vg[i] = vin[i]; }
}

__global__ void __launch_bounds__(1024)
kb_ls_select(int m, const int *__restrict__ mask, const unsigned long long *__restrict__ key, const unsigned int *__restrict__ val,
             const double *__restrict__ da, const double *__restrict__ db, double *scal) {
  const int b = blockIdx.x;
  if (!mask[b]) return;
  __shared__ double wa[32], wb[32];
  __shared__ double carry_a, carry_b;
  __shared__ int found;
  const size_t o2 = (size_t)b * 2 * m;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nL = (int)BSC(b, S_NL);
  if (tid == 0) { carry_a = BSC(b, S_ETA) + BSC(b, S_LS_A); carry_b = BSC(b, S_BETA) - BSC(b, S_LS_B); found = 0x7fffffff; }
  __syncthreads();
  for (int start = 0; start < nL; start += 1024) {
    const int i = start + tid;
    double ta = 0.0, tb = 0.0, s = 0.0;
    if (i < nL) { const unsigned int idx = val[o2 + i]; ta = da[o2 + idx]; tb = db[o2 + idx]; s = __longlong_as_double((long long)key[o2 + i]); }
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
      if (i == found) BSC(b, S_TAU) = -b_i / a_i;
      return;
    }
    if (tid == 1023) { carry_a += oa + ia; carry_b += ob + ib; }
    __syncthreads();
  }
  if (tid == 0) BSC(b, S_TAU) = -carry_b / carry_a;
}

__global__ void __launch_bounds__(256)
kb_update_iterate(int n, int m, const int *__restrict__ mask, const double *__restrict__ scal, double *x, double *x_prev,
                  const double *__restrict__ d, double *Qd, double *Qx, double *Ad, double *Ax) {
  const int b = blockIdx.x;
  if (!mask[b]) return;
  const double tau = BSC(b, S_TAU);
  const size_t on = (size_t)b * n, om = (size_t)b * m;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double xi = x[on + i];
    x_prev[on + i] = xi; x[on + i] = xi + tau * d[on + i];
    const double qd = Qd[on + i] * tau;
    Qd[on + i] = qd; Qx[on + i] = Qx[on + i] + qd;
  }
  for (int i = threadIdx.x; i < m; i += blockDim.x) {
    const double ad = Ad[om + i] * tau;
    Ad[om + i] = ad; Ax[om + i] = Ax[om + i] + ad;
  }
}

__global__ void kb_end_iter(int nb, int max_iter, BCtl *ctl, int *ndone) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nb) return;
  if (!ctl[b].done) {
    ctl[b].iter++;
    if (ctl[b].iter >= max_iter) { ctl[b].status = QPALM_MAX_ITER_REACHED; ctl[b].done = 1; }
  }
  if (ctl[b].done) atomicAdd(ndone, 1);
}

// store_solution (termination.c:242-252) + compute_objective (iteration.c:231-270)
__global__ void __launch_bounds__(256)
kb_store(int n, int m, BSet st, BCtl *ctl, const double *__restrict__ D, const double *__restrict__ E, const double *__restrict__ x,
         const double *__restrict__ yh, const double *__restrict__ Qx, const double *__restrict__ q, double *x_out, double *y_out) {
  const int b = blockIdx.x;
  __shared__ double scratch[32];
  const size_t on = (size_t)b * n, om = (size_t)b * m;
  const double cinv = ctl[b].cinv, inv_gamma = 1 / ctl[b].gamma;
  double obj = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double xi = x[on + i];
    x_out[on + i] = st.scaling ? xi * D[i] : xi;
    if (st.proximal) obj += (0.5 * (Qx[on + i] - inv_gamma * xi) + q[on + i]) * xi;
    else obj += (0.5 * Qx[on + i] + q[on + i]) * xi;
  }
  for (int i = threadIdx.x; i < m; i += blockDim.x) {
    double v = yh[om + i];
    if (st.scaling) { v *= cinv; v = v * E[i]; }
    y_out[om + i] = v;
  }
  obj = block_red<RED_SUM>(obj, scratch);
  if (threadIdx.x == 0) { if (st.scaling) obj *= cinv; ctl[b].objective = obj + st.data_c; }
}

// boost_gamma path of the outer update (qpalm.c:613-627, iteration.c:159-211) for the flagged instances:
// recompute the active set from Axys = Ax + y./sigma; unchanged => gamma <- max(gamma_max, 1e14 / gershgorin(A_J' S A_J)),
// else update_gamma.  The Gershgorin bound is formed from the instance's H record when it is current, otherwise from a
// fresh assembly in the L scratch (the factor is rebuilt afterwards anyway: reset_newton).
__global__ void __launch_bounds__(256)
kb_boost_active(int m, BSet st, BCtl *ctl, int *mask_boost, const double *__restrict__ Ax, const double *__restrict__ y,
                const double *__restrict__ sigma, const double *__restrict__ bmin, const double *__restrict__ bmax,
                const int *__restrict__ old, double *Axys, int *active) {
  const int b = blockIdx.x;
  if (!mask_boost[b]) return;
  __shared__ double scratch[32];
  const size_t om = (size_t)b * m;
  double na = 0, ne = 0, nl = 0;
  for (int i = threadIdx.x; i < m; i += blockDim.x) {
    const double t = y[om + i] / sigma[om + i];
    const double a = Ax[om + i] + t;
    Axys[om + i] = a;
    const int act = (a <= bmin[om + i]) || (a >= bmax[om + i]);
    active[om + i] = act;
    na += act; ne += act && !old[om + i]; nl += !act && old[om + i];
  }
  na = block_red<RED_SUM>(na, scratch); ne = block_red<RED_SUM>(ne, scratch); nl = block_red<RED_SUM>(nl, scratch);
  if (threadIdx.x == 0) {
    BCtl &c = ctl[b];
    c.nb_active = (int)na; c.nb_enter = (int)ne; c.nb_leave = (int)nl; c.boost = 0;
    if (ne == 0 && nl == 0) {
      c.boost = 1;
      if (na == 0) {   // no active constraints: gamma = 1e12 (iteration.c:198-200)
        c.gamma = 1e12; c.reset_newton = 1; mask_boost[b] = 0;
      } else { c.scratch = 1; c.npos = 0; c.nneg = 0; }   // Gershgorin needed: stays flagged
    } else {
      if (c.gamma < st.gamma_max) { c.gamma = fmin(c.gamma * st.gamma_upd, st.gamma_max); c.reset_newton = 1; }
      mask_boost[b] = 0;
    }
  }
}
__global__ void __launch_bounds__(1024)
kb_boost_list(int m, BCtl *ctl, const int *__restrict__ mask, const int *__restrict__ active, const double *__restrict__ sqrt_sigma,
              int *list_pos, double *w_pos, int *Kpos) {
  const int b = blockIdx.x;
  if (!mask[b]) { if (threadIdx.x == 0) Kpos[b] = 0; return; }
  __shared__ int warp_cnt[32];
  __shared__ int base;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t om = (size_t)b * m;
  if (tid == 0) base = 0;
  __syncthreads();
  for (int start = 0; start < m; start += 1024) {
    const int i = start + tid;
    const bool p = (i < m) && active[om + i];
    const unsigned bl = __ballot_sync(0xffffffffu, p);
    if (lane == 0) warp_cnt[warp] = __popc(bl);
    __syncthreads();
    int off = base;
    for (int w = 0; w < warp; w++) off += warp_cnt[w];
    if (p) { const int pos = off + __popc(bl & ((1u << lane) - 1u)); list_pos[om + pos] = i; w_pos[om + pos] = sqrt_sigma[om + i]; }
    __syncthreads();
    if (tid == 0) { int t = 0; for (int w = 0; w < 32; w++) t += warp_cnt[w]; base += t; }
    __syncthreads();
  }
  if (tid == 0) { Kpos[b] = (base + 15) / 16 * 16; ctl[b].npos = base; }
}
__global__ void kb_zero_lower(int npad, int ld, double *L, long long sd, const int *__restrict__ mask) {
  const int b = blockIdx.z;
  if (!mask[b]) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
  if (i >= npad || i < j) return;
  L[(size_t)b * sd + (size_t)i + (size_t)j * ld] = 0.0;
}
__global__ void __launch_bounds__(256)
kb_boost_gersh(int n, int ld, BSet st, BCtl *ctl, const int *__restrict__ mask, const double *__restrict__ L, long long sd) {
  const int b = blockIdx.x;
  if (!mask[b]) return;
  __shared__ double scratch[32];
  const double *M = L + (size_t)b * sd;
  double ub = -1.0e300;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {   // thread per row: |row i| of the symmetric matrix
    double acc = 0.0;
    for (int j = 0; j <= i; j++) acc += fabs(M[(size_t)i + (size_t)j * ld]);
    for (int j = i + 1; j < n; j++) acc += fabs(M[(size_t)j + (size_t)i * ld]);
    ub = fmax(ub, acc);
  }
  ub = block_red<RED_MAX>(ub, scratch);
  if (threadIdx.x == 0) {
    BCtl &c = ctl[b];
    c.gamma = fmax(st.gamma_max, 1e14 / ub);
    c.gamma_maxed = 1;
    c.reset_newton = 1;
  }
}
// after the boost decision: apply the Qx / Qd shifts for a changed gamma (iteration.c:205-209) and x0 <- x
__global__ void __launch_bounds__(256)
kb_boost_apply(int n, BCtl *ctl, const int *__restrict__ mask_was_boost, double *Qx, const double *__restrict__ x, double *Qd,
               const double *__restrict__ d, const double *__restrict__ scal) {
  const int b = blockIdx.x;
  if (!mask_was_boost[b]) return;
  const double g = ctl[b].gamma, gp = ctl[b].gamma_prev;
  if (g == gp) return;
  const size_t on = (size_t)b * n;
  const double tau = BSC(b, S_TAU);
  const int boosted = ctl[b].boost;   // the Qd shift belongs to boost_gamma only (iteration.c:207), not to update_gamma
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    Qx[on + j] = Qx[on + j] + (1.0 / g - 1.0 / gp) * x[on + j];
    if (boosted) Qd[on + j] = Qd[on + j] + (tau / g - tau / gp) * d[on + j];
  }
  if (threadIdx.x == 0) ctl[b].reset_newton = 1;
}
__global__ void kb_copy_mask(int nb, const int *src, int *dst) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < nb) dst[b] = src[b];
}

// out (cols x rows, column-major) = in' for in rows x cols column-major
__global__ void kb_transpose(int rows, int cols, const double *__restrict__ in, double *__restrict__ out) {
  __shared__ double tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int k = threadIdx.y; k < 32; k += 8) {
    const int r = r0 + threadIdx.x, c = c0 + k;
    tile[k][threadIdx.x] = (r < rows && c < cols) ? in[(size_t)r + (size_t)rows * c] : 0.0;
  }
  __syncthreads();
  for (int k = threadIdx.y; k < 32; k += 8) {
    const int c = c0 + threadIdx.x, r = r0 + k;
    if (r < rows && c < cols) out[(size_t)c + (size_t)cols * r] = tile[threadIdx.x][k];
  }
}

}  // namespace

// ==================================================================================================
// host side
// ==================================================================================================
extern "C" QPALMB200Batch *qpalm_b200_batch_setup(const QPALMData *shared, const QPALMSettings *s, c_int nb_max_) {
  if (!shared || !s || nb_max_ <= 0) return nullptr;
  if (!validate_settings(s)) return nullptr;
  if (s->nonconvex || s->enable_dual_termination) {
    fprintf(stderr, "[qpalm_b200] batch: nonconvex / dual-termination settings are not supported by the batch entry point\n");
    return nullptr;
  }
  const int n = (int)shared->n, m = (int)shared->m, nb_max = (int)nb_max_;
  if (2 * m > kSortMax) {
    fprintf(stderr, "[qpalm_b200] batch: 2m = %d exceeds the in-CTA line-search sort capacity (%d)\n", 2 * m, kSortMax);
    return nullptr;
  }
  if (shard_world() > 1) {
    fprintf(stderr, "[qpalm_b200] batch: instances shard by index across ranks (qpalm_b200/shard.py); do not combine with row-sharding\n");
    return nullptr;
  }
  QPALMB200Batch *B = new QPALMB200Batch();
  B->nb_max = nb_max; B->n = n; B->m = m; B->m2 = 2 * m;
  std::vector<double> zn((size_t)n + 1, 0.0), zm((size_t)m + 1, 0.0);
  if (engine_create(&B->shared, n, m, (const long long *)shared->A->p, (const long long *)shared->A->i, (const double *)shared->A->x,
                    (const long long *)shared->Q->p, (const long long *)shared->Q->i, (const double *)shared->Q->x,
                    zn.data(), zm.data(), zm.data(), false)) { delete B; return nullptr; }
  Engine *e = B->shared;
  B->stream = e->stream; B->npad = e->npad; B->ld = e->ld;
  if ((m > 0 && !e->A_dense) || !e->Q_dense) {
    fprintf(stderr, "[qpalm_b200] batch: the batch entry point needs dense shared Q and A (density >= 25%%)\n");
    engine_destroy(e); delete B; return nullptr;
  }
  BSet &st = B->set;
  st.max_iter = (int)s->max_iter; st.inner_max_iter = (int)s->inner_max_iter; st.proximal = (int)s->proximal; st.scaling = s->scaling > 0;
  st.reset_newton_iter = (int)s->reset_newton_iter; st.max_rank_update = (int)s->max_rank_update;
  st.eps_abs = s->eps_abs; st.eps_rel = s->eps_rel; st.eps_abs_in = s->eps_abs_in; st.eps_rel_in = s->eps_rel_in; st.rho = s->rho;
  st.eps_prim_inf = s->eps_prim_inf; st.eps_dual_inf = s->eps_dual_inf; st.theta = s->theta; st.delta = s->delta;
  st.sigma_max = s->sigma_max; st.sigma_init = s->sigma_init; st.gamma_init = s->gamma_init; st.gamma_upd = s->gamma_upd;
  st.gamma_max = s->gamma_max; st.max_rank_update_fraction = s->max_rank_update_fraction; st.sqrt_sigma_max = sqrt(s->sigma_max);
  st.data_c = shared->c;
  { const char *u = getenv("QPALM_B200_BATCH_UPDOWN"); st.batch_updown = u ? atoi(u) : 1; }
  { const char *u = getenv("QPALM_B200_BATCH_UPDOWN_MAX_RANK"); st.batch_updown_max_rank = u ? atoi(u) : 40; }
  { const char *u = getenv("QPALM_B200_BATCH_HINC"); st.batch_h_incremental = u ? atoi(u) : 0; }
  if (s->scaling) {   // Ruiz on the shared matrices; the cost scaling c is per instance (applied on the fly)
    double cc;
    if (engine_ruiz_scale(e, (int)s->scaling, &cc)) { engine_destroy(e); delete B; return nullptr; }
    // engine_ruiz_scale applied c = 1/max(1,|D*0|) = 1 to Q, so e->Qd now holds D Q D
  }
  B->Qs = e->Qd;
  if (m > 0) {   // second layout of the scaled A for the row-parallel A d of the persistent engine
    if (dev_alloc((void **)&B->Am, sizeof(double) * (size_t)m * n)) { engine_destroy(e); delete B; return nullptr; }
    QB_LAUNCH(kb_transpose, dim3(cdiv(m, 32), cdiv(n, 32)), dim3(32, 8), 0, e->stream, n, m, e->At, B->Am);
  }
  const size_t N = n, M = m, NB = nb_max, LL = (size_t)B->ld * B->npad;
  B->wcols = round_up(m > 16 ? m : 16, 16);
  int rc = 0;
  auto dv = [&](double **p, size_t len) { return dev_alloc((void **)p, sizeof(double) * (len ? len : 1)); };
  auto iv = [&](int **p, size_t len) { return dev_alloc((void **)p, sizeof(int) * (len ? len : 1)); };
  rc |= dv(&B->q_raw, NB * N); rc |= dv(&B->bmin_raw, NB * M); rc |= dv(&B->bmax_raw, NB * M); rc |= dv(&B->x_out, NB * N); rc |= dv(&B->y_out, NB * M);
  rc |= dv(&B->q, NB * N); rc |= dv(&B->bmin, NB * M); rc |= dv(&B->bmax, NB * M); rc |= dv(&B->x, NB * N); rc |= dv(&B->y, NB * M);
  rc |= dv(&B->Ax, NB * M); rc |= dv(&B->Qx, NB * N); rc |= dv(&B->Aty, NB * N); rc |= dv(&B->x_prev, NB * N); rc |= dv(&B->x0, NB * N);
  rc |= dv(&B->sigma, NB * M); rc |= dv(&B->sigma_inv, NB * M); rc |= dv(&B->sqrt_sigma, NB * M); rc |= dv(&B->Axys, NB * M); rc |= dv(&B->z, NB * M);
  rc |= dv(&B->pri_res, NB * M); rc |= dv(&B->pri_res_in, NB * M); rc |= dv(&B->yh, NB * M); rc |= dv(&B->Atyh, NB * N); rc |= dv(&B->df, NB * N);
  rc |= dv(&B->dphi, NB * N); rc |= dv(&B->d, NB * N); rc |= dv(&B->Qd, NB * N); rc |= dv(&B->Ad, NB * M); rc |= dv(&B->vpad, NB * B->npad);
  rc |= iv(&B->active, NB * M); rc |= iv(&B->active_old, NB * M); rc |= iv(&B->active_cand, NB * M); rc |= iv(&B->activeH, NB * M);
  rc |= iv(&B->list_pos, NB * M); rc |= iv(&B->list_neg, NB * M); rc |= dv(&B->sigmaH, NB * M); rc |= dv(&B->w_pos, NB * M); rc |= dv(&B->w_neg, NB * M);
  rc |= iv(&B->Kpos, NB); rc |= iv(&B->Kneg, NB);
  rc |= dv(&B->H, NB * LL); rc |= dv(&B->L, NB * LL); rc |= dv(&B->invdiag, NB * (size_t)B->npad * kPanel);
  rc |= dv(&B->W, NB * (size_t)B->ld * B->wcols);
  rc |= dev_alloc((void **)&B->keys, sizeof(unsigned long long) * NB * (2 * M + 1)); rc |= dev_alloc((void **)&B->vals, sizeof(unsigned int) * NB * (2 * M + 1));
  rc |= dv(&B->ls_da, NB * 2 * M); rc |= dv(&B->ls_db, NB * 2 * M);
  rc |= dv(&B->scal, NB * S_COUNT);
  rc |= dev_alloc((void **)&B->ctl, sizeof(BCtl) * NB);
  for (int **p : {&B->mask_outer, &B->mask_sigma, &B->mask_inner, &B->mask_refac, &B->mask_factor, &B->mask_scratch, &B->mask_fq, &B->mask_boost, &B->info})
    rc |= iv(p, NB);
  rc |= iv(&B->ndone, 4);
  rc |= iv(&B->queue, 4);
  rc |= dv(&B->x_ws, NB * N); rc |= dv(&B->y_ws, NB * M);
  if (getenv("QPALM_B200_BATCH_PROF")) rc |= dev_alloc((void **)&B->prof, sizeof(long long) * 32 * NB);
  if (const char *env = getenv("QPALM_B200_BATCH_ENGINE")) {   // tests / profiling: force one engine
    if (!strcmp(env, "lockstep")) B->engine = 1; else if (!strcmp(env, "persistent")) B->engine = 2;
  }
  if (rc) { fprintf(stderr, "[qpalm_b200] batch: device allocation failed\n"); qpalm_b200_batch_cleanup(B); return nullptr; }
  cudaMallocHost((void **)&B->ndone_host, sizeof(int) * 4);
  B->ctl_host.resize(NB);
  cudaEventCreate(&B->ev0); cudaEventCreate(&B->ev1);
  cudaFuncSetAttribute(kb_sort, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSortSmem);
  cudaDeviceSynchronize();
  return B;
}

extern "C" int qpalm_b200_batch_upload(QPALMB200Batch *B, c_int nb_, const c_float *q, const c_float *bmin, const c_float *bmax) {
  const int nb = (int)nb_;
  if (!B || nb <= 0 || nb > B->nb_max) return 1;
  QB_CUDA_TRY(cudaMemcpyAsync(B->q_raw, q, sizeof(double) * (size_t)nb * B->n, cudaMemcpyHostToDevice, B->stream));
  QB_CUDA_TRY(cudaMemcpyAsync(B->bmin_raw, bmin, sizeof(double) * (size_t)nb * B->m, cudaMemcpyHostToDevice, B->stream));
  QB_CUDA_TRY(cudaMemcpyAsync(B->bmax_raw, bmax, sizeof(double) * (size_t)nb * B->m, cudaMemcpyHostToDevice, B->stream));
  QB_CUDA_TRY(cudaStreamSynchronize(B->stream));
  return 0;
}

extern "C" int qpalm_b200_batch_warm_start(QPALMB200Batch *B, c_int nb_, const c_float *x_ws, const c_float *y_ws) {
  if (!B) return 1;
  if (!x_ws && !y_ws) { B->ws_nb = 0; B->ws_x = 0; B->ws_y = 0; return 0; }
  const int nb = (int)nb_;
  if (nb <= 0 || nb > B->nb_max) return 1;
  B->ws_nb = 0; B->ws_x = 0; B->ws_y = 0;   // the buffers are being overwritten: no half-copied warm start stays pending
  if (x_ws) QB_CUDA_TRY(cudaMemcpyAsync(B->x_ws, x_ws, sizeof(double) * (size_t)nb * B->n, cudaMemcpyHostToDevice, B->stream));
  if (y_ws && B->m > 0) QB_CUDA_TRY(cudaMemcpyAsync(B->y_ws, y_ws, sizeof(double) * (size_t)nb * B->m, cudaMemcpyHostToDevice, B->stream));
  QB_CUDA_TRY(cudaStreamSynchronize(B->stream));
  B->ws_nb = nb; B->ws_x = x_ws != nullptr; B->ws_y = y_ws != nullptr;
  return 0;
}

extern "C" int qpalm_b200_batch_solve_resident(QPALMB200Batch *B, c_int nb_, double *device_ms) {
  const int nb = (int)nb_;
  if (!B || nb <= 0 || nb > B->nb_max) return 1;
  Engine *e = B->shared;
  cudaStream_t s = B->stream;
  const int n = B->n, m = B->m, npad = B->npad, ld = B->ld;
  const BSet st = B->set;
  const long long sLL = (long long)ld * npad, sX = (long long)npad * kPanel, sW = (long long)ld * B->wcols;
  const long long launches0 = g_kernel_launches;
  const int gnb = cdiv(nb, 128);
  // a pending warm start is consumed by this solve (qpalm_solve resets `initialized` the same way)
  const int nwarm = B->ws_nb < nb ? B->ws_nb : nb, wx = B->ws_x, wy = B->ws_y;
  B->ws_nb = 0; B->ws_x = 0; B->ws_y = 0;
  // engine choice: the persistent one-CTA-per-instance kernel (batchp.cu) when the shapes fit its shared-memory plan,
  // else the lock-step engine below
  const bool persistent = (B->engine == 2) || (B->engine == 0 && batchp_supported(n, m));
  if (persistent) {
    if (!batchp_supported(n, m)) { fprintf(stderr, "[qpalm_b200] batch: shapes n=%d m=%d do not fit the persistent engine\n", n, m); return 1; }
    QB_CUDA_TRY(cudaEventRecord(B->ev0, s));
    // shape choice (batchp.cu header): the 4-CTA/SM build only when it turns two waves into one
    static int num_sms = 0;
    if (!num_sms) { int dev = 0; QB_CUDA_TRY(cudaGetDevice(&dev)); QB_CUDA_TRY(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev)); }
    static const char *shape_env = getenv("QPALM_B200_BATCH_SHAPE");   // "3" / "4" force a shape (A/B measurements)
    bool four = nb > 3 * num_sms && nb <= 4 * num_sms;
    if (shape_env && shape_env[0] == '3') four = false;
    if (shape_env && shape_env[0] == '4') four = true;
    if (four && !batchp4_supported(n, m)) four = false;
    if (int r = four ? batchp4_solve(B, nb, nwarm, wx, wy) : batchp_solve(B, nb, nwarm, wx, wy)) return r;
    QB_CUDA_TRY(cudaEventRecord(B->ev1, s));
    QB_CUDA_TRY(cudaEventSynchronize(B->ev1));
    float msp = 0; cudaEventElapsedTime(&msp, B->ev0, B->ev1);
    if (device_ms) *device_ms = msp;
    B->launches_last = g_kernel_launches - launches0;
    B->last_engine = 2;
    B->last_shape = four ? 4 : 3;
    QB_CUDA_TRY(cudaGetLastError());
    return 0;
  }
  B->last_engine = 1;
  B->last_shape = 0;
  QB_CUDA_TRY(cudaEventRecord(B->ev0, s));
  QB_LAUNCH(kb_init, nb, 256, 0, s, n, m, st, e->D, e->E, B->q_raw, B->bmin_raw, B->bmax_raw, B->q, B->bmin, B->bmax, B->x, B->y, B->Ax,
            B->Qx, B->Aty, B->x_prev, B->x0, B->sigma, B->sigma_inv, B->sqrt_sigma, B->Qd, B->Ad, B->d, B->pri_res_in, B->active,
            B->active_old, B->activeH, B->scal, B->ctl);
  if (nwarm && (wx || wy)) {
    QB_LAUNCH(kb_warm_set, nwarm, 256, 0, s, n, m, st, e->Dinv, e->Einv, wx ? B->x_ws : nullptr, wy ? B->y_ws : nullptr, B->ctl,
              B->x, B->x0, B->x_prev, B->y);
    if (wx) {
      QB_LAUNCH(kb_gemv_rows, dim3(cdiv(n, 256), nwarm), 256, sizeof(double) * n, s, n, n, n, B->Qs, B->x, (long long)n, B->Qd,
                (long long)n, B->ctl, (const int *)nullptr, 1);
      if (m > 0) QB_LAUNCH(kb_gemv_cols, dim3(cdiv(m, 8), nwarm), 256, sizeof(double) * n, s, n, m, n, e->At, B->x, (long long)n, B->Ad,
                           (long long)m, B->ctl, (const int *)nullptr);
      QB_LAUNCH(kb_warm_sigma, nwarm, 256, 0, s, n, m, st, B->x, B->q, B->Qd, B->Ad, B->bmin, B->bmax, B->Qx, B->Ax, B->sigma,
                B->sigma_inv, B->sqrt_sigma);
    }
  }
  const dim3 tri_grid(cdiv(npad, 256), npad, nb);
  for (int it = 0; it <= st.max_iter; it++) {
    // ---- residuals + termination scalars ----
    if (m > 0) QB_LAUNCH(kb_res_m, nb, 256, 0, s, m, st.scaling, B->ctl, B->Ax, B->y, B->sigma, B->sigma_inv, B->bmin, B->bmax, e->E, e->Einv,
                         B->Ad, B->active_old, B->Axys, B->z, B->pri_res, B->yh, B->active_cand, B->scal);
    if (m > 0) QB_LAUNCH(kb_gemv_rows, dim3(cdiv(n, 256), nb), 256, sizeof(double) * m, s, n, m, n, e->At, B->yh, (long long)m, B->Atyh,
                         (long long)n, B->ctl, (const int *)nullptr, 0);
    QB_LAUNCH(kb_res_n, nb, 256, 0, s, n, st, B->ctl, B->Qx, B->q, B->x0, B->x, B->x_prev, B->Atyh, B->Aty, e->D, e->Dinv, B->Qd, B->d,
              B->df, B->dphi, B->scal);
    QB_LAUNCH(kb_control, gnb, 128, 0, s, nb, n, m, st, B->ctl, B->scal, B->mask_outer, B->mask_sigma, B->mask_inner, B->mask_refac,
              B->mask_factor, B->mask_fq, B->mask_boost);
    // ---- outer updates ----
    if (m > 0) QB_LAUNCH(kb_update_sigma, nb, 256, 0, s, m, st, B->ctl, B->mask_sigma, B->pri_res, B->pri_res_in, B->active, B->sigma,
                         B->sigma_inv, B->sqrt_sigma, B->scal);
    QB_LAUNCH(kb_outer, nb, 256, 0, s, n, m, st, B->ctl, B->mask_outer, B->y, B->yh, B->Aty, B->Atyh, B->Qx, B->x, B->x0, B->pri_res_in, B->pri_res);
    if (st.proximal && m > 0) {   // boost_gamma candidates (rare): mask_sigma is reused as "was a boost candidate"
      QB_LAUNCH(kb_copy_mask, gnb, 128, 0, s, nb, B->mask_boost, B->mask_sigma);
      QB_LAUNCH(kb_boost_active, nb, 256, 0, s, m, st, B->ctl, B->mask_boost, B->Ax, B->y, B->sigma, B->bmin, B->bmax, B->active_old, B->Axys, B->active);
      QB_LAUNCH(kb_boost_list, nb, 1024, 0, s, m, B->ctl, B->mask_boost, B->active, B->sqrt_sigma, B->list_pos, B->w_pos, B->Kpos);
      QB_LAUNCH(kb_zero_lower, tri_grid, 256, 0, s, npad, ld, B->L, sLL, B->mask_boost);
      QB_LAUNCH(kb_gather, dim3(cdiv(npad, 256), B->wcols, nb), 256, 0, s, n, npad, m, e->At, B->list_pos, B->w_pos, B->Kpos, B->ctl, 0,
                B->mask_boost, B->W, ld, sW);
      if (int r = dgemm_nt_batched(s, nb, npad, npad, B->wcols, B->Kpos, B->W, ld, sW, B->W, ld, sW, B->L, ld, sLL, 1.0, 1.0, true, B->mask_boost)) return r;
      QB_LAUNCH(kb_boost_gersh, nb, 256, 0, s, n, ld, st, B->ctl, B->mask_boost, B->L, sLL);
      QB_LAUNCH(kb_boost_apply, nb, 256, 0, s, n, B->ctl, B->mask_sigma, B->Qx, B->x, B->Qd, B->d, B->scal);
    }
    // ---- inner step: Newton system ----
    if (m > 0) {
      QB_LAUNCH(kb_lists, nb, 1024, 0, s, m, B->ctl, B->mask_inner, B->mask_refac, B->active_cand, B->active, B->sigma, B->sqrt_sigma,
                B->activeH, B->sigmaH, B->list_pos, B->list_neg, B->w_pos, B->w_neg, B->Kpos, B->Kneg, B->mask_scratch);
      QB_LAUNCH(kb_init_from_Q, tri_grid, 256, 0, s, n, npad, ld, B->Qs, B->H, sLL, B->ctl, B->mask_scratch, 0);
      QB_LAUNCH(kb_gather, dim3(cdiv(npad, 256), B->wcols, nb), 256, 0, s, n, npad, m, e->At, B->list_pos, B->w_pos, B->Kpos, B->ctl, 0,
                B->mask_refac, B->W, ld, sW);
      if (int r = dgemm_nt_batched(s, nb, npad, npad, B->wcols, B->Kpos, B->W, ld, sW, B->W, ld, sW, B->H, ld, sLL, 1.0, 1.0, true, B->mask_refac)) return r;
      QB_LAUNCH(kb_gather, dim3(cdiv(npad, 256), B->wcols, nb), 256, 0, s, n, npad, m, e->At, B->list_neg, B->w_neg, B->Kneg, B->ctl, 1,
                B->mask_refac, B->W, ld, sW);
      if (int r = dgemm_nt_batched(s, nb, npad, npad, B->wcols, B->Kneg, B->W, ld, sW, B->W, ld, sW, B->H, ld, sLL, -1.0, 1.0, true, B->mask_refac)) return r;
      QB_LAUNCH(kb_copy_H_to_L, tri_grid, 256, 0, s, n, npad, ld, B->H, B->L, sLL, B->ctl, B->mask_refac);
    }
    QB_LAUNCH(kb_init_from_Q, tri_grid, 256, 0, s, n, npad, ld, B->Qs, B->L, sLL, B->ctl, B->mask_fq, 1);
    if (int r = potrf_lower_batched(s, nb, npad, B->L, ld, sLL, B->invdiag, sX, B->info, B->mask_factor)) return r;
    QB_LAUNCH(kb_neg_to_pad, dim3(cdiv(npad, 256), nb), 256, 0, s, n, npad, B->dphi, B->vpad, B->mask_inner);
    if (int r = chol_solve_batched(s, nb, npad, B->L, ld, sLL, B->invdiag, sX, B->vpad, (long long)npad, B->mask_inner)) return r;
    QB_LAUNCH(kb_commit, nb, 256, 0, s, n, npad, m, B->mask_inner, B->vpad, B->d, B->active, B->active_old);
    // ---- line search + iterate update ----
    QB_LAUNCH(kb_gemv_rows, dim3(cdiv(n, 256), nb), 256, sizeof(double) * n, s, n, n, n, B->Qs, B->d, (long long)n, B->Qd, (long long)n,
              B->ctl, B->mask_inner, 1);
    if (m > 0) {
      QB_LAUNCH(kb_gemv_cols, dim3(cdiv(m, 8), nb), 256, sizeof(double) * n, s, n, m, n, e->At, B->d, (long long)n, B->Ad, (long long)m,
                B->ctl, B->mask_inner);
    }
    QB_LAUNCH(kb_ls_build, nb, 256, 0, s, n, m, st, B->ctl, B->mask_inner, B->d, B->Qd, B->df, B->Ad, B->Ax, B->y, B->sigma, B->sqrt_sigma,
              B->bmin, B->bmax, B->keys, B->vals, B->ls_da, B->ls_db, B->scal);
    if (m > 0) QB_LAUNCH(kb_sort, nb, kSortThreads, kSortSmem, s, 2 * m, B->mask_inner, B->keys, B->vals);
    QB_LAUNCH(kb_ls_select, nb, 1024, 0, s, m, B->mask_inner, B->keys, B->vals, B->ls_da, B->ls_db, B->scal);
    QB_LAUNCH(kb_update_iterate, nb, 256, 0, s, n, m, B->mask_inner, B->scal, B->x, B->x_prev, B->d, B->Qd, B->Qx, B->Ad, B->Ax);
    QB_CUDA_TRY(cudaMemsetAsync(B->ndone, 0, sizeof(int), s));
    QB_LAUNCH(kb_end_iter, gnb, 128, 0, s, nb, st.max_iter, B->ctl, B->ndone);
    QB_CUDA_TRY(cudaMemcpyAsync(B->ndone_host, B->ndone, sizeof(int), cudaMemcpyDeviceToHost, s));
    QB_CUDA_TRY(cudaStreamSynchronize(s));
    if (B->ndone_host[0] >= nb) break;
  }
  QB_LAUNCH(kb_store, nb, 256, 0, s, n, m, st, B->ctl, e->D, e->E, B->x, B->yh, B->Qx, B->q, B->x_out, B->y_out);
  QB_CUDA_TRY(cudaEventRecord(B->ev1, s));
  QB_CUDA_TRY(cudaEventSynchronize(B->ev1));
  float ms = 0; cudaEventElapsedTime(&ms, B->ev0, B->ev1);
  if (device_ms) *device_ms = ms;
  B->launches_last = g_kernel_launches - launches0;
  QB_CUDA_TRY(cudaGetLastError());
  return 0;
}

extern "C" int qpalm_b200_batch_download(QPALMB200Batch *B, c_int nb_, c_float *x, c_float *y, QPALMInfo *info) {
  const int nb = (int)nb_;
  if (!B || nb <= 0 || nb > B->nb_max) return 1;
  QB_CUDA_TRY(cudaMemcpyAsync(x, B->x_out, sizeof(double) * (size_t)nb * B->n, cudaMemcpyDeviceToHost, B->stream));
  if (B->m > 0) QB_CUDA_TRY(cudaMemcpyAsync(y, B->y_out, sizeof(double) * (size_t)nb * B->m, cudaMemcpyDeviceToHost, B->stream));
  QB_CUDA_TRY(cudaMemcpyAsync(B->ctl_host.data(), B->ctl, sizeof(BCtl) * (size_t)nb, cudaMemcpyDeviceToHost, B->stream));
  QB_CUDA_TRY(cudaStreamSynchronize(B->stream));
  for (int b = 0; b < nb && info; b++) {
    const BCtl &c = B->ctl_host[b];
    memset(&info[b], 0, sizeof(QPALMInfo));
    update_status(&info[b], c.status);
    info[b].iter = c.iter; info[b].iter_out = c.iter_out;
    info[b].pri_res_norm = c.pri_res_norm; info[b].dua_res_norm = c.dua_res_norm; info[b].dua2_res_norm = c.dua2_res_norm;
    info[b].objective = c.objective; info[b].dual_objective = 0;
  }
  return 0;
}

extern "C" int qpalm_b200_batch_solve(QPALMB200Batch *B, c_int nb, const c_float *q, const c_float *bmin, const c_float *bmax,
                                      c_float *x, c_float *y, QPALMInfo *info) {
  if (int r = qpalm_b200_batch_upload(B, nb, q, bmin, bmax)) return r;
  double ms = 0;
  if (int r = qpalm_b200_batch_solve_resident(B, nb, &ms)) return r;
  if (int r = qpalm_b200_batch_download(B, nb, x, y, info)) return r;
  if (info) for (c_int b = 0; b < nb; b++) info[b].solve_time = ms * 1e-3;
  return 0;
}

// totals over the instances of the last download: [0] inner iterations, [1] outer iterations, [2] refactorisations,
// [3] sum of |J| over them, [4] engine used (1 lock-step, 2 persistent)
extern "C" int qpalm_b200_batch_stats(QPALMB200Batch *B, c_int nb, double *out8) {
  if (!B || nb <= 0 || nb > B->nb_max) return 1;
  QB_CUDA_TRY(cudaMemcpy(B->ctl_host.data(), B->ctl, sizeof(BCtl) * (size_t)nb, cudaMemcpyDeviceToHost));
  double a = 0, o = 0, r = 0, j = 0, u = 0, ur = 0, uf = 0;
  for (c_int b = 0; b < nb; b++) {
    const BCtl &c = B->ctl_host[b];
    a += c.n_inner; o += c.iter_out; r += c.n_refac; j += (double)c.refac_J; u += c.n_updown; ur += (double)c.updown_ranks; uf += c.n_updown_fail;
  }
  out8[0] = a; out8[1] = o; out8[2] = r; out8[3] = j; out8[4] = B->last_engine; out8[5] = u; out8[6] = ur; out8[7] = uf;
  return 0;
}

// persistent engine, totals over the instances of the last solve: [0] rows of A streamed through the H SYRK (summed over the
// refactorisations), [1] refactorisations that rebuilt H from c Q
extern "C" int qpalm_b200_batch_syrk_stats(QPALMB200Batch *B, c_int nb, double *out2) {
  if (!B || nb <= 0 || nb > B->nb_max) return 1;
  QB_CUDA_TRY(cudaMemcpy(B->ctl_host.data(), B->ctl, sizeof(BCtl) * (size_t)nb, cudaMemcpyDeviceToHost));
  double e = 0, r = 0;
  for (c_int b = 0; b < nb; b++) { e += (double)B->ctl_host[b].syrk_entries; r += B->ctl_host[b].n_scratch; }
  out2[0] = e; out2[1] = r;
  return 0;
}

extern "C" int qpalm_b200_batch_phase_profile(QPALMB200Batch *B, c_int nb, long long *out /* nb x 16 */) {
  if (!B || !B->prof) return 1;
  QB_CUDA_TRY(cudaMemcpy(out, B->prof, sizeof(long long) * 32 * (size_t)nb, cudaMemcpyDeviceToHost));
  return 0;
}

extern "C" long long qpalm_b200_batch_last_launches(const QPALMB200Batch *B) { return B ? B->launches_last : 0; }

extern "C" int qpalm_b200_batch_last_shape(const QPALMB200Batch *B) { return B ? B->last_shape : 0; }

// ------------------------------------------------------------------------------------------------
// test probes of the persistent engine's in-CTA building blocks (batchp.cu kbp_probe_*): host buffers in and out, like the
// operator ABI of Part 2.  shape picks the build: 3 the default one, 4 the -DQB_BP_VARIANT4 one.
// ------------------------------------------------------------------------------------------------
namespace {
struct ProbeBufs {   // device buffers of one probe call, freed on every return path
  std::vector<void *> p;
  bool failed = false;
  template <typename T> T *get(size_t count) {
    void *q = nullptr;
    if (dev_alloc(&q, sizeof(T) * (count ? count : 1))) { failed = true; return nullptr; }
    p.push_back(q);
    return static_cast<T *>(q);
  }
  ~ProbeBufs() { for (void *q : p) cudaFree(q); }
};
}  // namespace

static int probe_newton(c_int shape, c_int nb_, c_int n_, c_int m_, const c_float *At, const c_float *H0, c_int from_q, c_float sscale,
                        const c_int *cnt, const c_int *lists, const c_float *wts, c_float beta, const c_float *rhs, c_float *H_out,
                        c_float *L_out, c_float *d_fused, c_float *d_after, c_int *info, c_int rounds, c_float *d_rounds) {
  if ((shape != 3 && shape != 4) || nb_ < 1 || n_ < 1 || m_ < 1 || rounds < 0) return 1;
  const int nb = (int)nb_, n = (int)n_, m = (int)m_, ld = round_up(n, kPanel);
  const size_t NB = nb, N = n, M = m, LL = (size_t)ld * ld;
  std::vector<int> cnt_i(NB * 4), lists_i(NB * 3 * M, 0);
  for (size_t b = 0; b < NB; b++) {
    const c_int *c = cnt + 4 * b;
    if (c[0] < 0 || c[0] > m || c[1] < 0 || c[1] > m || c[2] < 0 || c[2] > m || c[3] < 0 || c[3] > c[2]) return 1;
    if (c[0] + c[1] > m) return 1;   // one SYRK stream holds both lists: at most m rows, as in the solver
    for (int k = 0; k < 4; k++) cnt_i[4 * b + k] = (int)c[k];
    for (int seg = 0; seg < 3; seg++)
      for (c_int q = 0; q < c[seg]; q++) {
        const size_t at = (b * 3 + seg) * M + q;
        if (lists[at] < 0 || lists[at] >= m) return 1;
        lists_i[at] = (int)lists[at];
      }
  }
  ProbeBufs d;
  BpProbeArgs P;
  memset(&P, 0, sizeof(P));
  P.nb = nb; P.n = n; P.m = m; P.ld = ld; P.from_q = from_q != 0; P.sscale = sscale; P.beta = beta;
  double *dAt = d.get<double>(N * M), *dH0 = d.get<double>(from_q ? N * N : NB * N * N), *dw = d.get<double>(NB * 3 * M);
  double *drhs = d.get<double>(NB * N);
  int *dcnt = d.get<int>(NB * 4), *dl = d.get<int>(NB * 3 * M);
  P.H = d.get<double>(NB * LL); P.L = d.get<double>(NB * LL); P.rdiag = d.get<double>(NB * ld);
  P.d_fused = d.get<double>(NB * N); P.d_after = d.get<double>(NB * N);
  P.rounds = (int)rounds; P.d_rounds = d.get<double>(NB * 2 * (size_t)rounds * N + 1);
  P.info = d.get<int>(NB); P.queue = d.get<int>(1);
  if (d.failed) return 2;
  P.At = dAt; P.H0 = dH0; P.wts = dw; P.rhs = drhs; P.cnt = dcnt; P.lists = dl;
  const cudaStream_t s = 0;
  QB_CUDA_TRY(cudaMemcpyAsync(dAt, At, sizeof(double) * N * M, cudaMemcpyHostToDevice, s));
  QB_CUDA_TRY(cudaMemcpyAsync(dH0, H0, sizeof(double) * (from_q ? N * N : NB * N * N), cudaMemcpyHostToDevice, s));
  QB_CUDA_TRY(cudaMemcpyAsync(dw, wts, sizeof(double) * NB * 3 * M, cudaMemcpyHostToDevice, s));
  QB_CUDA_TRY(cudaMemcpyAsync(drhs, rhs, sizeof(double) * NB * N, cudaMemcpyHostToDevice, s));
  QB_CUDA_TRY(cudaMemcpyAsync(dcnt, cnt_i.data(), sizeof(int) * NB * 4, cudaMemcpyHostToDevice, s));
  QB_CUDA_TRY(cudaMemcpyAsync(dl, lists_i.data(), sizeof(int) * NB * 3 * M, cudaMemcpyHostToDevice, s));
  if (int r = shape == 4 ? batchp4_probe_newton(P, s) : batchp_probe_newton(P, s)) return r;
  std::vector<double> hH(NB * LL), hL(NB * LL);
  std::vector<int> hinfo(NB);
  QB_CUDA_TRY(cudaMemcpyAsync(hH.data(), P.H, sizeof(double) * NB * LL, cudaMemcpyDeviceToHost, s));
  QB_CUDA_TRY(cudaMemcpyAsync(hL.data(), P.L, sizeof(double) * NB * LL, cudaMemcpyDeviceToHost, s));
  QB_CUDA_TRY(cudaMemcpyAsync(d_fused, P.d_fused, sizeof(double) * NB * N, cudaMemcpyDeviceToHost, s));
  QB_CUDA_TRY(cudaMemcpyAsync(d_after, P.d_after, sizeof(double) * NB * N, cudaMemcpyDeviceToHost, s));
  QB_CUDA_TRY(cudaMemcpyAsync(hinfo.data(), P.info, sizeof(int) * NB, cudaMemcpyDeviceToHost, s));
  if (rounds) QB_CUDA_TRY(cudaMemcpyAsync(d_rounds, P.d_rounds, sizeof(double) * NB * 2 * (size_t)rounds * N, cudaMemcpyDeviceToHost, s));
  QB_CUDA_TRY(cudaStreamSynchronize(s));
  for (size_t b = 0; b < NB; b++) {   // lower triangles, n x n column-major
    info[b] = hinfo[b];
    for (size_t j = 0; j < N; j++)
      for (size_t i = 0; i < N; i++) {
        H_out[b * N * N + i + N * j] = (i >= j) ? hH[b * LL + i + ld * j] : 0.0;
        L_out[b * N * N + i + N * j] = (i >= j) ? hL[b * LL + i + ld * j] : 0.0;
      }
  }
  return 0;
}

extern "C" int qpalm_b200_batchp_probe_newton(c_int shape, c_int nb, c_int n, c_int m, const c_float *At, const c_float *H0, c_int from_q,
                                              c_float sscale, const c_int *cnt, const c_int *lists, const c_float *wts, c_float beta,
                                              const c_float *rhs, c_float *H_out, c_float *L_out, c_float *d_fused, c_float *d_after,
                                              c_int *info) {
  return probe_newton(shape, nb, n, m, At, H0, from_q, sscale, cnt, lists, wts, beta, rhs, H_out, L_out, d_fused, d_after, info, 0, nullptr);
}

extern "C" int qpalm_b200_batchp_probe_solves(c_int shape, c_int nb, c_int n, c_int m, const c_float *At, const c_float *H0, c_int from_q,
                                              c_float sscale, const c_int *cnt, const c_int *lists, const c_float *wts, c_float beta,
                                              const c_float *rhs, c_float *H_out, c_float *L_out, c_float *d_fused, c_float *d_after,
                                              c_int *info, c_int rounds, c_float *d_rounds) {
  return probe_newton(shape, nb, n, m, At, H0, from_q, sscale, cnt, lists, wts, beta, rhs, H_out, L_out, d_fused, d_after, info, rounds,
                      d_rounds);
}

extern "C" int qpalm_b200_batchp_probe_sort(c_int shape, c_int nb_, c_int N_, unsigned long long *keys, unsigned int *vals) {
  if ((shape != 3 && shape != 4) || nb_ < 1 || N_ < 1) return 1;
  const int nb = (int)nb_, N = (int)N_;
  const size_t T = (size_t)nb * N;
  ProbeBufs d;
  unsigned long long *dk = d.get<unsigned long long>(T);
  unsigned int *dv = d.get<unsigned int>(T);
  int *dq = d.get<int>(1);
  if (d.failed) return 2;
  const cudaStream_t s = 0;
  QB_CUDA_TRY(cudaMemcpyAsync(dk, keys, sizeof(unsigned long long) * T, cudaMemcpyHostToDevice, s));
  QB_CUDA_TRY(cudaMemcpyAsync(dv, vals, sizeof(unsigned int) * T, cudaMemcpyHostToDevice, s));
  if (int r = shape == 4 ? batchp4_probe_sort(nb, N, dk, dv, dq, s) : batchp_probe_sort(nb, N, dk, dv, dq, s)) return r;
  QB_CUDA_TRY(cudaMemcpyAsync(keys, dk, sizeof(unsigned long long) * T, cudaMemcpyDeviceToHost, s));
  QB_CUDA_TRY(cudaMemcpyAsync(vals, dv, sizeof(unsigned int) * T, cudaMemcpyDeviceToHost, s));
  QB_CUDA_TRY(cudaStreamSynchronize(s));
  return 0;
}

extern "C" void qpalm_b200_batch_cleanup(QPALMB200Batch *B) {
  if (!B) return;
  void *ptrs[] = {B->q_raw, B->bmin_raw, B->bmax_raw, B->x_out, B->y_out, B->q, B->bmin, B->bmax, B->x, B->y, B->Ax, B->Qx, B->Aty, B->x_prev,
                  B->x0, B->sigma, B->sigma_inv, B->sqrt_sigma, B->Axys, B->z, B->pri_res, B->pri_res_in, B->yh, B->Atyh, B->df, B->dphi, B->d,
                  B->Qd, B->Ad, B->vpad, B->active, B->active_old, B->active_cand, B->activeH, B->list_pos, B->list_neg, B->sigmaH, B->w_pos,
                  B->w_neg, B->Kpos, B->Kneg, B->H, B->L, B->invdiag, B->W, B->keys, B->vals, B->ls_da, B->ls_db, B->scal, B->ctl,
                  B->mask_outer, B->mask_sigma, B->mask_inner, B->mask_refac, B->mask_factor, B->mask_scratch, B->mask_fq, B->mask_boost,
                  B->ndone, B->info, B->queue, B->prof, B->Am, B->x_ws, B->y_ws};
  for (void *p : ptrs) if (p) cudaFree(p);
  if (B->ndone_host) cudaFreeHost(B->ndone_host);
  if (B->ev0) cudaEventDestroy(B->ev0);
  if (B->ev1) cudaEventDestroy(B->ev1);
  if (B->shared) engine_destroy(B->shared);
  delete B;
}
