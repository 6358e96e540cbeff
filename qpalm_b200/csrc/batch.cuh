// batch.cuh -- state shared by the two batch engines (batch.cu: lock-step, one launch per step over all instances;
// batchp.cu: persistent, one CTA per instance for the whole solve).
#pragma once
#include "../../include/qpalm_b200.h"
#include "engine.cuh"
#include <vector>

namespace qb {
constexpr double kInf = 1e20;

struct BCtl {   // per-instance control state (device resident)
  int iter, iter_out, prev_iter, no_change, reset_newton, gamma_maxed, done, status;
  int nb_enter, nb_leave, nb_active, H_valid, scratch, npos, nneg, boost;
  double gamma, gamma_prev, eps_abs_in, eps_rel_in, c, cinv, pri_res_norm, dua_res_norm, dua2_res_norm;
  double eps_pri, eps_dua, eps_dua_in, objective, beta;
  int n_inner, n_refac;          // executed inner steps / Newton refactorisations (roofline byte model, SURVEY 8(d))
  long long refac_J;             // sum of |J| over the refactorisations
  int n_updown, n_updown_fail;   // rank-k update / downdate sweeps taken instead of a refactorisation (and downdates that lost definiteness)
  long long updown_ranks;        // sum of ranks over the sweeps
  long long syrk_entries;        // persistent engine: rows of A streamed through the H SYRK, summed over the refactorisations
  int n_scratch;                 // persistent engine: refactorisations that rebuilt H from c Q
};

struct BSet {   // settings the device needs (copied by value into kernels)
  int max_iter, inner_max_iter, proximal, scaling, reset_newton_iter, max_rank_update;
  double eps_abs, eps_rel, eps_abs_in, eps_rel_in, rho, eps_prim_inf, eps_dual_inf, theta, delta, sigma_max, sigma_init;
  double gamma_init, gamma_upd, gamma_max, max_rank_update_fraction, sqrt_sigma_max, data_c;
  int batch_updown;              // persistent engine: take rank updates where the reference does (QPALM_B200_BATCH_UPDOWN=0 disables)
  int batch_updown_max_rank;     // persistent engine: beyond this many changed rows an (incremental) refactorisation is cheaper than the
                                 // sweeps (same matrix either way; QPALM_B200_BATCH_UPDOWN_MAX_RANK)
  int batch_h_incremental;       // persistent engine: after reset_newton keep the H record and apply only the changed rows / sigmas
                                 // (QPALM_B200_BATCH_HINC=1; default 0 = rebuild H from Q as the reference's ldlcholQAtsigmaA does)
};
}  // namespace qb

struct QPALMB200Batch {
  int nb_max = 0, n = 0, m = 0, npad = 0, ld = 0, wcols = 0, m2 = 0;
  cudaStream_t stream = nullptr;
  qb::BSet set{};
  qb::Engine *shared = nullptr;   // holds the shared, Ruiz-scaled At / Q (dense) and D, E
  double *Am = nullptr;       // A as m x n column-major (second layout of the shared scaled A, persistent engine)
  double *Qs = nullptr;       // n x n dense full symmetric D Q D (copy of shared->Qd before the c scaling)
  // per-instance arrays [nb][len]
  double *q_raw = nullptr, *bmin_raw = nullptr, *bmax_raw = nullptr, *x_out = nullptr, *y_out = nullptr;
  double *q = nullptr, *bmin = nullptr, *bmax = nullptr, *x = nullptr, *y = nullptr, *Ax = nullptr, *Qx = nullptr, *Aty = nullptr;
  double *x_prev = nullptr, *x0 = nullptr, *sigma = nullptr, *sigma_inv = nullptr, *sqrt_sigma = nullptr, *Axys = nullptr, *z = nullptr;
  double *pri_res = nullptr, *pri_res_in = nullptr, *yh = nullptr, *Atyh = nullptr, *df = nullptr, *dphi = nullptr, *d = nullptr;
  double *Qd = nullptr, *Ad = nullptr, *vpad = nullptr, *tmp_n = nullptr;
  int *active = nullptr, *active_old = nullptr, *active_cand = nullptr, *activeH = nullptr, *list_pos = nullptr, *list_neg = nullptr;
  double *sigmaH = nullptr, *w_pos = nullptr, *w_neg = nullptr;
  int *Kpos = nullptr, *Kneg = nullptr;
  double *H = nullptr, *L = nullptr, *invdiag = nullptr, *W = nullptr;
  unsigned long long *keys = nullptr; unsigned int *vals = nullptr; double *ls_da = nullptr, *ls_db = nullptr;
  double *scal = nullptr;
  qb::BCtl *ctl = nullptr;
  int *mask_outer = nullptr, *mask_sigma = nullptr, *mask_inner = nullptr, *mask_refac = nullptr, *mask_factor = nullptr,
      *mask_scratch = nullptr, *mask_fq = nullptr, *mask_boost = nullptr, *ndone = nullptr, *info = nullptr;
  int *ndone_host = nullptr;
  QPALMInfo *info_host = nullptr;
  std::vector<qb::BCtl> ctl_host;
  long long launches_last = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  int *queue = nullptr;        // persistent engine: work-queue counter
  int engine = 0;              // 0 auto, 1 lock-step, 2 persistent (QPALM_B200_BATCH_ENGINE)
  int last_engine = 0;
  int last_shape = 0;          // CTA shape of the last solve: 0 lock-step, 3 or 4 persistent (CTAs per SM)
  long long *prof = nullptr;   // persistent engine: optional per-phase clock totals [nb][16]
  // pending warm start of the next solve (qpalm_b200_batch_warm_start): unscaled rows [nb_max][n] / [nb_max][m]; instances
  // b < ws_nb start from them, the part whose flag is 0 starts cold
  double *x_ws = nullptr, *y_ws = nullptr;
  int ws_nb = 0, ws_x = 0, ws_y = 0;
};

namespace qb {
// persistent engine (batchp.cu): true when the shapes fit its shared-memory plan
bool batchp_supported(int n, int m);
// nwarm: instances b < nwarm start from B->x_ws (when wx) / B->y_ws (when wy), the others cold
int batchp_solve(QPALMB200Batch *B, int nb, int nwarm, int wx, int wy);
// the same engine compiled in its 4-CTAs-per-SM shape (batchp.cu with -DQB_BP_VARIANT4)
bool batchp4_supported(int n, int m);
int batchp4_solve(QPALMB200Batch *B, int nb, int nwarm, int wx, int wy);

// test probes of the persistent engine's in-CTA building blocks (device pointers; qpalm_b200_batchp_probe_* in batch.cu).
// Per instance b: H0 is n x n (lds = n) at H0 + b n n, copied into H before the SYRK updates it in place; or with from_q the one
// shared matrix H0 scaled by sscale, the base of the SYRK (the solver's rebuild from c Q), and without SYRK lists the matrix the
// Cholesky factors directly (the solver's f.fq path); cnt[4 b ..] = {npos, nneg, nup, kpos}, npos + nneg <= m; lists / wts hold
// 3 m entries per instance: SYRK + rows at [0, m), SYRK - rows at [m, 2 m), update rows at [2 m, 3 m).  H, L: ld x ld per instance, rdiag: ld per instance.  rounds > 0: then 2 rounds more solves per instance into
// d_rounds (nb x 2 rounds x n), see qpalm_b200_batchp_probe_solves.
struct BpProbeArgs {
  int nb, n, m, ld, from_q, rounds;
  double sscale, beta;
  const double *At, *H0, *wts, *rhs;
  const int *cnt, *lists;
  double *H, *L, *rdiag, *d_fused, *d_after, *d_rounds;
  int *info, *queue;
};
int batchp_probe_newton(const BpProbeArgs &P, cudaStream_t s);
int batchp4_probe_newton(const BpProbeArgs &P, cudaStream_t s);
int batchp_probe_sort(int nb, int N, unsigned long long *keys, unsigned int *vals, int *queue, cudaStream_t s);
int batchp4_probe_sort(int nb, int N, unsigned long long *keys, unsigned int *vals, int *queue, cudaStream_t s);
}  // namespace qb
