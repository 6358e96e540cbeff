// ops.cu -- operator-level C ABI (include/qpalm_b200.h Part 2): host buffers in, host buffers out, each
// call runs the same device kernels the solver uses.  These are the entry points the parity tests drive
// "at identical iterates" against the oracle and the reference.
#include "../../include/qpalm_b200.h"
#include "engine.cuh"
#include "sparse_host.h"
#include <math.h>
#include <string.h>
#include <vector>
#include <string>

using namespace qb;

extern "C" int qpalm_b200_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}
extern "C" const char *qpalm_b200_version(void) { return "qpalm_b200 0.1 (sm_100a)"; }

namespace {
struct EmptyCSC {
  std::vector<long long> p, i; std::vector<double> x;
  explicit EmptyCSC(size_t ncol) : p(ncol + 1, 0), i(1, 0), x(1, 0.0) {}
};
// engine from optional A (m x n) and optional Q (n x n); missing pieces are empty
int make_engine(Engine **e, int n, int m, const solver_sparse *A, const solver_sparse *Q, bool need_LQ = false, int newton_override = 0) {
  EmptyCSC ea((size_t)n), eq((size_t)n);
  std::vector<double> zn((size_t)n + 1, 0.0), zm((size_t)m + 1, 0.0);
  const long long *Ap = A ? (const long long *)A->p : ea.p.data(), *Ai = A ? (const long long *)A->i : ea.i.data();
  const double *Ax = A ? (const double *)A->x : ea.x.data();
  const long long *Qp = Q ? (const long long *)Q->p : eq.p.data(), *Qi = Q ? (const long long *)Q->i : eq.i.data();
  const double *Qx = Q ? (const double *)Q->x : eq.x.data();
  return engine_create(e, n, m, Ap, Ai, Ax, Qp, Qi, Qx, zn.data(), zm.data(), zm.data(), need_LQ, newton_override);
}
int up_int(Engine *e, int *dst, const c_int *src, int len) {
  std::vector<int> t((size_t)len + 1);
  for (int i = 0; i < len; i++) t[i] = (int)src[i];
  QB_CUDA_TRY(cudaMemcpy(dst, t.data(), sizeof(int) * (size_t)len, cudaMemcpyHostToDevice));
  (void)e;
  return 0;
}
}  // namespace

extern "C" int qpalm_b200_mat_vec(const solver_sparse *A, const c_float *x, c_float *y) {
  Engine *e = nullptr;
  const int nrow = (int)A->nrow, ncol = (int)A->ncol;
  int rc;
  if (A->stype != 0) {   // symmetric: only the lower triangle is read (stype -1)
    if ((rc = make_engine(&e, ncol, 0, nullptr, A))) return rc;
    upload(e, e->x, x, ncol); spmv_Q(e, e->x, e->Qx); rc = download(e, y, e->Qx, ncol);
  } else {
    if ((rc = make_engine(&e, ncol, nrow, A, nullptr))) return rc;
    upload(e, e->x, x, ncol); spmv_A(e, e->x, e->Ax); rc = download(e, y, e->Ax, nrow);
  }
  engine_destroy(e);
  return rc;
}
extern "C" int qpalm_b200_mat_tpose_vec(const solver_sparse *A, const c_float *x, c_float *y) {
  if (A->stype != 0) return qpalm_b200_mat_vec(A, x, y);
  Engine *e = nullptr;
  const int nrow = (int)A->nrow, ncol = (int)A->ncol;
  int rc;
  if ((rc = make_engine(&e, ncol, nrow, A, nullptr))) return rc;
  upload(e, e->y, x, nrow); spmv_At(e, e->y, e->Aty); rc = download(e, y, e->Aty, ncol);
  engine_destroy(e);
  return rc;
}

namespace qb { int ruiz_norms_public(Engine *e, double *colnorm_dev, double *rownorm_dev); }

extern "C" int qpalm_b200_scale_data(solver_sparse *A, solver_sparse *Q, c_float *q, c_float *bmin, c_float *bmax,
                                     c_int scaling_iters, c_float *D, c_float *E, c_float *c_out) {
  const int n = (int)Q->ncol, m = (int)A->nrow;
  Engine *e = nullptr;
  int rc;
  if ((rc = make_engine(&e, n, m, A, Q))) return rc;
  upload(e, e->q, q, n); upload(e, e->bmin, bmin, m); upload(e, e->bmax, bmax, m);
  double cc = 1.0;
  rc = engine_ruiz_scale(e, (int)scaling_iters, &cc);
  *c_out = cc;
  rc |= download(e, D, e->D, n); rc |= download(e, E, e->E, m);
  rc |= download(e, q, e->q, n); rc |= download(e, bmin, e->bmin, m); rc |= download(e, bmax, e->bmax, m);
  // scaled matrix values back into the caller's CSC arrays
  const long long *Ap = (const long long *)A->p, *Ai = (const long long *)A->i; double *Axv = (double *)A->x;
  if (m > 0) {
    if (e->A_dense) {
      std::vector<double> At((size_t)n * m);
      rc |= download(e, At.data(), e->At, n * m);
      for (int j = 0; j < n; j++) for (long long k = Ap[j]; k < Ap[j + 1]; k++) Axv[k] = At[(size_t)j + (size_t)n * Ai[k]];
    } else rc |= download(e, Axv, e->A_csc.x, (int)Ap[n]);
  }
  const long long *Qp = (const long long *)Q->p, *Qi = (const long long *)Q->i; double *Qxv = (double *)Q->x;
  if (e->Q_dense) {
    std::vector<double> Qd((size_t)n * n);
    rc |= download(e, Qd.data(), e->Qd, n * n);
    for (int j = 0; j < n; j++) for (long long k = Qp[j]; k < Qp[j + 1]; k++) if (Qi[k] >= j) Qxv[k] = Qd[(size_t)Qi[k] + (size_t)n * j];
  } else {
    std::vector<int> rp((size_t)n + 1);
    std::vector<double> rx((size_t)e->Q_csr.nnz + 1);
    QB_CUDA_TRY(cudaMemcpy(rp.data(), e->Q_csr.p, sizeof(int) * ((size_t)n + 1), cudaMemcpyDeviceToHost));
    rc |= download(e, rx.data(), e->Q_csr.x, (int)e->Q_csr.nnz);
    std::vector<int> fill(rp.begin(), rp.end());
    for (int j = 0; j < n; j++) for (long long k = Qp[j]; k < Qp[j + 1]; k++) { const long long i = Qi[k]; if (i < j) continue; Qxv[k] = rx[fill[i]++]; }
  }
  engine_destroy(e);
  return rc;
}

extern "C" int qpalm_b200_mat_inf_norm_cols(const solver_sparse *M, c_float *E) {
  Engine *e = nullptr; int rc;
  if ((rc = make_engine(&e, (int)M->ncol, (int)M->nrow, M, nullptr))) return rc;
  rc = ruiz_norms_public(e, e->tmp_n, e->tmp_m);
  rc |= download(e, E, e->tmp_n, (int)M->ncol);
  engine_destroy(e);
  return rc;
}
extern "C" int qpalm_b200_mat_inf_norm_rows(const solver_sparse *M, c_float *E) {
  Engine *e = nullptr; int rc;
  if ((rc = make_engine(&e, (int)M->ncol, (int)M->nrow, M, nullptr))) return rc;
  rc = ruiz_norms_public(e, e->tmp_n, e->tmp_m);
  rc |= download(e, E, e->tmp_m, (int)M->nrow);
  engine_destroy(e);
  return rc;
}

extern "C" int qpalm_b200_residuals_active_set(const solver_sparse *A,
        const c_float *Ax, const c_float *y, const c_float *sigma, const c_float *bmin, const c_float *bmax,
        const c_float *Qx, const c_float *q, const c_float *x0, c_int proximal, c_float gamma,
        const c_int *active_old,
        c_float *Axys, c_float *z, c_float *pri_res, c_float *yh, c_float *Atyh, c_float *df, c_float *dphi,
        c_int *active, c_int *nb_active, c_int *enter, c_int *nb_enter, c_int *leave, c_int *nb_leave) {
  const int m = (int)A->nrow, n = (int)A->ncol;
  Engine *e = nullptr; int rc;
  if ((rc = make_engine(&e, n, m, A, nullptr))) return rc;
  std::vector<double> sinv((size_t)m + 1);
  for (int i = 0; i < m; i++) sinv[i] = 1.0 / sigma[i];
  upload(e, e->Ax, Ax, m); upload(e, e->y, y, m); upload(e, e->sigma, sigma, m); upload(e, e->sigma_inv, sinv.data(), m);
  upload(e, e->bmin, bmin, m); upload(e, e->bmax, bmax, m); upload(e, e->Qx, Qx, n); upload(e, e->q, q, n); upload(e, e->x0, x0, n);
  cudaStreamSynchronize(e->stream);
  up_int(e, e->active_old, active_old, m);
  e->scaling = 0;
  rc = step_residuals(e, proximal != 0, gamma, 0.0);
  rc |= step_compact_lists(e);
  rc |= sync_scalars(e);
  *nb_active = (c_int)e->scal_host[S_NB_ACTIVE]; *nb_enter = (c_int)e->scal_host[S_NB_ENTER]; *nb_leave = (c_int)e->scal_host[S_NB_LEAVE];
  rc |= download(e, Axys, e->Axys, m); rc |= download(e, z, e->z, m); rc |= download(e, pri_res, e->pri_res, m);
  rc |= download(e, yh, e->yh, m); rc |= download(e, Atyh, e->Atyh, n); rc |= download(e, df, e->df, n); rc |= download(e, dphi, e->dphi, n);
  rc |= download_int(e, (long long *)active, e->active, m);
  rc |= download_int(e, (long long *)enter, e->enter, (int)*nb_enter);
  rc |= download_int(e, (long long *)leave, e->leave, (int)*nb_leave);
  engine_destroy(e);
  return rc;
}

extern "C" int qpalm_b200_linesearch(c_int m_, c_float eta, c_float beta,
        const c_float *Ad, const c_float *Ax, const c_float *y, const c_float *sigma,
        const c_float *sqrt_sigma, const c_float *bmin, const c_float *bmax,
        c_float *tau, c_float *sorted_s, c_int *sorted_idx, c_int *nL) {
  const int m = (int)m_;
  Engine *e = nullptr; int rc;
  if ((rc = make_engine(&e, 1, m, nullptr, nullptr))) return rc;
  upload(e, e->Ad, Ad, m); upload(e, e->Ax, Ax, m); upload(e, e->y, y, m); upload(e, e->sigma, sigma, m);
  upload(e, e->sqrt_sigma, sqrt_sigma, m); upload(e, e->bmin, bmin, m); upload(e, e->bmax, bmax, m);
  double eb[2] = {eta, beta};
  QB_CUDA_TRY(cudaMemcpyAsync(e->scal_dev + S_ETA, eb, sizeof(double) * 2, cudaMemcpyHostToDevice, e->stream));
  rc = linesearch_device(e, m, e->Ad, e->Ax, e->y, e->sigma, e->sqrt_sigma, e->bmin, e->bmax);
  rc |= sync_scalars(e);
  *tau = e->scal_host[S_TAU];
  const int n_l = (int)e->scal_host[S_NL];
  if (nL) *nL = n_l;
  if (sorted_s && sorted_idx && n_l > 0) {
    std::vector<unsigned long long> k((size_t)n_l); std::vector<unsigned int> v((size_t)n_l);
    QB_CUDA_TRY(cudaMemcpy(k.data(), e->ls_key[0], sizeof(unsigned long long) * (size_t)n_l, cudaMemcpyDeviceToHost));
    QB_CUDA_TRY(cudaMemcpy(v.data(), e->ls_val[0], sizeof(unsigned int) * (size_t)n_l, cudaMemcpyDeviceToHost));
    for (int i = 0; i < n_l; i++) { memcpy(&sorted_s[i], &k[i], 8); sorted_idx[i] = (c_int)v[i]; }
  }
  engine_destroy(e);
  return rc;
}

extern "C" int qpalm_b200_newton_solve(const solver_sparse *Q, const solver_sparse *A, const c_float *sigma,
        const c_int *active, c_float beta, const c_float *rhs, c_float *d, c_float *L_out) {
  const int n = (int)Q->ncol, m = A ? (int)A->nrow : 0;
  Engine *e = nullptr; int rc;
  if ((rc = make_engine(&e, n, m, A, Q, false, L_out ? 1 : 0))) return rc;   // a dense L can only be returned by the dense path
  int na = 0;
  if (active && m > 0) {
    std::vector<double> ss((size_t)m);
    for (int i = 0; i < m; i++) { ss[i] = sqrt(sigma[i]); na += active[i] != 0; }
    upload(e, e->sigma, sigma, m); upload(e, e->sqrt_sigma, ss.data(), m);
    cudaStreamSynchronize(e->stream);
    up_int(e, e->active, active, m);
  }
  std::vector<double> neg((size_t)n);
  for (int i = 0; i < n; i++) neg[i] = -rhs[i];
  upload(e, e->dphi, neg.data(), n);
  rc = step_newton_refactor(e, active != nullptr && m > 0, true, beta, na);
  rc |= step_newton_solve(e);
  rc |= download(e, d, e->d, n);
  if (L_out) {
    std::vector<double> L((size_t)e->ld * e->npad);
    QB_CUDA_TRY(cudaMemcpy(L.data(), e->L, sizeof(double) * L.size(), cudaMemcpyDeviceToHost));
    for (int j = 0; j < n; j++) for (int i = 0; i < n; i++) L_out[(size_t)i + (size_t)n * j] = (i >= j) ? L[(size_t)i + (size_t)e->ld * j] : 0.0;
  }
  int info = 0;
  QB_CUDA_TRY(cudaMemcpy(&info, e->info_dev, sizeof(int), cudaMemcpyDeviceToHost));
  engine_destroy(e);
  return rc ? rc : (info ? 1000 + info : 0);
}

extern "C" int qpalm_b200_updown(c_int n_, c_int k_, c_float *L, const c_float *W, c_int update) {
  const int n = (int)n_, k = (int)k_;
  Engine *e = nullptr; int rc;
  if ((rc = make_engine(&e, n, 0, nullptr, nullptr, false, 1))) return rc;   // dense-factor operator: never the supernodal path
  const int ld = e->ld, npad = e->npad;
  std::vector<double> Lp((size_t)ld * npad, 0.0);
  for (int j = 0; j < npad; j++) for (int i = j; i < npad; i++)
    Lp[(size_t)i + (size_t)ld * j] = (i < n && j < n) ? L[(size_t)i + (size_t)n * j] : (i == j ? 1.0 : 0.0);
  QB_CUDA_TRY(cudaMemcpy(e->L, Lp.data(), sizeof(double) * Lp.size(), cudaMemcpyHostToDevice));
  QB_CUDA_TRY(cudaMemset(e->info_dev, 0, sizeof(int)));
  rc = 0;
  bool gen = use_updown_gen(e);   // same dispatch as step_newton_updown: generator-form passes of <= 32 columns (updown_gen.cu)
  for (int off = 0; off < k && !rc && gen; off += chol_updown_gen_max_rank()) {
    const int kk = k - off < chol_updown_gen_max_rank() ? k - off : chol_updown_gen_max_rank();
    std::vector<double> Wp((size_t)ld * kk, 0.0);
    for (int c = 0; c < kk; c++) for (int i = 0; i < n; i++) Wp[(size_t)i + (size_t)ld * c] = W[(size_t)i + (size_t)n * (off + c)];
    QB_CUDA_TRY(cudaStreamSynchronize(e->stream));
    QB_CUDA_TRY(cudaMemcpy(e->W, Wp.data(), sizeof(double) * Wp.size(), cudaMemcpyHostToDevice));
    rc = trtri_diag_blocks(e->stream, npad, e->L, ld, e->invdiag);
    if (!rc) rc = chol_updown_gen(e->stream, npad, e->L, ld, e->invdiag, e->W, ld, kk, update ? kk : 0, e->info_dev);
    if (rc == 1 && off == 0) { gen = false; rc = 0; }   // unavailable here: per-panel kernels below
  }
  for (int off = 0; off < k && !rc && !gen; off += 8) {
    const int kk = k - off < 8 ? k - off : 8;
    std::vector<double> Wp((size_t)ld * 8, 0.0);
    for (int c = 0; c < kk; c++) for (int i = 0; i < n; i++) Wp[(size_t)i + (size_t)ld * c] = W[(size_t)i + (size_t)n * (off + c)];
    QB_CUDA_TRY(cudaStreamSynchronize(e->stream));   // e->stream is non-blocking: order the copy after the previous sweep
    QB_CUDA_TRY(cudaMemcpy(e->W, Wp.data(), sizeof(double) * Wp.size(), cudaMemcpyHostToDevice));
    rc = chol_updown(e->stream, npad, e->L, ld, e->W, ld, kk, update ? +1 : -1, e->ud_coef, e->info_dev);
  }
  QB_CUDA_TRY(cudaStreamSynchronize(e->stream));
  QB_CUDA_TRY(cudaMemcpy(Lp.data(), e->L, sizeof(double) * Lp.size(), cudaMemcpyDeviceToHost));
  for (int j = 0; j < n; j++) for (int i = 0; i < n; i++) L[(size_t)i + (size_t)n * j] = (i >= j) ? Lp[(size_t)i + (size_t)ld * j] : 0.0;
  int info = 0;
  QB_CUDA_TRY(cudaMemcpy(&info, e->info_dev, sizeof(int), cudaMemcpyDeviceToHost));
  engine_destroy(e);
  return rc ? rc : (info ? 1000 : 0);
}


// ------------------------------------------------------------------------------------------------
// sparse Newton system (sparse.cuh): host-only symbolic analysis + device factor / update / solve
// ------------------------------------------------------------------------------------------------
namespace {
struct HostA { std::vector<int> cp, ci, rp, rj; };
void host_csr_csc(const solver_sparse *A, int n, HostA *h) {
  const int m = A ? (int)A->nrow : 0;
  h->cp.assign((size_t)n + 1, 0); h->rp.assign((size_t)m + 1, 0);
  if (!A || m == 0) return;
  const long long *Ap = (const long long *)A->p, *Ai = (const long long *)A->i;
  const long long nnz = Ap[n];
  h->ci.resize(nnz); h->rj.resize(nnz);
  for (int j = 0; j <= n; j++) h->cp[j] = (int)Ap[j];
  for (long long k = 0; k < nnz; k++) { h->ci[k] = (int)Ai[k]; h->rp[Ai[k] + 1]++; }
  for (int i = 0; i < m; i++) h->rp[i + 1] += h->rp[i];
  std::vector<int> fill(h->rp.begin(), h->rp.end() - 1);
  for (int j = 0; j < n; j++) for (long long k = Ap[j]; k < Ap[j + 1]; k++) h->rj[fill[Ai[k]]++] = j;
}
}  // namespace

struct QPALMB200Symbolic { SymHost h; };

extern "C" QPALMB200Symbolic *qpalm_b200_symbolic_analyze(const solver_sparse *Q, const solver_sparse *A) {
  const int n = (int)Q->ncol, m = A ? (int)A->nrow : 0;
  HostA ha; host_csr_csc(A, n, &ha);
  QPALMB200Symbolic *S = new QPALMB200Symbolic();
  if (symbolic_analyze(n, m, ha.cp.data(), ha.ci.data(), ha.rp.data(), ha.rj.data(), (const long long *)Q->p, (const long long *)Q->i,
                       true, &S->h) != 0) { delete S; return nullptr; }
  return S;
}
extern "C" int qpalm_b200_symbolic_info(const QPALMB200Symbolic *S, c_int out8[8], double *flops) {
  const SymHost &h = S->h;
  out8[0] = h.n; out8[1] = h.nsuper; out8[2] = h.nlevels; out8[3] = h.max_ns; out8[4] = h.max_nf; out8[5] = h.nnzS; out8[6] = h.nnzL;
  out8[7] = h.upd_total;
  if (flops) *flops = h.flops;
  return 0;
}
extern "C" c_int qpalm_b200_symbolic_array(const QPALMB200Symbolic *S, const char *name, c_int *out, c_int cap) {
  const SymHost &h = S->h;
  const std::vector<int> *v = nullptr; const std::vector<long long> *w = nullptr;
  const std::string nm(name);
  if (nm == "perm") v = &h.perm; else if (nm == "iperm") v = &h.iperm; else if (nm == "sn_first") v = &h.sn_first;
  else if (nm == "sn_of_col") v = &h.sn_of_col; else if (nm == "rows_off") v = &h.rows_off; else if (nm == "rowidx") v = &h.rowidx;
  else if (nm == "rel") v = &h.rel; else if (nm == "sn_parent") v = &h.sn_parent; else if (nm == "child_ptr") v = &h.child_ptr;
  else if (nm == "child_idx") v = &h.child_idx; else if (nm == "lvl_ptr") v = &h.lvl_ptr; else if (nm == "lvl_sn") v = &h.lvl_sn;
  else if (nm == "panel_off") w = &h.panel_off; else if (nm == "upd_off") w = &h.upd_off;
  else return -1;
  const c_int len = v ? (c_int)v->size() : (c_int)w->size();
  if (out) for (c_int i = 0; i < len && i < cap; i++) out[i] = v ? (c_int)(*v)[i] : (c_int)(*w)[i];
  return len;
}
extern "C" void qpalm_b200_symbolic_free(QPALMB200Symbolic *S) { delete S; }

extern "C" int qpalm_b200_sparse_newton(const solver_sparse *Q, const solver_sparse *A, const c_float *sigma, const c_int *active,
        c_float beta, const c_float *rhs, c_float *d, c_float *L_out, c_int *perm_out, const c_int *enter, c_int nb_enter,
        const c_int *leave, c_int nb_leave, c_float *rowsums_out) {
  const int n = (int)Q->ncol, m = A ? (int)A->nrow : 0;
  Engine *e = nullptr; int rc;
  setenv("QPALM_B200_NEWTON", "sparse", 1);
  rc = make_engine(&e, n, m, A, Q);
  unsetenv("QPALM_B200_NEWTON");
  if (rc) return rc;
  if (!e->sp) { engine_destroy(e); return 7; }
  int na = 0;
  if (m > 0) {
    std::vector<double> ss((size_t)m);
    std::vector<c_int> act((size_t)m, 0);
    for (int i = 0; i < m; i++) { ss[i] = sqrt(sigma[i]); if (active) act[i] = active[i]; na += act[i] != 0; }
    upload(e, e->sigma, sigma, m); upload(e, e->sqrt_sigma, ss.data(), m);
    cudaStreamSynchronize(e->stream);
    up_int(e, e->active, act.data(), m);
  }
  std::vector<double> neg((size_t)n);
  for (int i = 0; i < n; i++) neg[i] = -rhs[i];
  upload(e, e->dphi, neg.data(), n);
  QB_CUDA_TRY(cudaMemset(e->info_dev, 0, sizeof(int)));
  if (rowsums_out) {   // Gershgorin row sums of A_J' Sigma_J A_J in the ORIGINAL ordering (boost_gamma)
    double ub = 0;
    rc = step_gershgorin_AtSA(e, &ub);
    rowsums_out[0] = ub;
  }
  rc |= step_newton_refactor(e, m > 0, true, beta, na);
  if (nb_enter > 0) { up_int(e, e->enter, enter, (int)nb_enter); }
  if (nb_leave > 0) { up_int(e, e->leave, leave, (int)nb_leave); }
  if (nb_enter + nb_leave > 0) rc |= step_newton_updown(e, (int)nb_enter, (int)nb_leave);
  rc |= step_newton_solve(e);
  rc |= download(e, d, e->d, n);
  if (L_out && perm_out) rc |= sparse_chol_download(e->sp, e->stream, e->spL, L_out, (long long *)perm_out);
  int info = 0;
  QB_CUDA_TRY(cudaMemcpy(&info, e->info_dev, sizeof(int), cudaMemcpyDeviceToHost));
  engine_destroy(e);
  return rc ? rc : (info ? 1000 + info : 0);
}

namespace {
struct LdlBuffers {   // device buffers of one sparse_ldl call, released on every return path
  SparseChol *sp = nullptr;
  cudaStream_t st = nullptr;
  int *Kp = nullptr, *Ki = nullptr, *info = nullptr;
  double *Kx = nullptr, *panels = nullptr, *rhs = nullptr, *x = nullptr;
  ~LdlBuffers() {
    if (st) cudaStreamSynchronize(st);
    sparse_chol_destroy(sp);
    void *ptrs[] = {Kp, Ki, info, Kx, panels, rhs, x};
    for (void *p : ptrs) if (p) cudaFree(p);
    if (st) cudaStreamDestroy(st);
  }
};
}  // namespace

extern "C" int qpalm_b200_sparse_ldl(const solver_sparse *K, c_int n_pos, const c_float *rhs, c_float *x, c_float *L_out,
        c_int *perm_out, c_float *panels_out, c_int panels_cap, c_int *panels_len) {
  if (!K || !rhs || !x || K->nrow != K->ncol || K->ncol < 1 || K->ncol > (1 << 30) || n_pos < 0 || n_pos > K->ncol) return 1;
  const int N = (int)K->ncol;
  const long long *Kp = (const long long *)K->p, *Ki = (const long long *)K->i;
  const double *Kv = (const double *)K->x;
  // lower triangle, strictly ascending rows per column: the assembly stores (does not add) each entry, so a duplicate would be lost
  std::vector<int> cnt((size_t)N + 1, 0);
  for (int j = 0; j < N; j++) {
    if (Kp[j + 1] < Kp[j]) return 2;
    long long last = -1;
    for (long long k = Kp[j]; k < Kp[j + 1]; k++) {
      const long long i = Ki[k];
      if (i < 0 || i >= N || i <= last) return 2;
      last = i;
      if (i < j) continue;
      cnt[i]++;
      if (i != j) cnt[j]++;
    }
  }
  // full symmetric CSR (row i: entries (i, j <= i) in ascending j, then (i, k > i) in ascending k), as the engine keeps Q
  std::vector<int> rp((size_t)N + 1, 0);
  for (int i = 0; i < N; i++) rp[i + 1] = rp[i] + cnt[i];
  const size_t nnzF = (size_t)rp[N];
  std::vector<int> rj(nnzF + 1), fill(rp.begin(), rp.end());
  std::vector<double> rx(nnzF + 1);
  for (int j = 0; j < N; j++) for (long long k = Kp[j]; k < Kp[j + 1]; k++) if (Ki[k] >= j) { const int p = fill[Ki[k]]++; rj[p] = j; rx[p] = Kv[k]; }
  for (int j = 0; j < N; j++) for (long long k = Kp[j]; k < Kp[j + 1]; k++) if (Ki[k] > j) { const int p = fill[j]++; rj[p] = (int)Ki[k]; rx[p] = Kv[k]; }

  LdlBuffers b;
  QB_CUDA_TRY(cudaStreamCreate(&b.st));
  if (int r = sparse_ldl_analyze(&b.sp, N, (int)n_pos, Kp, Ki, b.st)) return r;
  const SparseCholInfo *I = sparse_chol_info(b.sp);
  if (panels_len) *panels_len = (c_int)I->nnzL;
  QB_CUDA_TRY(cudaMalloc((void **)&b.Kp, sizeof(int) * ((size_t)N + 1)));
  QB_CUDA_TRY(cudaMalloc((void **)&b.Ki, sizeof(int) * (nnzF + 1)));
  QB_CUDA_TRY(cudaMalloc((void **)&b.Kx, sizeof(double) * (nnzF + 1)));
  QB_CUDA_TRY(cudaMalloc((void **)&b.info, sizeof(int)));
  QB_CUDA_TRY(cudaMalloc((void **)&b.panels, sizeof(double) * sparse_chol_factor_doubles(b.sp)));
  QB_CUDA_TRY(cudaMalloc((void **)&b.rhs, sizeof(double) * (size_t)N));
  QB_CUDA_TRY(cudaMalloc((void **)&b.x, sizeof(double) * (size_t)N));
  QB_CUDA_TRY(cudaMemcpyAsync(b.Kp, rp.data(), sizeof(int) * ((size_t)N + 1), cudaMemcpyHostToDevice, b.st));
  QB_CUDA_TRY(cudaMemcpyAsync(b.Ki, rj.data(), sizeof(int) * (nnzF + 1), cudaMemcpyHostToDevice, b.st));
  QB_CUDA_TRY(cudaMemcpyAsync(b.Kx, rx.data(), sizeof(double) * (nnzF + 1), cudaMemcpyHostToDevice, b.st));
  QB_CUDA_TRY(cudaMemcpyAsync(b.rhs, rhs, sizeof(double) * (size_t)N, cudaMemcpyHostToDevice, b.st));
  QB_CUDA_TRY(cudaMemsetAsync(b.info, 0, sizeof(int), b.st));
  if (int r = sparse_chol_assemble(b.sp, b.st, b.panels, true, b.Kp, b.Ki, b.Kx, nullptr, nullptr, nullptr, nullptr, nullptr,
                                   nullptr, nullptr, nullptr, 0.0)) return r;
  if (int r = sparse_chol_factor(b.sp, b.st, b.panels, b.info)) return r;
  if (int r = sparse_chol_solve(b.sp, b.st, b.panels, b.rhs, b.x, false)) return r;
  int info = 0;
  QB_CUDA_TRY(cudaMemcpyAsync(x, b.x, sizeof(double) * (size_t)N, cudaMemcpyDeviceToHost, b.st));
  QB_CUDA_TRY(cudaMemcpyAsync(&info, b.info, sizeof(int), cudaMemcpyDeviceToHost, b.st));
  QB_CUDA_TRY(cudaStreamSynchronize(b.st));
  if (panels_out && panels_cap >= I->nnzL)
    QB_CUDA_TRY(cudaMemcpy(panels_out, b.panels, sizeof(double) * (size_t)I->nnzL, cudaMemcpyDeviceToHost));
  if (L_out && perm_out)
    if (int r = sparse_chol_download(b.sp, b.st, b.panels, L_out, (long long *)perm_out)) return r;
  return info ? 1000 + info : 0;
}

extern "C" int qpalm_b200_kkt_newton(const solver_sparse *Q, const solver_sparse *A, const c_float *sigma, const c_int *active,
        c_float beta, const c_float *rhs, c_float *d, c_int *refine_out, c_float *norms_out) {
  if (!Q || !A || !sigma || !active || !rhs || !d || A->nrow < 1 || A->ncol != Q->ncol) return 1;
  const int n = (int)Q->ncol, m = (int)A->nrow;
  Engine *e = nullptr;
  if (int rc = make_engine(&e, n, m, A, Q, false, 3)) return rc;   // 3: the KKT path asked for (FACTORIZE_KKT)
  if (!e->kkt) { engine_destroy(e); return 7; }                   // dense-classified data never gets the KKT engine
  std::vector<double> sinv((size_t)m);
  for (int i = 0; i < m; i++) sinv[i] = 1.0 / sigma[i];
  upload(e, e->sigma, sigma, m); upload(e, e->sigma_inv, sinv.data(), m);
  std::vector<double> neg((size_t)n);
  for (int i = 0; i < n; i++) neg[i] = -rhs[i];
  upload(e, e->dphi, neg.data(), n);
  cudaStreamSynchronize(e->stream);
  up_int(e, e->active, active, m);
  QB_CUDA_TRY(cudaMemset(e->info_dev, 0, sizeof(int)));
  const long long r0 = kkt_refine_count(e->kkt);
  int rc = kkt_refactor(e->kkt, e, beta);
  if (!rc) rc = kkt_solve(e->kkt, e);
  if (!rc) rc = download(e, d, e->d, n);
  if (refine_out) *refine_out = (c_int)(kkt_refine_count(e->kkt) - r0);
  if (norms_out) kkt_last_norms(e->kkt, norms_out);
  int info = 0;
  if (!rc) rc = -(int)cudaMemcpy(&info, e->info_dev, sizeof(int), cudaMemcpyDeviceToHost);
  engine_destroy(e);
  return rc ? rc : (info ? 1000 + info : 0);
}

extern "C" int qpalm_b200_lobpcg(const solver_sparse *Q, const c_float *x0, c_float *lambda_out, c_int *iters_out) {
  Engine *e = nullptr; int rc;
  if ((rc = make_engine(&e, (int)Q->ncol, 0, nullptr, Q))) return rc;
  long long its = 0;
  rc = lobpcg_device(e, x0, lambda_out, &its);
  if (iters_out) *iters_out = its;
  engine_destroy(e);
  return rc;
}

// ---- micro-benchmarks for the FP64 tensor roofline ---------------------------------------------------
__global__ void k_fill_rand(double *p, size_t len, unsigned long long seed) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < len; i += (size_t)gridDim.x * blockDim.x) {
    unsigned long long s = seed + i * 0x9E3779B97F4A7C15ull;
    s ^= s >> 30; s *= 0xBF58476D1CE4E5B9ull; s ^= s >> 27; s *= 0x94D049BB133111EBull; s ^= s >> 31;
    p[i] = (double)(s >> 11) * (1.0 / 9007199254740992.0) - 0.5;
  }
}
extern "C" int qpalm_b200_bench_dsyrk(c_int n_, c_int k_, c_int reps, double *ms_out) {
  const int n = round_up((int)n_, 128), k = round_up((int)k_, 16);
  double *W = nullptr, *C = nullptr;
  QB_CUDA_TRY(cudaMalloc(&W, sizeof(double) * (size_t)n * k));
  QB_CUDA_TRY(cudaMalloc(&C, sizeof(double) * (size_t)n * n));
  cudaStream_t s; QB_CUDA_TRY(cudaStreamCreate(&s));
  QB_LAUNCH(k_fill_rand, 1024, 256, 0, s, W, (size_t)n * k, 1234ull);
  QB_CUDA_TRY(cudaMemsetAsync(C, 0, sizeof(double) * (size_t)n * n, s));
  cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
  int rc = dgemm_nt(s, n, n, k, W, n, W, n, C, n, 1.0, 1.0, true);   // warm-up
  cudaEventRecord(a, s);
  for (int r = 0; r < reps && !rc; r++) rc = dgemm_nt(s, n, n, k, W, n, W, n, C, n, 1.0, 1.0, true);
  cudaEventRecord(b, s);
  QB_CUDA_TRY(cudaEventSynchronize(b));
  float ms = 0; cudaEventElapsedTime(&ms, a, b);
  *ms_out = ms / (reps > 0 ? reps : 1);
  cudaEventDestroy(a); cudaEventDestroy(b); cudaStreamDestroy(s); cudaFree(W); cudaFree(C);
  return rc;
}
__global__ void k_make_spd(int n, double *A) {   // A <- small random symmetric part + n on the diagonal (lower used)
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
  if (i < n && i == j) A[(size_t)i + (size_t)n * j] += (double)n;
}
extern "C" int qpalm_b200_bench_potrf(c_int n_, c_int reps, double *ms_out) {
  const int n = round_up((int)n_, 128);
  double *A = nullptr, *L = nullptr, *X = nullptr; int *info = nullptr;
  QB_CUDA_TRY(cudaMalloc(&A, sizeof(double) * (size_t)n * n));
  QB_CUDA_TRY(cudaMalloc(&L, sizeof(double) * (size_t)n * n));
  QB_CUDA_TRY(cudaMalloc(&X, sizeof(double) * (size_t)n * 128));
  QB_CUDA_TRY(cudaMalloc(&info, sizeof(int)));
  QB_CUDA_TRY(cudaMemset(info, 0, sizeof(int)));
  cudaStream_t s; QB_CUDA_TRY(cudaStreamCreate(&s));
  QB_LAUNCH(k_fill_rand, 1024, 256, 0, s, A, (size_t)n * n, 99ull);
  dim3 g(cdiv(n, 256), n);
  QB_LAUNCH(k_make_spd, g, 256, 0, s, n, A);
  cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
  float total = 0; int rc = 0;
  for (int r = 0; r < reps + 1 && !rc; r++) {
    QB_CUDA_TRY(cudaMemcpyAsync(L, A, sizeof(double) * (size_t)n * n, cudaMemcpyDeviceToDevice, s));
    cudaEventRecord(a, s);
    rc = potrf_lower(s, n, L, n, X, info);
    cudaEventRecord(b, s);
    QB_CUDA_TRY(cudaEventSynchronize(b));
    float ms = 0; cudaEventElapsedTime(&ms, a, b);
    if (r > 0) total += ms;
  }
  *ms_out = total / (reps > 0 ? reps : 1);
  int hinfo = 0; cudaMemcpy(&hinfo, info, sizeof(int), cudaMemcpyDeviceToHost);
  cudaEventDestroy(a); cudaEventDestroy(b); cudaStreamDestroy(s); cudaFree(A); cudaFree(L); cudaFree(X); cudaFree(info);
  return rc ? rc : hinfo;
}

// one rank-k update (then the matching downdate so the factor stays bounded) on a factored random SPD matrix, as the solver
// runs it: generator-form passes of <= 32 columns, each with the refresh of the inverted diagonal blocks the next pass needs.
// ms per rank-k update or downdate, averaged over 2 * reps of them
extern "C" int qpalm_b200_bench_updown(c_int n_, c_int k_, c_int reps, double *ms_out) {
  const int n = round_up((int)n_, 128), k = (int)k_;
  if (k < 1) return 1;
  double *L = nullptr, *X = nullptr, *W = nullptr; int *info = nullptr;
  QB_CUDA_TRY(cudaMalloc(&L, sizeof(double) * (size_t)n * n));
  QB_CUDA_TRY(cudaMalloc(&X, sizeof(double) * (size_t)n * 128));
  QB_CUDA_TRY(cudaMalloc(&W, sizeof(double) * (size_t)n * k));
  QB_CUDA_TRY(cudaMalloc(&info, sizeof(int)));
  QB_CUDA_TRY(cudaMemset(info, 0, sizeof(int)));
  cudaStream_t s; QB_CUDA_TRY(cudaStreamCreate(&s));
  QB_LAUNCH(k_fill_rand, 1024, 256, 0, s, L, (size_t)n * n, 99ull);
  QB_LAUNCH(k_fill_rand, 256, 256, 0, s, W, (size_t)n * k, 7ull);
  dim3 g(cdiv(n, 256), n);
  QB_LAUNCH(k_make_spd, g, 256, 0, s, n, L);
  int rc = potrf_lower(s, n, L, n, X, info);
  cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
  float total = 0;
  const int KMAX = chol_updown_gen_max_rank();
  for (int r = 0; r < reps + 1 && !rc; r++) {
    cudaEventRecord(a, s);
    for (int update = 1; update >= 0 && !rc; update--)
      for (int off = 0; off < k && !rc; off += KMAX) {
        const int kk = k - off < KMAX ? k - off : KMAX;
        rc = chol_updown_gen(s, n, L, n, X, W + (size_t)n * off, n, kk, update ? kk : 0, info);
        if (!rc) rc = trtri_diag_blocks(s, n, L, n, X);
      }
    cudaEventRecord(b, s);
    QB_CUDA_TRY(cudaEventSynchronize(b));
    float ms = 0; cudaEventElapsedTime(&ms, a, b);
    if (r > 0) total += ms;
  }
  *ms_out = total / (2.0 * (reps > 0 ? reps : 1));
  int hinfo = 0; cudaMemcpy(&hinfo, info, sizeof(int), cudaMemcpyDeviceToHost);
  chol_updown_gen_release(s);
  cudaEventDestroy(a); cudaEventDestroy(b); cudaStreamDestroy(s); cudaFree(L); cudaFree(X); cudaFree(W); cudaFree(info);
  return rc ? rc : hinfo;
}

// sparse products at a caller-given shape (C1 / C2 of BASELINE.json): ms per A x, A' y and Q x through the solver's kernels.
// out3 = {ms A x, ms A' y, ms Q x}; algorithmic bytes per product are 12 nnz + 4 (rows + 1) + 8 (rows + cols) (SURVEY 8(d)).
extern "C" int qpalm_b200_bench_spmv(const solver_sparse *A, const solver_sparse *Q, c_int reps, double *out3, c_int *nnz3) {
  Engine *e = nullptr;
  const int n = (int)Q->ncol, m = (int)A->nrow;
  if (int rc = make_engine(&e, n, m, A, Q, false, 2)) return rc;
  if (e->A_dense || e->Q_dense) { engine_destroy(e); return 7; }
  vec_set(e, e->x, 1.0, n); vec_set(e, e->y, 1.0, m);
  cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
  for (int which = 0; which < 3; which++) {
    auto run = [&]() { return which == 0 ? spmv_A(e, e->x, e->Ax) : (which == 1 ? spmv_At(e, e->y, e->Aty) : spmv_Q(e, e->x, e->Qx)); };
    run();
    cudaEventRecord(a, e->stream);
    for (int r = 0; r < reps; r++) run();
    cudaEventRecord(b, e->stream);
    QB_CUDA_TRY(cudaEventSynchronize(b));
    float ms = 0; cudaEventElapsedTime(&ms, a, b);
    out3[which] = ms / (reps > 0 ? reps : 1);
  }
  nnz3[0] = e->A_csr.nnz; nnz3[1] = e->A_csc.nnz; nnz3[2] = e->Q_csr.nnz;
  cudaEventDestroy(a); cudaEventDestroy(b);
  engine_destroy(e);
  return 0;
}

// ---- batch API: implemented in batch.cu ---------------------------------------------------------------

// FP64 tensor-pipe issue-rate peak: register-resident mma.sync m8n8k4 chains, no memory traffic.
// MEASURED_PEAKS.json has no FP64 entry, so bench.py uses this as the denominator of the tensor roofline.
__global__ void __launch_bounds__(256) k_dmma_peak(int iters, double *sink) {
  double acc[16][2];
#pragma unroll
  for (int i = 0; i < 16; i++) { acc[i][0] = threadIdx.x * 1e-9; acc[i][1] = i * 1e-9; }
  double a = 1.0 + threadIdx.x * 1e-6, b = 1.0 - threadIdx.x * 1e-6;
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int i = 0; i < 16; i++)
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                   : "+d"(acc[i][0]), "+d"(acc[i][1]) : "d"(a), "d"(b));
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 16; i++) s += acc[i][0] + acc[i][1];
  if (s == 123.456) sink[0] = s;
}
extern "C" int qpalm_b200_bench_dmma_peak(double *tflops_out) {
  double *sink = nullptr;
  QB_CUDA_TRY(cudaMalloc(&sink, 8));
  cudaStream_t s; QB_CUDA_TRY(cudaStreamCreate(&s));
  cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
  const int iters = 4096, grid = 148 * 8;
  QB_LAUNCH(k_dmma_peak, grid, 256, 0, s, 64, sink);
  double best = 0;
  for (int r = 0; r < 3; r++) {
    cudaEventRecord(a, s);
    QB_LAUNCH(k_dmma_peak, grid, 256, 0, s, iters, sink);
    cudaEventRecord(b, s);
    QB_CUDA_TRY(cudaEventSynchronize(b));
    float ms = 0; cudaEventElapsedTime(&ms, a, b);
    const double flops = (double)grid * 8 /*warps*/ * iters * 16.0 * 512.0;
    const double tf = flops / (ms * 1e-3) / 1e12;
    if (tf > best) best = tf;
  }
  *tflops_out = best;
  cudaEventDestroy(a); cudaEventDestroy(b); cudaStreamDestroy(s); cudaFree(sink);
  return 0;
}

// scalar FP64 FMA issue-rate peak (register-resident DFMA chains, 16 independent accumulators per thread): the bound of every
// kernel that does its arithmetic with plain fma() instead of DMMA.  warps_per_sm: resident warps per SM during the probe.
__global__ void __launch_bounds__(256) k_dfma_peak(int iters, double *sink) {
  double acc[16];
#pragma unroll
  for (int i = 0; i < 16; i++) acc[i] = threadIdx.x * 1e-9 + i * 1e-7;
  const double a = 1.0 + threadIdx.x * 1e-9, b = 1e-9;
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int i = 0; i < 16; i++) acc[i] = fma(acc[i], a, b);
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 16; i++) s += acc[i];
  if (s == 123.456) sink[0] = s;
}
extern "C" int qpalm_b200_bench_dfma_peak(double *tflops_out) {
  double *sink = nullptr;
  QB_CUDA_TRY(cudaMalloc(&sink, 8));
  cudaStream_t s; QB_CUDA_TRY(cudaStreamCreate(&s));
  cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
  const int iters = 8192, grid = 148 * 8;
  QB_LAUNCH(k_dfma_peak, grid, 256, 0, s, 64, sink);
  double best = 0;
  for (int r = 0; r < 3; r++) {
    cudaEventRecord(a, s);
    QB_LAUNCH(k_dfma_peak, grid, 256, 0, s, iters, sink);
    cudaEventRecord(b, s);
    QB_CUDA_TRY(cudaEventSynchronize(b));
    float ms = 0; cudaEventElapsedTime(&ms, a, b);
    const double flops = (double)grid * 256 * iters * 16.0 * 2.0;
    const double tf = flops / (ms * 1e-3) / 1e12;
    if (tf > best) best = tf;
  }
  *tflops_out = best;
  cudaEventDestroy(a); cudaEventDestroy(b); cudaStreamDestroy(s); cudaFree(sink);
  return 0;
}

// HBM roofline probes for the matrix-vector kernels: dense At (n x m) products at the solver's shapes.
extern "C" int qpalm_b200_bench_gemv(c_int n_, c_int m_, c_int reps, double *ms_cols_out, double *ms_rows_out) {
  const int n = (int)n_, m = (int)m_;
  Engine e;   // minimal engine: only what the two dense kernels need
  QB_CUDA_TRY(cudaStreamCreate(&e.stream));
  e.n = n; e.m = m; e.A_dense = true; e.m_loc = m; e.m_cap = m;
  QB_CUDA_TRY(cudaMalloc(&e.At, sizeof(double) * (size_t)n * m));
  QB_CUDA_TRY(cudaMalloc(&e.x, sizeof(double) * n)); QB_CUDA_TRY(cudaMalloc(&e.y, sizeof(double) * m));
  QB_CUDA_TRY(cudaMalloc(&e.Ax, sizeof(double) * m)); QB_CUDA_TRY(cudaMalloc(&e.Aty, sizeof(double) * n));
  const int rowctas = cdiv(n, 128); int splits = cdiv(2048, rowctas); splits = splits < 1 ? 1 : (splits > 64 ? 64 : splits);
  e.gemv_splits = splits;
  QB_CUDA_TRY(cudaMalloc(&e.gemv_partials, sizeof(double) * (size_t)splits * n));
  QB_LAUNCH(k_fill_rand, 2048, 256, 0, e.stream, e.At, (size_t)n * m, 5ull);
  QB_LAUNCH(k_fill_rand, 64, 256, 0, e.stream, e.x, (size_t)n, 6ull);
  QB_LAUNCH(k_fill_rand, 64, 256, 0, e.stream, e.y, (size_t)m, 7ull);
  cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
  spmv_A(&e, e.x, e.Ax); spmv_At(&e, e.y, e.Aty);
  float ms = 0;
  cudaEventRecord(a, e.stream);
  for (int r = 0; r < reps; r++) spmv_A(&e, e.x, e.Ax);
  cudaEventRecord(b, e.stream); QB_CUDA_TRY(cudaEventSynchronize(b)); cudaEventElapsedTime(&ms, a, b);
  *ms_cols_out = ms / reps;
  cudaEventRecord(a, e.stream);
  for (int r = 0; r < reps; r++) spmv_At(&e, e.y, e.Aty);
  cudaEventRecord(b, e.stream); QB_CUDA_TRY(cudaEventSynchronize(b)); cudaEventElapsedTime(&ms, a, b);
  *ms_rows_out = ms / reps;
  cudaEventDestroy(a); cudaEventDestroy(b);
  cudaFree(e.At); cudaFree(e.x); cudaFree(e.y); cudaFree(e.Ax); cudaFree(e.Aty); cudaFree(e.gemv_partials);
  chol_solve_release(e.stream);
  cudaStreamDestroy(e.stream);
  return 0;
}

// ---- test probes of the dense Newton-system kernels (dense.cu), run unchanged on caller data ---------------------------
// Host buffers in and out; the work runs on a fresh non-blocking stream, as in the engines.
namespace {
struct DenseProbe {   // stream and device buffers of one probe call, released on every return path
  cudaStream_t s = nullptr;
  std::vector<void *> p;
  bool failed = false;
  template <typename T> T *get(size_t count) {
    void *q = nullptr;
    if (dev_alloc(&q, sizeof(T) * (count ? count : 1))) { failed = true; return nullptr; }
    p.push_back(q);
    return static_cast<T *>(q);
  }
  template <typename T> T *up(const T *src, size_t count) {   // nullptr for a null source
    if (!src) return nullptr;
    T *d = get<T>(count);
    if (d && cudaMemcpyAsync(d, src, sizeof(T) * count, cudaMemcpyHostToDevice, s) != cudaSuccess) { failed = true; return nullptr; }
    return d;
  }
  std::vector<int> flags(const c_int *src, size_t count) {   // c_int (64-bit) array -> int array
    std::vector<int> t(count + 1, 0);
    for (size_t i = 0; i < count; i++) t[i] = (int)src[i];
    return t;
  }
  ~DenseProbe() {
    if (s) { cudaStreamSynchronize(s); chol_solve_release(s); chol_updown_gen_release(s); }
    for (void *q : p) cudaFree(q);
    if (s) cudaStreamDestroy(s);
  }
};
}  // namespace

extern "C" int qpalm_b200_dense_probe_gemm(c_int nb_, c_int M_, c_int N_, c_int K_, const c_int *Kz, const c_int *mask,
                                           const c_float *A, c_int lda, c_int sA, const c_float *B, c_int ldb, c_int sB,
                                           c_float *C, c_int ldc, c_int sC, c_float alpha, c_float beta, c_int lower_only,
                                           c_int in_place, c_int *tile_rows) {
  if (nb_ < 1 || M_ < 1 || N_ < 1 || K_ < 0 || M_ % 128 || N_ % 128 || K_ % 16 || M_ > (1 << 20) || N_ > (1 << 20) || K_ > (1 << 20)) return 1;
  if (in_place) { A = C; lda = ldc; sA = sC; if (N_ != 128 || K_ > N_) return 1; }
  if ((K_ > 0 && (!A || !B)) || !C || lda < M_ || ldb < N_ || ldc < M_ || (lda | ldb | ldc | sA | sB | sC) & 1) return 1;
  if (nb_ > 1 && (sA < lda * K_ || sB < ldb * K_ || sC < ldc * N_)) return 1;
  const int nb = (int)nb_, M = (int)M_, N = (int)N_, K = (int)K_;
  std::vector<int> kz, mk;
  DenseProbe d;
  if (Kz) {
    kz = d.flags(Kz, (size_t)nb);
    for (int b = 0; b < nb; b++) if (kz[b] < 0 || kz[b] > K || kz[b] % 16) return 1;   // the kernel runs Kz / 16 k-tiles
  }
  if (mask) mk = d.flags(mask, (size_t)nb);
  QB_CUDA_TRY(cudaStreamCreateWithFlags(&d.s, cudaStreamNonBlocking));
  const size_t nA = (size_t)(nb - 1) * sA + (size_t)lda * K, nB = (size_t)(nb - 1) * sB + (size_t)ldb * K;
  const size_t nC = (size_t)(nb - 1) * sC + (size_t)ldc * N;
  double *dC = d.up(C, nC);
  const double *dA = in_place ? dC : d.up(A, nA), *dB = d.up(B, nB);
  const int *dKz = Kz ? d.up(kz.data(), (size_t)nb) : nullptr, *dmask = mask ? d.up(mk.data(), (size_t)nb) : nullptr;
  if (d.failed) return 2;
  if (int r = dgemm_nt_batched(d.s, nb, M, N, K, dKz, dA, (int)lda, sA, dB, (int)ldb, sB, dC, (int)ldc, sC, alpha, beta,
                               lower_only != 0, dmask)) return r;
  if (tile_rows) *tile_rows = dgemm_last_tile_rows();
  QB_CUDA_TRY(cudaMemcpyAsync(C, dC, sizeof(double) * nC, cudaMemcpyDeviceToHost, d.s));
  QB_CUDA_TRY(cudaStreamSynchronize(d.s));
  return 0;
}

extern "C" int qpalm_b200_dense_probe_potrf(c_int nb_, c_int npad_, c_float *L, c_float *invdiag, const c_int *mask, c_int *info,
                                            c_int mode) {
  if (nb_ < 1 || npad_ < 128 || npad_ % 128 || npad_ > (1 << 16) || (mode != 0 && mode != 1) || !L || !invdiag || !info) return 1;
  if (mode == 0 && (nb_ != 1 || mask)) return 1;
  const int nb = (int)nb_, npad = (int)npad_;
  const size_t sL = (size_t)npad * npad, sX = (size_t)npad * kPanel;
  DenseProbe d;
  std::vector<int> mk = mask ? d.flags(mask, (size_t)nb) : std::vector<int>((size_t)nb, 1), inf = d.flags(info, (size_t)nb);
  QB_CUDA_TRY(cudaStreamCreateWithFlags(&d.s, cudaStreamNonBlocking));
  double *dL = d.up(L, nb * sL), *dX = d.up(invdiag, nb * sX);
  int *dinfo = d.up(inf.data(), (size_t)nb), *dmask = mode == 1 ? d.up(mk.data(), (size_t)nb) : nullptr;
  if (d.failed) return 2;
  // mode 0: the single-matrix entry (look-ahead for npad > 1024); mode 1: the batched schedule, never with look-ahead
  if (int r = mode == 0 ? potrf_lower(d.s, npad, dL, npad, dX, dinfo)
                        : potrf_lower_batched(d.s, nb, npad, dL, npad, (long long)sL, dX, (long long)sX, dinfo, dmask)) return r;
  QB_CUDA_TRY(cudaMemcpyAsync(L, dL, sizeof(double) * nb * sL, cudaMemcpyDeviceToHost, d.s));
  QB_CUDA_TRY(cudaMemcpyAsync(invdiag, dX, sizeof(double) * nb * sX, cudaMemcpyDeviceToHost, d.s));
  QB_CUDA_TRY(cudaMemcpyAsync(inf.data(), dinfo, sizeof(int) * nb, cudaMemcpyDeviceToHost, d.s));
  QB_CUDA_TRY(cudaStreamSynchronize(d.s));
  for (int b = 0; b < nb; b++) info[b] = inf[b];
  return 0;
}

extern "C" int qpalm_b200_dense_probe_trtri(c_int npad_, const c_float *L, c_float *invdiag) {
  if (npad_ < 128 || npad_ % 128 || npad_ > (1 << 16) || !L || !invdiag) return 1;
  const int npad = (int)npad_;
  DenseProbe d;
  QB_CUDA_TRY(cudaStreamCreateWithFlags(&d.s, cudaStreamNonBlocking));
  const double *dL = d.up(L, (size_t)npad * npad);
  double *dX = d.get<double>((size_t)npad * kPanel);
  if (d.failed) return 2;
  if (int r = trtri_diag_blocks(d.s, npad, dL, npad, dX)) return r;
  QB_CUDA_TRY(cudaMemcpyAsync(invdiag, dX, sizeof(double) * npad * kPanel, cudaMemcpyDeviceToHost, d.s));
  QB_CUDA_TRY(cudaStreamSynchronize(d.s));
  return 0;
}

extern "C" int qpalm_b200_dense_probe_solve(c_int nb_, c_int npad_, const c_float *L, const c_float *invdiag, c_float *V, c_int rounds_,
                                            const c_int *sizes, const c_int *mask, c_int mode, c_int *grid) {
  if (nb_ < 1 || npad_ < 128 || npad_ % 128 || npad_ > (1 << 16) || rounds_ < 1 || (mode != 0 && mode != 1) || !L || !invdiag || !V) return 1;
  if (mode == 0 && (nb_ != 1 || mask)) return 1;
  const int nb = (int)nb_, npad = (int)npad_, rounds = (int)rounds_;
  for (int r = 0; r < rounds && sizes; r++) if (sizes[r] < 128 || sizes[r] > npad || sizes[r] % 128) return 1;
  const size_t sL = (size_t)npad * npad, sX = (size_t)npad * kPanel, sV = (size_t)rounds * npad;
  DenseProbe d;
  std::vector<int> mk = mask ? d.flags(mask, (size_t)nb) : std::vector<int>();
  QB_CUDA_TRY(cudaStreamCreateWithFlags(&d.s, cudaStreamNonBlocking));
  const double *dL = d.up(L, nb * sL), *dX = d.up(invdiag, nb * sX);
  double *dV = d.up(V, nb * sV);
  const int *dmask = mask ? d.up(mk.data(), (size_t)nb) : nullptr;
  if (d.failed) return 2;
  // round r: V[b, r, :size_r] <- (L L')^{-1} V[b, r, :size_r] with the leading size_r x size_r block of L (its own factor)
  for (int r = 0; r < rounds; r++) {
    const int n = sizes ? (int)sizes[r] : npad;
    double *v = dV + (size_t)r * npad;
    if (int e = mode == 0 ? chol_solve(d.s, n, dL, npad, dX, v)
                          : chol_solve_batched(d.s, nb, n, dL, npad, (long long)sL, dX, (long long)sX, v, (long long)sV, dmask)) return e;
    if (grid) grid[r] = mode == 0 ? chol_solve_last_grid() : 0;
  }
  QB_CUDA_TRY(cudaMemcpyAsync(V, dV, sizeof(double) * nb * sV, cudaMemcpyDeviceToHost, d.s));
  QB_CUDA_TRY(cudaStreamSynchronize(d.s));
  return 0;
}

extern "C" int qpalm_b200_dense_probe_updown(c_int npad_, c_float *L, const c_float *W, c_int passes_, const c_int *k,
                                             const c_int *kpos, const c_int *sizes, c_int mode, c_int grid_cap, c_int *info,
                                             c_int *grid, c_float *What, c_float *Z, c_float *D) {
  if (npad_ < 128 || npad_ % 128 || npad_ > (1 << 16) || passes_ < 1 || (mode != 0 && mode != 1) || !L || !W || !k || !kpos || !info) return 1;
  const int npad = (int)npad_, passes = (int)passes_;
  size_t kt = 0;
  for (int r = 0; r < passes; r++) {
    const c_int kmax = mode == 0 ? chol_updown_gen_max_rank() : 8;
    if (k[r] < 1 || k[r] > kmax || kpos[r] < 0 || kpos[r] > k[r]) return 1;
    if (mode == 1 && kpos[r] != 0 && kpos[r] != k[r]) return 1;                        // the per-panel sweep has one sign per call
    if (sizes && (sizes[r] < 128 || sizes[r] > npad || sizes[r] % 128)) return 1;
    kt += (size_t)k[r];
  }
  if ((What || Z || D) && mode != 0) return 1;
  DenseProbe d;
  QB_CUDA_TRY(cudaStreamCreateWithFlags(&d.s, cudaStreamNonBlocking));
  double *dL = d.up(L, (size_t)npad * npad);
  double *dW = d.up(W, (size_t)npad * kt);       // a copy: the per-panel sweep overwrites its W
  double *dX = d.get<double>((size_t)npad * kPanel), *coef = d.get<double>(2 * 32 * 18 + 16);
  int *dinfo = d.get<int>(1);
  if (d.failed) return 2;
  struct Cap {   // the grid cap holds for this call only, on every return path
    explicit Cap(int c) { chol_updown_gen_set_grid_cap(c); }
    ~Cap() { chol_updown_gen_set_grid_cap(0); }
  } cap(mode == 0 ? (int)grid_cap : 0);
  std::vector<int> inf((size_t)passes, 0);
  size_t off = 0;
  int n = npad, kk = 0;
  for (int r = 0; r < passes; r++) {
    n = sizes ? (int)sizes[r] : npad;
    kk = (int)k[r];
    double *w = dW + off * npad;
    QB_CUDA_TRY(cudaMemsetAsync(dinfo, 0, sizeof(int), d.s));
    if (mode == 0) {
      if (int e = trtri_diag_blocks(d.s, n, dL, npad, dX)) return e;
      const int e = chol_updown_gen(d.s, n, dL, npad, dX, w, npad, kk, (int)kpos[r], dinfo);
      if (e == 1) return 3;
      if (e) return e;
    } else if (int e = chol_updown(d.s, n, dL, npad, w, npad, kk, kpos[r] ? +1 : -1, coef, dinfo)) {
      return e;
    }
    if (grid) {
      int gmax = 0;
      grid[2 * r] = mode == 0 ? chol_updown_gen_last_grid(&gmax) : 0;
      grid[2 * r + 1] = gmax;
    }
    QB_CUDA_TRY(cudaMemcpyAsync(&inf[r], dinfo, sizeof(int), cudaMemcpyDeviceToHost, d.s));
    off += (size_t)kk;
  }
  if (What || Z || D) {   // the last pass's What | Z | D, column stride n in the work space, npad here (rows >= n untouched)
    const double *ws = chol_updown_gen_workspace(d.s);
    if (!ws) return 1;
    const double *src[3] = {ws, ws + (size_t)n * 32, ws + (size_t)n * 64};
    c_float *dst[3] = {What, Z, D};
    for (int q = 0; q < 3; q++)
      if (dst[q]) QB_CUDA_TRY(cudaMemcpy2DAsync(dst[q], sizeof(double) * npad, src[q], sizeof(double) * n, sizeof(double) * n,
                                                q == 2 ? 1 : kk, cudaMemcpyDeviceToHost, d.s));
  }
  QB_CUDA_TRY(cudaMemcpyAsync(L, dL, sizeof(double) * npad * npad, cudaMemcpyDeviceToHost, d.s));
  QB_CUDA_TRY(cudaStreamSynchronize(d.s));
  for (int r = 0; r < passes; r++) info[r] = inf[r];
  return 0;
}
