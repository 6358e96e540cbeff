// engine.cuh -- device-resident state of one QPALM workspace and the kernels' host-side launchers.
//
// One Engine per QPALMWorkspace (hung off work->solver->LD).  Everything the inner iteration touches
// lives in HBM for the lifetime of the workspace:
//   A    sparse:  CSR (rows, for A*x and for gathering rows of A) + CSC (columns, for A'*y), int32 indices
//        dense :  At = A' column-major n x m (ld n): A*x is a per-column dot, A'*y a row-parallel GEMV,
//                 and the columns of the reference's At_sqrt_sigma are contiguous
//   Q    sparse:  full symmetric CSR expanded from the stored lower triangle;  dense: n x n column-major
//   H    npad x npad column-major, lower triangle: Q + A_J' Sigma_J A_J for the recorded (activeH, sigmaH)
//   L    npad x npad column-major, lower triangle: Cholesky factor of H + I/gamma (+ identity pad)
//   vectors of length n / m / 2m; a block of reduction partials and a 64-double scalar block that is
//   copied to pinned host memory once per iteration (the only host<->device sync of an iteration).
#pragma once
#include "common.cuh"
#include "dense.cuh"
#include "sparse.cuh"

namespace qb {

// indices into the per-iteration scalar block (device -> pinned host, one copy per iteration)
enum Scalar {
  S_PRI_RES = 0,     // max |Einv * pri_res|
  S_PRI_RES_RAW,     // max |pri_res|                    (update_sigma)
  S_NORM_AX,         // max |Einv * Ax|
  S_NORM_Z,          // max |Einv * z|
  S_NORM_EDY,        // max |E * (yh - y)|               (primal infeasibility)
  S_OOB,             // bmax' max(dy,0) + bmin' min(dy,0)
  S_ADX_MAX,         // max over rows with finite bmax of Einv*Ad   (dual infeasibility)
  S_ADX_MIN,         // min over rows with finite bmin of Einv*Ad
  S_DUA_RES,         // max |Dinv (dphi - (x-x0)/gamma)|  (not yet times cinv)
  S_DUA2_RES,        // max |Dinv dphi|
  S_NORM_QX, S_NORM_Q, S_NORM_ATYH,
  S_NORM_ATDY,       // max |Dinv (Atyh - Aty)|
  S_NORM_DDX,        // max |D (x - x_prev)|
  S_DXDX, S_DXQDX, S_QDX,
  S_ETA, S_BETA,     // d'Qd, d'df
  S_LS_A, S_LS_B,    // line-search a0, b0 partial sums over J
  S_TAU,
  S_OBJ,             // objective sum
  S_NB_ACTIVE, S_NB_ENTER, S_NB_LEAVE, S_NL, S_NB_SIGMA_CHANGED, S_INFO,
  S_TMP0, S_TMP1, S_TMP2, S_TMP3, S_TMP4, S_TMP5, S_TMP6, S_TMP7,
  S_L0, S_L1, S_L2, S_L3, S_L4, S_L5, S_L6, S_L7, S_L8, S_L9, S_LMAX,
  S_COUNT = 64
};

struct KktEngine;            // kkt.cu: the KKT factorization path of the Newton step (SURVEY 8 row f3)

struct SparseDev {           // CSR or CSC, int32 indices
  int rows = 0, cols = 0; long long nnz = 0;
  int *p = nullptr, *i = nullptr; double *x = nullptr;
};

struct Engine {
  int device = 0;
  cudaStream_t stream = nullptr;
  // one zero-filled slab for the ~80 iterate / work vectors (a cudaMalloc + cudaMemset per vector cost 113 ms of the
  // setup at m = 359k); buffers carved from it are not freed individually
  char *arena = nullptr;
  size_t arena_cap = 0, arena_off = 0;
  int n = 0, m = 0, npad = 0, ld = 0;
  bool A_dense = false, Q_dense = false;
  // row-sharding (shard.cu): this rank holds constraint rows [m_lo, m_lo + m_loc) of A in `At` (n x m_loc); vectors of
  // length m are replicated and padded to sh_world * m_cap entries so that the in-place allgather blocks are equal-sized
  int sh_world = 1, sh_rank = 0, m_lo = 0, m_loc = 0, m_cap = 0;
  SparseDev A_csr, A_csc, Q_csr;      // sparse forms
  double *At = nullptr;               // dense A' (n x m, ld n)
  double *Qd = nullptr;               // dense Q  (n x n, ld n), full symmetric
  // problem vectors (scaled)
  double *q = nullptr, *bmin = nullptr, *bmax = nullptr;
  double *D = nullptr, *Dinv = nullptr, *E = nullptr, *Einv = nullptr;
  double c = 1.0, cinv = 1.0;
  int scaling = 0;
  // iterates and work vectors
  double *x = nullptr, *y = nullptr, *Ax = nullptr, *Qx = nullptr, *Aty = nullptr, *x_prev = nullptr, *x0 = nullptr;
  double *sigma = nullptr, *sigma_inv = nullptr, *sqrt_sigma = nullptr, *sig_fac = nullptr;
  double *Axys = nullptr, *z = nullptr, *pri_res = nullptr, *pri_res_in = nullptr, *yh = nullptr, *Atyh = nullptr;
  double *df = nullptr, *dphi = nullptr, *d = nullptr, *Qdv = nullptr, *Ad = nullptr;
  double *delta_y = nullptr, *delta_x = nullptr, *tmp_n = nullptr, *tmp_m = nullptr, *tmp_n2 = nullptr;
  double *vpad = nullptr;             // npad-length rhs/solution of the Newton system
  int *active = nullptr, *active_old = nullptr, *active_cand = nullptr, *enter = nullptr, *leave = nullptr, *changed = nullptr;
  int *list_pos = nullptr, *list_neg = nullptr;  // refactor diff lists
  double *w_pos = nullptr, *w_neg = nullptr;     // per-list-entry column scale
  int *activeH = nullptr; double *sigmaH = nullptr; bool H_valid = false;
  // line search
  unsigned long long *ls_key[2] = {nullptr, nullptr};
  unsigned int *ls_val[2] = {nullptr, nullptr};
  double *ls_da = nullptr, *ls_db = nullptr;      // per-breakpoint toggle values (indexed by original idx)
  unsigned int *rs_hist = nullptr; int rs_tiles = 0;
  // Newton system
  double *H = nullptr, *L = nullptr, *invdiag = nullptr, *W = nullptr, *LQ = nullptr, *invdiagQ = nullptr;
  int wcols = 0;                      // columns of the gather panel W (multiple of 16)
  // sparse Newton system (sparse.cuh): supernodal factor instead of the dense H / L when the Schur complement stays sparse
  SparseChol *sp = nullptr;
  double *spL = nullptr, *spLQ = nullptr;   // numeric factors in the panel layout (Newton system; Q alone for the dual objective)
  // KKT path (kkt.cu): when set, the Newton direction comes from the quasi-definite augmented system instead of the Schur
  // complement; the factor is current for (active, sigma, gamma) iff kkt_valid
  KktEngine *kkt = nullptr;
  bool kkt_valid = false;
  double *ud_coef = nullptr;
  // reductions / scalars
  double *partials = nullptr; int partial_blocks = 0;
  double *gemv_partials = nullptr; int gemv_splits = 0;
  double *scal_dev = nullptr, *scal_host = nullptr;   // S_COUNT doubles each (host pinned)
  int *info_dev = nullptr, *info_host = nullptr;   // factorization status (device / pinned host mirror, copied with the scalar block)
  // statistics (QPALMB200Stats)
  long long launches0 = 0;
  long long n_inner = 0, n_outer = 0, n_refactor = 0, refactor_active_sum = 0, n_updown = 0, updown_rank_sum = 0, n_spmv = 0, n_sigma_update = 0, sigma_update_rank_sum = 0;
  double alg_bytes = 0, dense_flops = 0, ms_factor = 0, ms_updown = 0, ms_total = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, evs0 = nullptr, evs1 = nullptr;
  // tunables
  int updown_max_rank = 8;           // one sweep of the rank-k kernel
  bool updown_gen_ok = true;         // cleared when the generator-form update pass (updown_gen.cu) is unavailable on this device
  double updown_gen_scale = 1.0;     // static cost model of the generator-form passes (api.cu prefer_updown): scale factor, QPALM_B200_UPDOWN_GEN_SCALE
  int updown_force = 0;              // QPALM_B200_UPDOWN_FORCE=1: bypass the cost model (tests)
  double last_updown_ms = -1.0;      // CUDA-event time of the most recent update/downdate call (sparse cost model)
  double last_refactor_ms = -1.0;    // CUDA-event time of the most recent refactorisation (cost model input)
  //   // device cost model: beyond this a (incremental) refactorisation is cheaper (DESIGN.md)
};

// ---- construction -------------------------------------------------------------------------------
// Host CSC (int64) -> device.  A: m x n general; Q: n x n, only row >= col entries are read.
int engine_create(Engine **out, int n, int m, const long long *Ap, const long long *Ai, const double *Ax,
                  const long long *Qp, const long long *Qi, const double *Qx,
                  const double *q, const double *bmin, const double *bmax, bool need_LQ,
                  int newton_override = 0 /* 0: density heuristics (or QPALM_B200_NEWTON), 1: dense factor, 2: supernodal */);
void engine_destroy(Engine *e);

// ---- setup-time operations ------------------------------------------------------------------------
int engine_ruiz_scale(Engine *e, int iters, double *c_out);     // scale_data with Qx = 0 (setup)
int engine_ruiz_rescale(Engine *e, int iters, double *c_out);   // re-entry from qpalm_update_settings (uses e->Qx)
int engine_download_scaled_data(Engine *e, double *A_x_csc, double *Q_x_csc_lower_pattern,
                                const long long *Qp, const long long *Qi);

// ---- products -------------------------------------------------------------------------------------
int spmv_A(Engine *e, const double *x, double *y);     // y = A x   (m)
int spmv_At(Engine *e, const double *x, double *y);    // y = A' x  (n)
int spmv_Q(Engine *e, const double *x, double *y);     // y = Q x   (n)

// ---- generic small helpers ------------------------------------------------------------------------
int dev_alloc(void **p, size_t bytes);
int vec_copy(Engine *e, const double *src, double *dst, int len);
int vec_set(Engine *e, double *dst, double v, int len);
int vec_axpy(Engine *e, double a, const double *x, double *y, int len);   // y += a x
int vec_scale(Engine *e, double a, double *x, int len);
int vec_ewprod(Engine *e, const double *a, const double *b, double *c, int len);
int upload(Engine *e, double *dst, const double *src, int len);
int download(Engine *e, double *dst, const double *src, int len);
int download_int(Engine *e, long long *dst, const int *src, int len);   // widens to int64
int sync_scalars(Engine *e);   // scal_dev -> scal_host, stream synchronize

// ---- row-sharding collectives (shard.cu; no-ops on a single GPU) ------------------------------------
int shard_world();
int shard_rank();
int shard_allreduce(const double *send, double *recv, size_t count, bool max_op, cudaStream_t s);
int shard_allgather(double *buf, size_t count_per_rank, cudaStream_t s);

// ---- iteration steps (each: a handful of fused kernels, no host sync) ------------------------------
int step_residuals(Engine *e, bool proximal, double gamma, double tau);  // a3 + a4 + a5 counts + a14 reductions
int step_compact_lists(Engine *e);                                       // ordered enter[] / leave[] lists
int step_newton_refactor(Engine *e, bool with_constraints, bool from_scratch, double beta, int nb_active);
int step_newton_updown(Engine *e, int nb_enter, int nb_leave);
bool use_updown_gen(const Engine *e);
int step_newton_solve(Engine *e);                                        // d = -(L L')^{-1} dphi
int step_commit_active(Engine *e);                                       // active_old <- active
int step_linesearch(Engine *e, bool proximal, double gamma);             // Qd, Ad, eta, beta, tau (on device)
int step_update_iterate(Engine *e);                                      // x, Qx, Ax, Qd, Ad with tau from device
int step_update_sigma(Engine *e, double theta, double delta, double sigma_max, double sqrt_sigma_max);
int step_objective(Engine *e, bool proximal, double gamma);              // S_OBJ
int step_gershgorin_AtSA(Engine *e, double *ub_host);                    // boost_gamma's bound (syncs)
int step_dual_objective(Engine *e, double *val_host);                    // needs LQ (syncs)
int factor_Q_for_dual(Engine *e);
int initialize_sigma(Engine *e, double sigma_init);
int sigma_changed_update(Engine *e, int nb_changed);                     // ldlupdate_sigma_changed
int scale_Q_values(Engine *e, double cc, bool use_D);                    // Q <- cc * (D Q D or Q)
int gather_rows_public(Engine *e, const int *list, const double *scale, bool scale_by_row, int cnt, int kpad);                       // iteration.c:50-84 (syncs once)

// ---- line-search building blocks (also used by the operator ABI) -----------------------------------
int linesearch_device(Engine *e, int m, const double *Ad, const double *Ax, const double *y, const double *sigma,
                      const double *sqrt_sigma, const double *bmin, const double *bmax);  // eta/beta in scal_dev

// ---- KKT factorization path (kkt.cu; newton.c:22-95, solver_interface.c:20-70,119-247) ---------------
bool kkt_heuristic_prefers_kkt(int n, int m, const long long *Ap, const long long *Ai, const long long *Qp, const long long *Qi);
int kkt_create(KktEngine **out, Engine *e, int n, int m, const long long *Ap, const long long *Ai, const long long *Qp, const long long *Qi);
void kkt_destroy(KktEngine *K);
int kkt_refactor(KktEngine *K, Engine *e, double beta);   // values for the committed active set + L S L'
int kkt_solve(KktEngine *K, Engine *e);                   // e->d from K z = [-dphi; 0], with iterative refinement
long long kkt_factor_nnz(const KktEngine *K);
long long kkt_factor_count(const KktEngine *K);
long long kkt_refine_count(const KktEngine *K);
void kkt_last_norms(const KktEngine *K, double out2[2]);   // {|res|inf, ref} of the last residual kkt_solve formed

// ---- LOBPCG (nonconvex.c:29-168) ---------------------------------------------------------------------
int lobpcg_device(Engine *e, const double *x0_host, double *lambda_out, long long *iters_out);

}  // namespace qb
