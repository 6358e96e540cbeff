// api.cu -- the drop-in C API (include/qpalm_b200.h Part 1): host-side control flow of QPALM driving the
// device engine.  The control flow (outer/inner loop, tolerance schedule, gamma logic, refactor-vs-update
// decision) restates src/qpalm.c:401-736 and src/newton.c:96-118 of the reference; every numerical step
// is a kernel sequence in kernels.cu / dense.cu.  One host<->device synchronisation per iteration.
#include "../../include/qpalm_b200.h"
#include "engine.cuh"
#include <math.h>
#include <string.h>
#include <time.h>

using namespace qb;

#define c_max(a, b) (((a) > (b)) ? (a) : (b))
#define c_min(a, b) (((a) < (b)) ? (a) : (b))
#define c_absval(x) (((x) < 0) ? -(x) : (x))

static Engine *eng(const QPALMWorkspace *w) { return (Engine *)w->solver->LD; }

// ------------------------------------------------------------------------------------------------
// host helpers the reference also exports
// ------------------------------------------------------------------------------------------------
extern "C" void update_status(QPALMInfo *info, c_int v) {   // util.c:61-99
  info->status_val = v;
  const char *s = "unrecognised status value";
  switch (v) {
    case QPALM_SOLVED: s = "solved"; break;
    case QPALM_DUAL_TERMINATED: s = "dual terminated"; break;
    case QPALM_PRIMAL_INFEASIBLE: s = "primal infeasible"; break;
    case QPALM_DUAL_INFEASIBLE: s = "dual infeasible"; break;
    case QPALM_TIME_LIMIT_REACHED: s = "time limit exceeded"; break;
    case QPALM_MAX_ITER_REACHED: s = "maximum iterations reached"; break;
    case QPALM_UNSOLVED: s = "unsolved"; break;
    case QPALM_ERROR: s = "error"; break;
    default: fprintf(stderr, "ERROR in update_status: Unrecognised status value %ld\n", (long)v);
  }
  strcpy(info->status, s);
}

#define QP_EPRINT(...) do { fprintf(stderr, "ERROR in %s: ", __func__); fprintf(stderr, __VA_ARGS__); fprintf(stderr, "\n"); } while (0)

extern "C" c_int validate_data(const QPALMData *data) {   // validate.c:18-40
  if (!data) { QP_EPRINT("Missing data"); return FALSE; }
  for (size_t j = 0; j < data->m; j++)
    if (data->bmin[j] > data->bmax[j]) {
      QP_EPRINT("Lower bound at index %d is greater than upper bound: %.4e > %.4e", (int)j, data->bmin[j], data->bmax[j]);
      return FALSE;
    }
  return TRUE;
}

extern "C" c_int validate_settings(const QPALMSettings *s) {   // validate.c:43-221
  if (!s) { QP_EPRINT("Missing settings!"); return FALSE; }
#define BAD(cond, msg) if (cond) { QP_EPRINT(msg); return FALSE; }
  BAD(s->max_iter <= 0, "max_iter must be positive")
  BAD(s->inner_max_iter <= 0, "inner_max_iter must be positive")
  BAD(s->eps_abs < 0, "eps_abs must be nonnegative")
  BAD(s->eps_rel < 0, "eps_rel must be nonnegative")
  BAD((s->eps_rel == 0) && (s->eps_abs == 0), "at least one of eps_abs and eps_rel must be positive")
  BAD(s->eps_abs_in < 0, "eps_abs_in must be nonnegative")
  BAD(s->eps_rel_in < 0, "eps_rel_in must be nonnegative")
  BAD((s->eps_rel_in == 0) && (s->eps_abs_in == 0), "at least one of eps_abs_in and eps_rel_in must be positive")
  BAD(s->rho <= 0 || s->rho >= 1, "rho must be positive and smaller than 1")
  BAD(s->eps_prim_inf < 0, "eps_prim_inf must be nonnegative")
  BAD(s->eps_dual_inf < 0, "eps_dual_inf must be nonnegative")
  BAD(s->theta > 1, "theta must be smaller than ot equal 1")
  BAD(s->delta <= 1, "delta must be greater than 1")
  BAD(s->sigma_max <= 0, "sigma_max must be positive")
  BAD(s->sigma_init <= 0, "sigma_init must be positive")
  BAD((s->proximal != 0) && (s->proximal != 1), "proximal must be either 0 or 1")
  BAD(s->gamma_init <= 0, "gamma_init must be positive")
  BAD(s->gamma_upd < 1, "gamma update factor must be greater than or equal to 1")
  BAD(s->gamma_max < s->gamma_init, "gamma max must be greater than or equal to gamma")
  BAD(s->scaling < 0, "scaling must be greater than or equal to zero")
  BAD((s->nonconvex != 0) && (s->nonconvex != 1), "nonconvex must be either 0 or 1")
  BAD((s->warm_start != 0) && (s->warm_start != 1), "warm_start must be either 0 or 1")
  BAD((s->verbose != 0) && (s->verbose != 1), "verbose must be either 0 or 1")
  BAD(s->print_iter <= 0, "print_iter must be positive")
  BAD(s->reset_newton_iter <= 0, "reset_newton_iter must be positive")
  BAD((s->enable_dual_termination != 0) && (s->enable_dual_termination != 1), "enable_dual_termination must be either 0 or 1")
#undef BAD
  return TRUE;
}

extern "C" void qpalm_set_default_settings(QPALMSettings *s) {   // qpalm.c:39-70, constants.h:65-116
  s->max_iter = 10000; s->inner_max_iter = 100; s->eps_abs = 1e-4; s->eps_rel = 1e-4;
  s->eps_abs_in = 1; s->eps_rel_in = 1; s->rho = 0.1; s->eps_prim_inf = 1e-5; s->eps_dual_inf = 1e-5;
  s->theta = 0.25; s->delta = 100; s->sigma_max = 1e9; s->sigma_init = 2e1; s->proximal = TRUE;
  s->gamma_init = 1e7; s->gamma_upd = 10; s->gamma_max = 1e7; s->scaling = 10; s->nonconvex = FALSE;
  s->verbose = TRUE; s->print_iter = 1; s->warm_start = FALSE; s->reset_newton_iter = 10000;
  s->enable_dual_termination = FALSE; s->dual_objective_limit = QPALM_INFTY; s->time_limit = QPALM_INFTY;
  s->ordering = 0; s->factorization_method = FACTORIZE_KKT_OR_SCHUR; s->max_rank_update = 160;
  s->max_rank_update_fraction = 0.1;
}

// ------------------------------------------------------------------------------------------------
// timers (util.c:283-303)
// ------------------------------------------------------------------------------------------------
static void tic(QPALMWorkspace *w) {
  struct timespec t; clock_gettime(CLOCK_MONOTONIC, &t);
  w->timer->tic_sec = t.tv_sec; w->timer->tic_nsec = t.tv_nsec;
}
static double toc(QPALMWorkspace *w) {
  struct timespec t; clock_gettime(CLOCK_MONOTONIC, &t);
  return (double)(t.tv_sec - w->timer->tic_sec) + 1e-9 * (double)(t.tv_nsec - w->timer->tic_nsec);
}

static solver_sparse *csc_copy_host(const solver_sparse *S) {
  solver_sparse *C = (solver_sparse *)calloc(1, sizeof(solver_sparse));
  const c_int *Sp = (const c_int *)S->p;
  const size_t nnz = (size_t)Sp[S->ncol];
  *C = *S;
  C->p = malloc((S->ncol + 1) * sizeof(c_int)); C->i = malloc((nnz + 1) * sizeof(c_int)); C->x = malloc((nnz + 1) * sizeof(c_float));
  memcpy(C->p, S->p, (S->ncol + 1) * sizeof(c_int)); memcpy(C->i, S->i, nnz * sizeof(c_int)); memcpy(C->x, S->x, nnz * sizeof(c_float));
  C->nzmax = nnz ? nnz : 1; C->nz = NULL; C->z = NULL;
  return C;
}
static void csc_free_host(solver_sparse *S) { if (S) { free(S->p); free(S->i); free(S->x); free(S); } }

// ------------------------------------------------------------------------------------------------
// qpalm_setup (qpalm.c:73-319)
// ------------------------------------------------------------------------------------------------
extern "C" QPALMWorkspace *qpalm_setup(const QPALMData *data, const QPALMSettings *settings) {
  if (!validate_data(data)) { QP_EPRINT("Data validation returned failure"); return NULL; }
  if (!validate_settings(settings)) { QP_EPRINT("Settings validation returned failure"); return NULL; }
  const size_t n = data->n, m = data->m;
  if (n > 2000000000ull || m > 1000000000ull) { QP_EPRINT("problem dimensions exceed the int32 device index range"); return NULL; }

  QPALMWorkspace *work = (QPALMWorkspace *)calloc(1, sizeof(QPALMWorkspace));
  work->timer = (QPALMTimer *)calloc(1, sizeof(QPALMTimer));
  tic(work);
  work->settings = (QPALMSettings *)malloc(sizeof(QPALMSettings));
  *work->settings = *settings;
  work->sqrt_delta = sqrt(settings->delta);
  work->gamma = settings->gamma_init;
  work->solver = (QPALMSolver *)calloc(1, sizeof(QPALMSolver));
  work->data = (QPALMData *)calloc(1, sizeof(QPALMData));
  work->data->n = n; work->data->m = m; work->data->c = data->c;
  auto vcopy = [](const c_float *a, size_t len) { c_float *b = (c_float *)malloc((len + 1) * sizeof(c_float)); memcpy(b, a, len * sizeof(c_float)); return b; };
  work->data->bmin = vcopy(data->bmin, m); work->data->bmax = vcopy(data->bmax, m); work->data->q = vcopy(data->q, n);
  // Host copies of the matrices are kept only for modest sizes (they are never read by the solver; the
  // device holds the scaled working copies).  The reference keeps scaled CHOLMOD copies here.
  // (work->data->A / Q stay NULL above 2^24 stored entries: a caller that reads the workspace must not expect them)
  const c_int *Ap = (m > 0 && data->A) ? (const c_int *)data->A->p : nullptr, *Qp = (const c_int *)data->Q->p;
  if ((size_t)(Ap ? Ap[n] : 0) + (size_t)Qp[n] <= (size_t)1 << 24 && data->A) {
    work->data->A = csc_copy_host(data->A); work->data->A->stype = 0;
    work->data->Q = csc_copy_host(data->Q);
  }
#define VN(f) work->f = (c_float *)calloc(n + 1, sizeof(c_float))
#define VM(f) work->f = (c_float *)calloc(m + 1, sizeof(c_float))
#define V2M(f) work->f = (c_float *)calloc(2 * m + 1, sizeof(c_float))
  VN(x); VM(y); VM(Ax); VN(Qx); VN(x_prev); VN(Aty); VN(x0); VM(temp_m); VN(temp_n); VM(sigma); VM(sigma_inv);
  VM(z); VM(Axys); VM(pri_res); VM(pri_res_in); VN(df); VN(xx0); VN(dphi); VN(dphi_prev); VM(sqrt_sigma);
  V2M(delta); V2M(alpha); V2M(delta2); V2M(delta_alpha); V2M(temp_2m);
  work->s = (array_element *)calloc(2 * m + 1, sizeof(array_element));
  work->index_L = (c_int *)calloc(2 * m + 1, sizeof(c_int)); work->index_P = (c_int *)calloc(2 * m + 1, sizeof(c_int));
  work->index_J = (c_int *)calloc(2 * m + 1, sizeof(c_int));
  VM(delta_y); VN(Atdelta_y); VN(delta_x); VN(Qdelta_x); VM(Adelta_x);
  VN(neg_dphi); VN(d); VN(Qd); VM(Ad); VM(yh); VN(Atyh); VN(D_temp); VM(E_temp);
#undef VN
#undef VM
#undef V2M
  work->initialized = FALSE;
  {   // the reference wraps these work vectors in cholmod_dense headers (qpalm.c:190-250) and its test-suite reaches them
      // through work->solver->Qd etc.: same layout (cholmod_core.h:1894-1905), the x pointer aliases the host mirror
    struct DenseHdr { size_t nrow, ncol, nzmax, d; void *x, *z; int xtype, dtype; };
    auto wrap = [](c_float *x, size_t len) { DenseHdr *h = (DenseHdr *)calloc(1, sizeof(DenseHdr)); h->nrow = len; h->ncol = 1; h->nzmax = len; h->d = len; h->x = x; h->xtype = 1; return (void *)h; };
    work->solver->neg_dphi = wrap(work->neg_dphi, n); work->solver->d = wrap(work->d, n); work->solver->Qd = wrap(work->Qd, n);
    work->solver->Ad = wrap(work->Ad, m); work->solver->yh = wrap(work->yh, m); work->solver->Atyh = wrap(work->Atyh, n);
    work->solver->E_temp = wrap(work->E_temp, m); work->solver->D_temp = wrap(work->D_temp, n);
  }
  work->solver->factorization_method = FACTORIZE_SCHUR;   // solver_interface.c:72-73
  work->solver->active_constraints = (c_int *)calloc(m + 1, sizeof(c_int));
  work->solver->active_constraints_old = (c_int *)calloc(m + 1, sizeof(c_int));
  work->solver->enter = (c_int *)calloc(m + 1, sizeof(c_int));
  work->solver->leave = (c_int *)calloc(m + 1, sizeof(c_int));
  work->solver->reset_newton = TRUE;
  work->solution = (QPALMSolution *)calloc(1, sizeof(QPALMSolution));
  work->solution->x = (c_float *)calloc(n + 1, sizeof(c_float));
  work->solution->y = (c_float *)calloc(m + 1, sizeof(c_float));
  work->info = (QPALMInfo *)calloc(1, sizeof(QPALMInfo));

  Engine *e = nullptr;
  // factorization_method (constants.h: 0 KKT, 1 SCHUR, 2 KKT_OR_SCHUR): KKT is honoured (kkt.cu); SCHUR and the default
  // KKT_OR_SCHUR take the Schur path like the reference's CHOLMOD build, except that sparse problems whose Schur complement
  // fills in fall to the KKT system by the reference's own criterion (engine_create)
  int rc = engine_create(&e, (int)n, (int)m, (const long long *)data->A->p, (const long long *)data->A->i, (const double *)data->A->x,
                         (const long long *)data->Q->p, (const long long *)data->Q->i, (const double *)data->Q->x,
                         data->q, data->bmin, data->bmax, settings->enable_dual_termination != 0,
                         settings->factorization_method == FACTORIZE_KKT ? 3 : (settings->factorization_method == FACTORIZE_SCHUR ? 5 : 0));
  if (rc) {
    QP_EPRINT("device engine creation failed (code %d); this library has no CPU fallback", rc);
    work->solver->LD = NULL;
    qpalm_cleanup(work);
    return NULL;
  }
  work->solver->LD = e;
  if (e->kkt) work->solver->factorization_method = FACTORIZE_KKT;

  if (settings->scaling) {
    work->scaling = (QPALMScaling *)calloc(1, sizeof(QPALMScaling));
    work->scaling->D = (c_float *)calloc(n + 1, sizeof(c_float)); work->scaling->Dinv = (c_float *)calloc(n + 1, sizeof(c_float));
    work->scaling->E = (c_float *)calloc(m + 1, sizeof(c_float)); work->scaling->Einv = (c_float *)calloc(m + 1, sizeof(c_float));
    double cc = 1.0;
    rc = engine_ruiz_scale(e, (int)settings->scaling, &cc);
    e->scaling = 1; e->c = cc; e->cinv = 1.0 / cc;
    work->scaling->c = cc; work->scaling->cinv = 1.0 / cc;
    rc |= download(e, work->scaling->D, e->D, (int)n); rc |= download(e, work->scaling->Dinv, e->Dinv, (int)n);
    rc |= download(e, work->scaling->E, e->E, (int)m); rc |= download(e, work->scaling->Einv, e->Einv, (int)m);
    rc |= download(e, work->data->q, e->q, (int)n); rc |= download(e, work->data->bmin, e->bmin, (int)m);
    rc |= download(e, work->data->bmax, e->bmax, (int)m);
    memcpy(work->D_temp, work->scaling->D, n * sizeof(c_float));
    if (rc) { QP_EPRINT("device scaling failed"); qpalm_cleanup(work); return NULL; }
  }
  if (work->settings->nonconvex) {   // set_settings_nonconvex, nonconvex.c:171-183
    c_float *x0 = (c_float *)malloc((n + 1) * sizeof(c_float));
    for (size_t i = 0; i < n; i++) x0[i] = (c_float)rand() / RAND_MAX;   // nonconvex.c:41-44 (unseeded rand)
    double lambda = 0; long long its = 0;
    rc = lobpcg_device(e, x0, &lambda, &its);
    free(x0);
    if (rc) { QP_EPRINT("device LOBPCG failed"); qpalm_cleanup(work); return NULL; }
    if (lambda < 0) {
      work->settings->proximal = TRUE;
      work->settings->gamma_init = 1 / c_absval(lambda);
      work->settings->gamma_max = work->settings->gamma_init;
      work->gamma_maxed = TRUE;
    } else work->settings->nonconvex = FALSE;
  }
  update_status(work->info, QPALM_UNSOLVED);
  work->info->solve_time = 0.0; work->info->run_time = 0.0;
  work->info->setup_time = toc(work);
  return work;
}

// ------------------------------------------------------------------------------------------------
// qpalm_warm_start (qpalm.c:322-399)
// ------------------------------------------------------------------------------------------------
extern "C" void qpalm_warm_start(QPALMWorkspace *work, c_float *x_ws, c_float *y_ws) {
  Engine *e = eng(work);
  work->gamma = work->settings->gamma_init;
  if (work->info->status_val != QPALM_UNSOLVED) work->info->setup_time = 0;
  tic(work);
  const int n = (int)work->data->n, m = (int)work->data->m;
  if (x_ws != NULL) {
    for (int i = 0; i < n; i++) work->x[i] = x_ws[i];
    if (work->settings->scaling) for (int i = 0; i < n; i++) work->x[i] = work->x[i] * work->scaling->Dinv[i];
    upload(e, e->x, work->x, n);
    vec_copy(e, e->x, e->x0, n); vec_copy(e, e->x, e->x_prev, n);
    spmv_Q(e, e->x, e->Qdv);
    vec_copy(e, e->Qdv, e->Qx, n);
    if (work->settings->proximal) vec_axpy(e, 1 / work->settings->gamma_init, e->x, e->Qx, n);   // Qx = Qd + x/gamma
    spmv_A(e, e->x, e->Ad);
    vec_copy(e, e->Ad, e->Ax, m);
    step_objective(e, work->settings->proximal != 0, work->gamma);
    sync_scalars(e);
    double obj = e->scal_host[S_OBJ];
    if (work->settings->scaling) obj *= work->scaling->cinv;
    work->info->objective = obj + work->data->c;
  } else {
    vec_set(e, e->x, 0., n); vec_set(e, e->x_prev, 0., n); vec_set(e, e->x0, 0., n); vec_set(e, e->Qx, 0., n);
    vec_set(e, e->Ax, 0., m);
    vec_set(e, e->Qdv, 0., n); vec_set(e, e->Ad, 0., m); vec_set(e, e->d, 0., n);
    work->info->objective = 0.0;
  }
  if (y_ws != NULL) {
    for (int i = 0; i < m; i++) work->y[i] = y_ws[i];
    if (work->settings->scaling) for (int i = 0; i < m; i++) { work->y[i] = work->y[i] * work->scaling->Einv[i]; work->y[i] *= work->scaling->c; }
    upload(e, e->y, work->y, m);
  } else vec_set(e, e->y, 0., m);
  initialize_sigma(e, work->settings->sigma_init);
  work->sqrt_sigma_max = sqrt(work->settings->sigma_max);
  cudaStreamSynchronize(e->stream);
  work->initialized = TRUE;
  work->info->setup_time += toc(work);
}

// ------------------------------------------------------------------------------------------------
// host mirrors
// ------------------------------------------------------------------------------------------------
static void mirror_iterates(QPALMWorkspace *work) {
  Engine *e = eng(work);
  const int n = e->n, m = e->m;
  download(e, work->x, e->x, n); download(e, work->y, e->y, m); download(e, work->Ax, e->Ax, m); download(e, work->Qx, e->Qx, n);
  download(e, work->Aty, e->Aty, n); download(e, work->x_prev, e->x_prev, n); download(e, work->x0, e->x0, n);
  download(e, work->sigma, e->sigma, m); download(e, work->sigma_inv, e->sigma_inv, m); download(e, work->sqrt_sigma, e->sqrt_sigma, m);
  download(e, work->Axys, e->Axys, m); download(e, work->z, e->z, m); download(e, work->pri_res, e->pri_res, m);
  download(e, work->pri_res_in, e->pri_res_in, m); download(e, work->yh, e->yh, m); download(e, work->Atyh, e->Atyh, n);
  download(e, work->df, e->df, n); download(e, work->dphi, e->dphi, n); download(e, work->d, e->d, n);
  download(e, work->Qd, e->Qdv, n); download(e, work->Ad, e->Ad, m);
  for (int i = 0; i < n; i++) work->neg_dphi[i] = -work->dphi[i];
  download_int(e, (long long *)work->solver->active_constraints, e->active, m);
  download_int(e, (long long *)work->solver->active_constraints_old, e->active_old, m);
}

static double objective_now(QPALMWorkspace *work) {
  Engine *e = eng(work);
  step_objective(e, work->settings->proximal != 0, work->gamma);
  sync_scalars(e);
  double obj = e->scal_host[S_OBJ];
  if (work->settings->scaling) obj *= work->scaling->cinv;
  return obj + work->data->c;
}

static void store_solution(QPALMWorkspace *work) {   // termination.c:242-252
  Engine *e = eng(work);
  const int n = e->n, m = e->m;
  mirror_iterates(work);
  if (work->settings->scaling) {
    for (int i = 0; i < n; i++) work->solution->x[i] = work->x[i] * work->scaling->D[i];
    for (int i = 0; i < m; i++) { work->yh[i] *= work->scaling->cinv; work->solution->y[i] = work->yh[i] * work->scaling->E[i]; }
  } else {
    memcpy(work->solution->x, work->x, n * sizeof(c_float)); memcpy(work->solution->y, work->yh, m * sizeof(c_float));
  }
  work->info->objective = objective_now(work);
}

static void finish(QPALMWorkspace *work, c_int iter, c_int iter_out) {
  Engine *e = eng(work);
  cudaEventRecord(e->ev1, e->stream);
  cudaEventSynchronize(e->ev1);
  float ms = 0; cudaEventElapsedTime(&ms, e->ev0, e->ev1); e->ms_total += ms;
  work->info->iter = iter; work->info->iter_out = iter_out;
  work->info->solve_time = toc(work);
  work->info->run_time = work->info->setup_time + work->info->solve_time;
  work->initialized = FALSE;
  work->tau = e->scal_host[S_TAU];
}

static double dual_objective_now(QPALMWorkspace *work) {   // iteration.c:272-299
  double v = 0;
  step_dual_objective(eng(work), &v);
  if (work->settings->scaling) v *= work->scaling->cinv;
  return v + work->data->c;
}

// pending CUDA-event timing of the last refactorisation / update sweep (events complete at the next sync)
struct Pending { int kind; };   // 0 none, 1 factor, 2 updown
static void collect(Engine *e, Pending &p) {
  if (!p.kind) return;
  float ms = 0;
  if (cudaEventElapsedTime(&ms, e->evs0, e->evs1) == cudaSuccess) {
    if (p.kind == 1) { e->ms_factor += ms; e->last_refactor_ms = ms; } else { e->ms_updown += ms; e->last_updown_ms = ms; }
  }
  p.kind = 0;
}

__global__ void k_recompute_active(int m, const double *__restrict__ Ax, const double *__restrict__ y, const double *__restrict__ sigma,
                                   const double *__restrict__ bmin, const double *__restrict__ bmax, const int *__restrict__ old,
                                   double *Axys, int *active, double *scal) {
  // qpalm.c:614-618: Axys = Ax + y./sigma ; set_active_constraints ; set_entering_leaving_constraints (counts only)
  __shared__ int cnt[3];
  if (threadIdx.x < 3) cnt[threadIdx.x] = 0;
  __syncthreads();
  int na = 0, ne = 0, nl = 0;
  for (int i = threadIdx.x; i < m; i += blockDim.x) {
    const double t = y[i] / sigma[i];
    const double a = Ax[i] + t;
    Axys[i] = a;
    const int act = (a <= bmin[i]) || (a >= bmax[i]);
    active[i] = act;
    na += act; ne += act && !old[i]; nl += !act && old[i];
  }
  atomicAdd(&cnt[0], na); atomicAdd(&cnt[1], ne); atomicAdd(&cnt[2], nl);
  __syncthreads();
  if (threadIdx.x == 0) { scal[S_NB_ACTIVE] = cnt[0]; scal[S_NB_ENTER] = cnt[1]; scal[S_NB_LEAVE] = cnt[2]; }
}

static void update_gamma(QPALMWorkspace *work) {   // iteration.c:147-157
  Engine *e = eng(work);
  if (work->gamma < work->settings->gamma_max) {
    const c_float prev = work->gamma;
    work->gamma = c_min(work->gamma * work->settings->gamma_upd, work->settings->gamma_max);
    work->solver->reset_newton = TRUE;
    vec_axpy(e, 1 / work->gamma - 1 / prev, e->x, e->Qx, e->n);
  }
}

static void boost_gamma(QPALMWorkspace *work) {   // iteration.c:159-211
  Engine *e = eng(work);
  const c_float prev = work->gamma;
  if (work->solver->nb_active_constraints) {
    double ub = 0;
    step_gershgorin_AtSA(e, &ub);
    work->gamma = c_max(work->settings->gamma_max, 1e14 / ub);
    work->gamma_maxed = TRUE;
    work->solver->reset_newton = TRUE;   // the bound was formed in the factor's storage
  } else work->gamma = 1e12;
  if (prev != work->gamma) {
    vec_axpy(e, 1.0 / work->gamma - 1.0 / prev, e->x, e->Qx, e->n);
    const double tau = e->scal_host[S_TAU];
    vec_axpy(e, tau / work->gamma - tau / prev, e->d, e->Qdv, e->n);
    work->solver->reset_newton = TRUE;
  }
}

// Refactor-vs-update cost model (DESIGN.md section 4): the rank-k sweep is a chain of npad/32 dependent panel steps
// (~83 us each at n = 8000, measured on B200), a refactorisation is a panel chain plus DMMA-bound updates.  Dense
// factor: a static model, so the choice never depends on timing; sparse factor: the measured time of the last sweep
// against the last refactorisation.  Same matrix either way.
static bool prefer_updown(const Engine *e, int k) {
  if (k <= 0) return false;
  if (e->kkt) return false;   // KKT path: a changed row is rewritten and the system refactorised (kkt.cu)
  if (e->updown_max_rank == 0) return false;   // QPALM_B200_UPDOWN_MAX_RANK=0: always refactorise, whatever the update path
  if (use_updown_gen(e)) {   // generator-form passes, <= 32 ranks each (updown_gen.cu)
    if (e->updown_force) return true;
    // STATIC model again: per pass a chain of npad/128 block steps of the k-column triangular solve (step time set by the
    // 128 x 128 x k products of one SM), the tile-parallel apply pass over the factor, the small generator kernels and the
    // refresh of the inverted diagonal blocks.  Measured on B200, see DESIGN.md section 4.
    // pass time (ms) = a * (npad / 128) + b * (npad / 8064)^2 + c, fitted to the measured passes at npad = 1024 and 8064:
    //   <= 8 columns 0.11 / 0.48 ms, <= 16 columns 0.13 / 0.56 ms, <= 32 columns 0.17 / 0.95 ms
    const double nblk = e->npad / 128.0, sz = (e->npad / 8064.0) * (e->npad / 8064.0);
    const double pass8 = 0.0030 * nblk + 0.21 * sz + 0.085, pass16 = 0.0035 * nblk + 0.25 * sz + 0.09, pass32 = 0.0065 * nblk + 0.42 * sz + 0.12;
    const int full = k / 32, rem = k % 32;
    const double t_ud = e->updown_gen_scale * (full * pass32 + (rem > 16 ? pass32 : (rem > 8 ? pass16 : (rem > 0 ? pass8 : 0.0))));
    const double t_rf = (e->npad / 128.0) * 0.12 + ((double)e->n * e->n * e->n / 3.0) / 25e9;
    return t_ud < t_rf;
  }
  if (e->sh_world > 1) return false;   // row-sharded factor without the generator form: refactorise
  if (k > (e->sp ? 8 * e->updown_max_rank : e->updown_max_rank)) return false;
  if (e->updown_force) return true;
  if (e->sp) {
    // Sparse factor: a STATIC rule as well (round 1 compared measured times here, which made re-solves irreproducible).  A sweep
    // of <= 8 ranks is ONE CTA walking the union of the etree paths (k_ud_sweep), a refactorisation is ~3 launches per 32-column
    // block and level over all SMs; in every measurement kept (grid QPs n = 10^4 .. 9 10^4) the refactorisation won as soon as
    // more than one sweep was needed, so: a single sweep when the factor is small enough for one CTA to stream it quickly.
    const SparseCholInfo *I = sparse_chol_info(e->sp);
    return k <= 8 && I->nnzL <= 2000000;
  }
  // Dense factor: a STATIC model (no measured times: the choice must not depend on timing, or re-solves would not be
  // reproducible, tests/src/test_basic_qp.c:298-305).  With a single 128-column panel both paths are launch-bound and
  // cost a fraction of a millisecond: follow the reference's own choice (rank update) so that tiny ill-conditioned
  // problems (tests/src/test_dua_inf_qp.c) round alike.
  if (e->npad <= 128) return true;
  const double t_rf = (e->npad / 128.0) * 0.12 + ((double)e->n * e->n * e->n / 3.0) / 25e9;      // ms: panel chain + DMMA flops
  const double t_ud = (e->npad / 32.0) * (0.060 + 0.008 * k);                                   // ms, B200 (measured 83 us per 32-column panel step at n = 8000)
  return t_ud < t_rf;
}

// update_sigma (iteration.c:86-145)
static void update_sigma(QPALMWorkspace *work, Pending &pend) {
  Engine *e = eng(work);
  const QPALMSettings *st = work->settings;
  const size_t n = work->data->n, m = work->data->m;
  step_update_sigma(e, st->theta, st->delta, st->sigma_max, work->sqrt_sigma_max);
  sync_scalars(e);
  collect(e, pend);
  work->nb_sigma_changed = (c_int)e->scal_host[S_NB_SIGMA_CHANGED];
  // first_factorization is never set in the CHOLMOD build (SURVEY.md appendix C.3)
  if ((st->proximal && work->gamma < st->gamma_max) ||
      (work->nb_sigma_changed > c_min(st->max_rank_update_fraction * (n + m), 0.25 * st->max_rank_update))) {
    work->solver->reset_newton = TRUE;
  } else if (work->nb_sigma_changed == 0) {
  } else if (!prefer_updown(e, (int)work->nb_sigma_changed)) {
    // device cost model: beyond a few ranks a refactorisation is cheaper than sequential column sweeps
    // (same matrix either way; DESIGN.md "refactor vs update")
    work->solver->reset_newton = TRUE;
  } else {   // ldlupdate_sigma_changed (solver_interface.c:443-503)
    sigma_changed_update(e, (int)work->nb_sigma_changed);
    e->n_sigma_update++; e->sigma_update_rank_sum += work->nb_sigma_changed;
    pend.kind = 2;
  }
}

// ------------------------------------------------------------------------------------------------
// qpalm_solve (qpalm.c:401-736)
// ------------------------------------------------------------------------------------------------
extern "C" void qpalm_solve(QPALMWorkspace *work) {
  Engine *e = eng(work);
  QPALMSettings *st = work->settings;
  QPALMSolver *sv = work->solver;
  const size_t n = work->data->n, m = work->data->m;
  if (st->verbose) {
    printf("\n                 QPALM Version 1.0 (B200 engine)  \n\n");
    printf("Iter |   P. res   |   D. res   |  Stepsize  |  Objective \n");
    printf("==========================================================\n");
  }
  work->eps_abs_in = st->eps_abs_in; work->eps_rel_in = st->eps_rel_in;
  sv->reset_newton = TRUE;
  work->gamma = st->gamma_init;
  work->gamma_maxed = (FALSE || st->nonconvex);
  cudaMemsetAsync(e->active_old, 0, sizeof(int) * (m ? m : 1), e->stream);
  if (!work->initialized) qpalm_warm_start(work, NULL, NULL);
  tic(work);
  cudaEventRecord(e->ev0, e->stream);
  {
    double tau0 = work->tau;
    cudaMemcpyAsync(e->scal_dev + S_TAU, &tau0, sizeof(double), cudaMemcpyHostToDevice, e->stream);
    cudaStreamSynchronize(e->stream);
  }
  Pending pend{0};
  static const bool trace = getenv("QPALM_B200_TRACE") != nullptr;
  const bool prox0 = st->proximal != 0;
  (void)prox0;
  if (st->enable_dual_termination) {   // qpalm.c:459-472
    if (!e->LQ && !e->spLQ) { QP_EPRINT("enable_dual_termination must be set at qpalm_setup time"); update_status(work->info, QPALM_ERROR); return; }
    factor_Q_for_dual(e);
    work->info->dual_objective = dual_objective_now(work);
  } else work->info->dual_objective = QPALM_NULL;

  c_int iter, iter_out = 0, prev_iter = 0, no_change = 0;
  bool newton_factored = false;   // the previous iteration refactorised the Newton system: its status is in the next readback
  cudaMemsetAsync(e->info_dev, 0, sizeof(int), e->stream);   // (the factor of Q for the dual objective may have left a flag)
  c_float eps_k_abs = st->eps_abs_in, eps_k_rel = st->eps_rel_in, eps_k;
  const double *h = e->scal_host;
  const double BA = e->A_dense ? 8.0 * (double)m * (double)n : 12.0 * (double)(e->A_csr.nnz) + 4.0 * ((double)n + 1);
  const double BQ = e->Q_dense ? 8.0 * (double)n * ((double)n + 1) / 2 : 12.0 * (double)(e->Q_csr.nnz + (long long)n) / 2 + 4.0 * ((double)n + 1);

  for (iter = 0; iter < st->max_iter; iter++) {
    const bool proximal = st->proximal != 0;
    step_residuals(e, proximal, work->gamma, 0.0);
    if (sync_scalars(e)) { update_status(work->info, QPALM_ERROR); finish(work, iter, iter_out); return; }
    collect(e, pend);
    if (newton_factored && e->info_host[0] != 0) {
      // The last factorization met a non-positive pivot (H + I/gamma not numerically positive definite: an indefinite Q solved
      // with nonconvex = 0, or a singular Q without the proximal term).  The factor holds NaN from that column on, so every
      // later comparison would be false and the loop would run to max_iter on garbage: stop with an error instead.
      QP_EPRINT("the Newton system is not positive definite (non-positive pivot at column %d); set nonconvex / proximal", e->info_host[0] - 1);
      update_status(work->info, QPALM_ERROR);
      cudaMemsetAsync(e->info_dev, 0, sizeof(int), e->stream);
      e->info_host[0] = 0;
      finish(work, iter, iter_out);
      return;
    }
    work->tau = h[S_TAU];
    // ---- calculate_residuals_and_tolerances (termination.c:44-128) ----
    const double cinv = st->scaling ? work->scaling->cinv : 1.0;
    work->info->pri_res_norm = h[S_PRI_RES];
    work->info->dua_res_norm = h[S_DUA_RES] * (st->scaling ? cinv : 1.0);
    work->info->dua2_res_norm = h[S_DUA2_RES] * (st->scaling ? cinv : 1.0);
    // NB the scaled branch of the reference takes the norm over the first m entries of [Einv*Ax; Einv*z]
    // only (termination.c:99), i.e. |Einv*Ax|inf; kept as is.
    const double nrm_axz = st->scaling ? h[S_NORM_AX] : c_max(h[S_NORM_AX], h[S_NORM_Z]);
    work->eps_pri = st->eps_abs + st->eps_rel * nrm_axz;
    double max_norm = c_max(h[S_NORM_QX], c_max(h[S_NORM_Q], h[S_NORM_ATYH]));
    if (st->scaling) max_norm *= cinv;
    work->eps_dua = st->eps_abs + st->eps_rel * max_norm;
    work->eps_dua_in = work->eps_abs_in + work->eps_rel_in * max_norm;

    // ---- check_termination (termination.c:19-42) ----
    int terminated = 0;
    if ((work->info->pri_res_norm < work->eps_pri) && (work->info->dua_res_norm < work->eps_dua)) {
      update_status(work->info, QPALM_SOLVED);
      store_solution(work);
      terminated = 1;
    } else {
      const double eps_pinf = st->eps_prim_inf * h[S_NORM_EDY];   // is_primal_infeasible, termination.c:136-182
      const bool pinf = (eps_pinf != 0) && (h[S_NORM_ATDY] <= eps_pinf) && (h[S_OOB] <= -eps_pinf);
      if (pinf) {
        update_status(work->info, QPALM_PRIMAL_INFEASIBLE);
        mirror_iterates(work);
        download(e, work->delta_y, e->delta_y, (int)m);
        if (st->scaling) for (size_t i = 0; i < m; i++) { work->delta_y[i] *= work->scaling->cinv; work->delta_y[i] = work->scaling->E[i] * work->delta_y[i]; }
        terminated = 1;
      } else {
        const double eps_dinf = st->eps_dual_inf * h[S_NORM_DDX];   // is_dual_infeasible, termination.c:184-240
        bool dinf = false;
        if (eps_dinf != 0) {
          const bool blocked = (m > 0) && ((h[S_ADX_MAX] >= eps_dinf) || (h[S_ADX_MIN] <= -eps_dinf));
          if (!blocked) {
            const double cc = st->scaling ? work->scaling->c : 1.0;
            const double e2 = st->eps_dual_inf * st->eps_dual_inf;
            dinf = (h[S_DXQDX] <= -cc * e2 * h[S_DXDX]) || ((h[S_DXQDX] <= cc * e2 * h[S_DXDX]) && (h[S_QDX] <= -cc * eps_dinf));
          }
        }
        if (dinf) {
          update_status(work->info, QPALM_DUAL_INFEASIBLE);
          mirror_iterates(work);
          download(e, work->delta_x, e->delta_x, (int)n);
          if (st->scaling) for (size_t i = 0; i < n; i++) work->delta_x[i] = work->scaling->D[i] * work->delta_x[i];
          terminated = 1;
        }
      }
    }
    if (terminated) {
      finish(work, iter, iter_out);
      if (st->verbose) { printf("%4ld | %.4e | %.4e | %.4e | %.4e \n", (long)iter, work->info->pri_res_norm, work->info->dua_res_norm, work->tau, work->info->objective); printf("\nQPALM finished: %s, iterations %ld (outer %ld)\n", work->info->status, (long)iter, (long)iter_out); }
      return;
    } else if ((work->info->dua2_res_norm <= work->eps_dua_in) || (no_change == 3)) {   // qpalm.c:515
      no_change = 0;
      if (iter_out > 0 && work->info->pri_res_norm > work->eps_pri) update_sigma(work, pend);
      vec_copy(e, e->yh, e->y, (int)m); vec_copy(e, e->Atyh, e->Aty, (int)n);
      if (st->enable_dual_termination) {
        work->info->dual_objective = dual_objective_now(work);
        if (work->info->dual_objective > st->dual_objective_limit) {
          update_status(work->info, QPALM_DUAL_TERMINATED);
          store_solution(work);
          finish(work, iter, iter_out);
          return;
        }
      }
      work->eps_abs_in = c_max(st->eps_abs, st->rho * work->eps_abs_in);
      work->eps_rel_in = c_max(st->eps_rel, st->rho * work->eps_rel_in);
      if (st->nonconvex) {   // qpalm.c:586-609
        eps_k = eps_k_abs + eps_k_rel * nrm_axz;
        if (work->info->pri_res_norm < eps_k) {
          vec_copy(e, e->x, e->x0, (int)n);
          eps_k_abs = c_max(st->eps_abs, st->rho * eps_k_abs);
          eps_k_rel = c_max(st->eps_rel, st->rho * eps_k_rel);
        }
      } else if (st->proximal) {   // qpalm.c:612-630
        if (!work->gamma_maxed && iter_out > 0 && sv->nb_enter == 0 && sv->nb_leave == 0 && work->info->pri_res_norm < work->eps_pri) {
          if (m > 0) {
            QB_LAUNCH(k_recompute_active, 1, 1024, 0, e->stream, (int)m, e->Ax, e->y, e->sigma, e->bmin, e->bmax, e->active_old,
                      e->Axys, e->active, e->scal_dev);
          }
          sync_scalars(e);
          collect(e, pend);
          sv->nb_active_constraints = (c_int)h[S_NB_ACTIVE]; sv->nb_enter = (c_int)h[S_NB_ENTER]; sv->nb_leave = (c_int)h[S_NB_LEAVE];
          if (m == 0) { sv->nb_active_constraints = 0; sv->nb_enter = 0; sv->nb_leave = 0; }
          if (sv->nb_enter == 0 && sv->nb_leave == 0) boost_gamma(work); else update_gamma(work);
        } else update_gamma(work);
        vec_copy(e, e->x, e->x0, (int)n);
      }
      vec_copy(e, e->pri_res, e->pri_res_in, (int)m);
      iter_out++; prev_iter = iter; e->n_outer++;
      e->alg_bytes += 8.0 * (7.0 * m + 4.0 * n);
      if (st->verbose && (iter % st->print_iter) == 0) printf("%4ld | ---------------------------------------------------\n", (long)iter);
    } else if (iter == prev_iter + st->inner_max_iter) {   // qpalm.c:647-660
      no_change = 0;
      if (iter_out > 0 && work->info->pri_res_norm > work->eps_pri) update_sigma(work, pend);
      if (st->proximal) { update_gamma(work); if (!st->nonconvex) vec_copy(e, e->x, e->x0, (int)n); }
      vec_copy(e, e->pri_res, e->pri_res_in, (int)m);
      iter_out++; prev_iter = iter; e->n_outer++;
    } else {   // inner iteration, qpalm.c:662-678 -> update_primal_iterate (iteration.c:213-229)
      if (sv->nb_enter + sv->nb_leave) no_change = 0; else no_change++;
      if ((iter % st->reset_newton_iter) == 0) sv->reset_newton = TRUE;
      // ---- newton_set_direction (newton.c:17-120), SCHUR branch ----
      const int na = (m > 0) ? (int)h[S_NB_ACTIVE] : 0, ne = (m > 0) ? (int)h[S_NB_ENTER] : 0, nl = (m > 0) ? (int)h[S_NB_LEAVE] : 0;
      sv->nb_active_constraints = na; sv->nb_enter = ne; sv->nb_leave = nl;
      const double beta = st->proximal ? 1.0 / work->gamma : 0.0;
      const double rank_limit = c_min(st->max_rank_update_fraction * (double)(n + m), (double)st->max_rank_update);
      bool need_refactor = false, from_scratch = false, do_updown = false, factor_q = false;
      if (e->kkt) {   // FACTORIZE_KKT branch of newton_set_direction (newton.c:22-95)
        if (m > 0) cudaMemcpyAsync(e->active, e->active_cand, sizeof(int) * m, cudaMemcpyDeviceToDevice, e->stream);
        const bool refac = sv->reset_newton || !e->kkt_valid || (ne + nl) > 0;
        if (trace) fprintf(stderr, "[qpalm_b200 trace] iter %ld out %ld active %d enter %d leave %d -> KKT %s\n", (long)iter, (long)iter_out, na, ne, nl,
                           refac ? "refactor" : "reuse factor");
        newton_factored = refac;
        if (refac) { cudaMemsetAsync(e->info_dev, 0, sizeof(int), e->stream); kkt_refactor(e->kkt, e, beta); e->kkt_valid = true; pend.kind = 1; }
        kkt_solve(e->kkt, e);
        step_commit_active(e);
        sv->reset_newton = FALSE;
        step_linesearch(e, proximal, work->gamma);
        step_update_iterate(e);
        e->n_inner++;
        e->alg_bytes += 2.0 * BA + BQ + 8.0 * (38.0 * m + 26.0 * n);
        goto end_of_iteration;
      }
      // Beyond its rank limit the reference refactorises (newton.c:98-108: a cost heuristic for cholmod_updown on a CPU).  The
      // generator-form passes (updown_gen.cu) cost a fraction of a refactorisation, so the device cost model may still take the
      // update there -- the same matrix either way.  A zero limit (max_rank_update = 0: "always refactorise") is honoured.
      const bool over = (double)(ne + nl) > rank_limit;
      const bool over_but_update = over && !sv->reset_newton && na && rank_limit > 0 && use_updown_gen(e) && prefer_updown(e, ne + nl);
      if ((sv->reset_newton && na) || (over && !over_but_update)) { need_refactor = true; from_scratch = sv->reset_newton != 0; }
      else if (na) {
        if (ne + nl > 0) { if (over_but_update || prefer_updown(e, ne + nl)) do_updown = true; else need_refactor = true; }
      } else factor_q = true;
      if (trace) fprintf(stderr, "[qpalm_b200 trace] iter %ld out %ld active %d enter %d leave %d -> %s\n", (long)iter, (long)iter_out, na, ne, nl,
                         do_updown ? "rank update" : (need_refactor ? (from_scratch ? "refactor (scratch)" : "refactor (incremental H)") : (factor_q ? "factor Q" : "reuse factor")));
      if (do_updown) {
        step_compact_lists(e);   // commits active <- candidate and lists enter / leave
        int hinfo = 0;
        cudaMemsetAsync(e->info_dev, 0, sizeof(int), e->stream);
        step_newton_updown(e, ne, nl);
        cudaMemcpyAsync(&hinfo, e->info_dev, sizeof(int), cudaMemcpyDeviceToHost, e->stream);
        cudaStreamSynchronize(e->stream);
        pend.kind = 2; collect(e, pend);
        if (hinfo) { need_refactor = true; from_scratch = true; }   // downdate lost definiteness: rebuild
      } else if (m > 0) {
        cudaMemcpyAsync(e->active, e->active_cand, sizeof(int) * m, cudaMemcpyDeviceToDevice, e->stream);
      }
      newton_factored = need_refactor || factor_q;
      if (newton_factored) cudaMemsetAsync(e->info_dev, 0, sizeof(int), e->stream);
      if (need_refactor) { step_newton_refactor(e, true, from_scratch, beta, na); pend.kind = 1; }
      else if (factor_q) { step_newton_refactor(e, false, true, beta, 0); pend.kind = 1; }
      step_newton_solve(e);
      step_commit_active(e);
      sv->reset_newton = FALSE;
      // ---- exact_linesearch + iterate update ----
      step_linesearch(e, proximal, work->gamma);
      step_update_iterate(e);
      e->n_inner++;
      e->alg_bytes += 2.0 * BA + BQ + 8.0 * (38.0 * m + 26.0 * n);
      if (st->verbose && (iter % st->print_iter) == 0) {
        const double obj = objective_now(work);
        printf("%4ld | %.4e | %.4e | %.4e | %.4e \n", (long)iter, work->info->pri_res_norm, work->info->dua_res_norm, h[S_TAU], obj);
      }
    }
  end_of_iteration:
    const c_float now = work->info->setup_time + toc(work);   // qpalm.c:680-708
    if (now > st->time_limit) {
      update_status(work->info, QPALM_TIME_LIMIT_REACHED);
      sync_scalars(e);
      store_solution(work);
      finish(work, iter, iter_out);
      return;
    }
  }
  update_status(work->info, QPALM_MAX_ITER_REACHED);
  sync_scalars(e);
  store_solution(work);
  finish(work, iter, iter_out);
}

// ------------------------------------------------------------------------------------------------
// qpalm_update_* (qpalm.c:739-871)
// ------------------------------------------------------------------------------------------------
extern "C" void qpalm_update_settings(QPALMWorkspace *work, const QPALMSettings *settings) {
  if (!validate_settings(settings)) { QP_EPRINT("Settings validation returned failure"); update_status(work->info, QPALM_ERROR); return; }
  Engine *e = eng(work);
  const int n = e->n, m = e->m;
  if (work->settings->scaling > settings->scaling) {
    QP_EPRINT("Decreasing the number of scaling iterations is not allowed");
    update_status(work->info, QPALM_ERROR);
    return;
  } else if (work->settings->scaling < settings->scaling) {
    if (!work->scaling) {
      work->scaling = (QPALMScaling *)calloc(1, sizeof(QPALMScaling));
      work->scaling->D = (c_float *)calloc(n + 1, sizeof(c_float)); work->scaling->Dinv = (c_float *)calloc(n + 1, sizeof(c_float));
      work->scaling->E = (c_float *)calloc(m + 1, sizeof(c_float)); work->scaling->Einv = (c_float *)calloc(m + 1, sizeof(c_float));
      for (int i = 0; i < n; i++) work->scaling->D[i] = work->scaling->Dinv[i] = 1.0;
      for (int i = 0; i < m; i++) work->scaling->E[i] = work->scaling->Einv[i] = 1.0;
      work->scaling->c = work->scaling->cinv = 1.0;
    }
    memcpy(work->temp_n, work->scaling->D, n * sizeof(c_float)); memcpy(work->temp_m, work->scaling->E, m * sizeof(c_float));
    const c_float c_temp = work->scaling->c;
    double cc = 1.0;
    engine_ruiz_rescale(e, (int)(settings->scaling - work->settings->scaling), &cc);
    download(e, work->scaling->D, e->D, n); download(e, work->scaling->E, e->E, m);
    memcpy(work->D_temp, work->scaling->D, n * sizeof(c_float));
    for (int i = 0; i < n; i++) work->scaling->D[i] = work->scaling->D[i] * work->temp_n[i];
    for (int i = 0; i < m; i++) work->scaling->E[i] = work->scaling->E[i] * work->temp_m[i];
    work->scaling->c = cc * c_temp;
    for (int i = 0; i < n; i++) work->scaling->Dinv[i] = 1.0 / work->scaling->D[i];
    for (int i = 0; i < m; i++) work->scaling->Einv[i] = 1.0 / work->scaling->E[i];
    work->scaling->cinv = 1 / work->scaling->c;
    upload(e, e->D, work->scaling->D, n); upload(e, e->Dinv, work->scaling->Dinv, n);
    upload(e, e->E, work->scaling->E, m); upload(e, e->Einv, work->scaling->Einv, m);
    e->scaling = 1; e->c = work->scaling->c; e->cinv = work->scaling->cinv;
    download(e, work->data->q, e->q, n); download(e, work->data->bmin, e->bmin, m); download(e, work->data->bmax, e->bmax, m);
    download(e, work->Qx, e->Qx, n);
  }
  *work->settings = *settings;
  work->sqrt_delta = sqrt(work->settings->delta);
}

extern "C" void qpalm_update_bounds(QPALMWorkspace *work, const c_float *bmin, const c_float *bmax) {
  Engine *e = eng(work);
  const size_t m = work->data->m;
  if (bmin != NULL && bmax != NULL)
    for (size_t j = 0; j < m; j++)
      if (bmin[j] > bmax[j]) {
        QP_EPRINT("Lower bound at index %d is greater than upper bound: %.4e > %.4e", (int)j, work->data->bmin[j], work->data->bmax[j]);
        update_status(work->info, QPALM_ERROR);
        return;
      }
  if (bmin != NULL) memcpy(work->data->bmin, bmin, m * sizeof(c_float));
  if (bmax != NULL) memcpy(work->data->bmax, bmax, m * sizeof(c_float));
  if (work->settings->scaling) {
    if (bmin != NULL) for (size_t j = 0; j < m; j++) work->data->bmin[j] = work->scaling->E[j] * work->data->bmin[j];
    if (bmax != NULL) for (size_t j = 0; j < m; j++) work->data->bmax[j] = work->scaling->E[j] * work->data->bmax[j];
  }
  if (bmin != NULL) upload(e, e->bmin, work->data->bmin, (int)m);
  if (bmax != NULL) upload(e, e->bmax, work->data->bmax, (int)m);
  cudaStreamSynchronize(e->stream);
}

extern "C" void qpalm_update_q(QPALMWorkspace *work, const c_float *q) {
  Engine *e = eng(work);
  const int n = e->n;
  memcpy(work->data->q, q, n * sizeof(c_float));
  if (work->settings->scaling) {
    for (int i = 0; i < n; i++) work->data->q[i] = work->scaling->D[i] * work->data->q[i];
    const c_float c_old = work->scaling->c;
    download(e, work->Qx, e->Qx, n); download(e, work->x, e->x, n);
    if (work->settings->proximal) for (int i = 0; i < n; i++) work->Qx[i] = work->Qx[i] + (-1 / work->gamma) * work->x[i];
    double nrm = 0;
    for (int i = 0; i < n; i++) { work->temp_n[i] = work->data->q[i] + work->scaling->cinv * work->Qx[i]; nrm = c_max(nrm, c_absval(work->temp_n[i])); }
    work->scaling->c = 1 / c_max(1.0, nrm);
    work->scaling->cinv = 1 / work->scaling->c;
    for (int i = 0; i < n; i++) work->data->q[i] *= work->scaling->c;
    const c_float c_ratio = work->scaling->c / c_old;
    scale_Q_values(e, c_ratio, false);
    for (int i = 0; i < n; i++) work->Qx[i] *= c_ratio;
    if (work->settings->proximal) {
      work->gamma = work->settings->gamma_init;
      for (int i = 0; i < n; i++) work->Qx[i] = work->Qx[i] + (1 / work->gamma) * work->x[i];
    }
    upload(e, e->Qx, work->Qx, n);
    e->c = work->scaling->c; e->cinv = work->scaling->cinv;
  }
  upload(e, e->q, work->data->q, n);
  cudaStreamSynchronize(e->stream);
}

extern "C" void qpalm_cleanup(QPALMWorkspace *work) {   // qpalm.c:874-1096
  if (!work) return;
  if (work->solver && work->solver->LD) engine_destroy((Engine *)work->solver->LD);
  if (work->data) { csc_free_host(work->data->Q); csc_free_host(work->data->A); free(work->data->q); free(work->data->bmin); free(work->data->bmax); free(work->data); }
  if (work->scaling) { free(work->scaling->D); free(work->scaling->Dinv); free(work->scaling->E); free(work->scaling->Einv); free(work->scaling); }
#define FR(f) free(work->f)
  FR(x); FR(y); FR(Ax); FR(Qx); FR(x_prev); FR(Aty); FR(x0); FR(temp_m); FR(temp_n); FR(sigma); FR(sigma_inv);
  FR(z); FR(Axys); FR(pri_res); FR(pri_res_in); FR(df); FR(xx0); FR(dphi); FR(dphi_prev); FR(sqrt_sigma);
  FR(delta); FR(alpha); FR(delta2); FR(delta_alpha); FR(temp_2m); FR(s); FR(index_L); FR(index_P); FR(index_J);
  FR(delta_y); FR(Atdelta_y); FR(delta_x); FR(Qdelta_x); FR(Adelta_x);
  FR(neg_dphi); FR(d); FR(Qd); FR(Ad); FR(yh); FR(Atyh); FR(D_temp); FR(E_temp);
#undef FR
  free(work->settings);
  if (work->solver) {
    free(work->solver->active_constraints); free(work->solver->active_constraints_old); free(work->solver->enter); free(work->solver->leave);
    free(work->solver->neg_dphi); free(work->solver->d); free(work->solver->Qd); free(work->solver->Ad); free(work->solver->yh);
    free(work->solver->Atyh); free(work->solver->E_temp); free(work->solver->D_temp);
    free(work->solver);
  }
  if (work->solution) { free(work->solution->x); free(work->solution->y); free(work->solution); }
  free(work->timer); free(work->info); free(work);
}

extern "C" int qpalm_b200_get_stats(const QPALMWorkspace *work, QPALMB200Stats *out) {
  if (!work || !work->solver || !work->solver->LD) return 1;
  const Engine *e = eng(work);
  out->kernel_launches = g_kernel_launches - e->launches0;
  out->inner_iterations = e->n_inner; out->outer_iterations = e->n_outer; out->refactorizations = e->n_refactor;
  out->refactor_active_sum = e->refactor_active_sum; out->updown_calls = e->n_updown; out->updown_rank_sum = e->updown_rank_sum;
  out->spmv_calls = e->n_spmv; out->algorithmic_bytes = e->alg_bytes; out->dense_flops = e->dense_flops;
  out->device_ms_factor = e->ms_factor; out->device_ms_updown = e->ms_updown; out->device_ms_total = e->ms_total;
  out->sparse_factor_nnz = e->kkt ? kkt_factor_nnz(e->kkt) : (e->sp ? sparse_chol_info(e->sp)->nnzL : 0);
  out->kkt_factorizations = kkt_factor_count(e->kkt); out->kkt_refinement_steps = kkt_refine_count(e->kkt);
  out->sparse_supernodes = e->sp ? sparse_chol_info(e->sp)->nsuper : 0;
  out->sparse_levels = e->sp ? sparse_chol_info(e->sp)->nlevels : 0;
  out->sigma_update_calls = e->n_sigma_update; out->sigma_update_rank_sum = e->sigma_update_rank_sum;
  return 0;
}
