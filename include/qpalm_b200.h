/*
 * qpalm_b200.h -- C ABI of the Blackwell-native QPALM inner-iteration library (libqpalm_b200.so).
 *
 * Part 1 is the DROP-IN boundary: the eight public entry points of the reference
 * (/root/reference/include/qpalm.h:43-138) with byte-identical struct layouts
 * (/root/reference/include/types.h:37-314, CHOLMOD build, -DDLONG -DPROFILING) and the CHOLMOD
 * compressed-column input layout (suitesparse/CHOLMOD/Include/cholmod_core.h:1214-1263).
 * A caller compiled against the reference headers can be relinked against this library unchanged.
 *
 * Part 2 is the operator-level C ABI (plain pointers and sizes, host buffers in / host buffers out)
 * for the individual hot-path steps; each entry names the reference function it replaces.  These are
 * what the parity tests drive, one step at a time, "at identical iterates".
 *
 * Part 3 is the additive batch entry point (no counterpart in the reference, SURVEY.md 8(b)).
 *
 * Everything here runs on the GPU.  There is no CPU fallback: when no CUDA device is usable the
 * entry points fail loudly (qpalm_setup returns NULL and prints the CUDA error; operator calls
 * return a negative cudaError_t).
 */
#ifndef QPALM_B200_H
#define QPALM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------------
 * Part 1a -- scalar types and constants (reference: include/global_opts.h:31-62, constants.h)
 * ---------------------------------------------------------------------------------------------- */
typedef double  c_float;   /* reference: Real = double                      */
typedef int64_t c_int;     /* reference: SuiteSparse_long (LP64: 8 bytes)   */

#ifndef TRUE
#define TRUE 1
#define FALSE 0
#endif

#define QPALM_SOLVED              (1)
#define QPALM_DUAL_TERMINATED     (2)
#define QPALM_MAX_ITER_REACHED    (-2)
#define QPALM_PRIMAL_INFEASIBLE   (-3)
#define QPALM_DUAL_INFEASIBLE     (-4)
#define QPALM_TIME_LIMIT_REACHED  (-5)
#define QPALM_UNSOLVED            (-10)
#define QPALM_ERROR               (0)
#ifndef QPALM_NULL
#define QPALM_NULL 0
#endif
#ifndef QPALM_INFTY
#define QPALM_INFTY ((c_float)1e20)
#endif
#define FACTORIZE_KKT 0
#define FACTORIZE_SCHUR 1
#define FACTORIZE_KKT_OR_SCHUR 2

/* ------------------------------------------------------------------------------------------------
 * Part 1b -- input matrix layout.  Field for field the layout of cholmod_sparse; define
 * QPALM_B200_USE_CHOLMOD_H before including this header to use the real type instead.
 * Conventions every caller of the reference follows: itype = 2 (int64 p, i), xtype = 1 (real),
 * dtype = 0 (double), sorted = packed = 1; A has stype 0, Q has stype -1 (only entries with
 * row >= col are read; an upper triangle, if stored, is ignored).
 * ---------------------------------------------------------------------------------------------- */
#ifdef QPALM_B200_USE_CHOLMOD_H
#include "cholmod.h"
typedef cholmod_sparse solver_sparse;
#else
typedef struct qpalm_csc {
  size_t nrow, ncol, nzmax;
  void  *p;      /* int64[ncol+1] column pointers            */
  void  *i;      /* int64[nzmax]  row indices                */
  void  *nz;     /* unused (packed)                          */
  void  *x;      /* double[nzmax] values                     */
  void  *z;      /* unused (real)                            */
  int    stype, itype, xtype, dtype, sorted, packed;
} solver_sparse;
#endif

/* ------------------------------------------------------------------------------------------------
 * Part 1c -- public structs (identical field order to include/types.h)
 * ---------------------------------------------------------------------------------------------- */
typedef struct array_element { c_float x; size_t i; } array_element;        /* types.h:37-40   */

typedef struct { c_float *x, *y; } QPALMSolution;                            /* types.h:50-53   */

typedef struct { c_float *D, *Dinv, *E, *Einv; c_float c, cinv; } QPALMScaling; /* types.h:63-70 */

typedef struct {                                                             /* types.h:76-95   */
  c_int   iter, iter_out;
  char    status[32];
  c_int   status_val;
  c_float pri_res_norm, dua_res_norm, dua2_res_norm;
  c_float objective, dual_objective;
  c_float setup_time, solve_time, run_time;   /* -DPROFILING fields, always present here */
} QPALMInfo;

typedef struct {                                                             /* types.h:104-113 */
  size_t n, m;
  solver_sparse *Q, *A;
  c_float *q;
  c_float  c;
  c_float *bmin, *bmax;
} QPALMData;

typedef struct {                                                             /* types.h:119-150 */
  c_int   max_iter, inner_max_iter;
  c_float eps_abs, eps_rel, eps_abs_in, eps_rel_in, rho, eps_prim_inf, eps_dual_inf;
  c_float theta, delta, sigma_max, sigma_init;
  c_int   proximal;
  c_float gamma_init, gamma_upd, gamma_max;
  c_int   scaling, nonconvex, verbose, print_iter, warm_start, reset_newton_iter;
  c_int   enable_dual_termination;
  c_float dual_objective_limit, time_limit;
  c_int   ordering, factorization_method, max_rank_update;
  c_float max_rank_update_fraction;
} QPALMSettings;

/* types.h:155-187.  The CHOLMOD object pointers of the reference are opaque here: this library
 * keeps the matrices, the factor and all iterates in device memory behind `LD` (the engine handle);
 * the remaining pointers stay NULL.  The integer bookkeeping fields are live and mirror the device. */
typedef struct {
  c_int factorization_method;
  void *kkt, *kkt_full, *At;
  c_int *first_row_A; c_float *first_elem_A;
  void *LD;            /* engine handle (device-resident state) */
  void *sym, *LD_Q, *sym_Q;
  void *E_temp, *D_temp, *neg_dphi, *rhs_kkt, *sol_kkt, *d, *Ad, *Qd, *yh, *Atyh;
  c_int first_factorization, reset_newton;
  c_int *active_constraints, *active_constraints_old;
  c_int nb_active_constraints;
  c_int *enter; c_int nb_enter;
  c_int *leave; c_int nb_leave;
  void *At_scale, *At_sqrt_sigma;
} QPALMSolver;

typedef struct { int64_t tic_sec, tic_nsec, toc_sec, toc_nsec; } QPALMTimer;  /* util.h (linux) */

typedef struct {                                                             /* types.h:197-314 */
  QPALMData *data;                      /* SCALED problem vectors q,bmin,bmax (host mirror); Q,A: caller-layout copies */
  c_float *x, *y, *Ax, *Qx, *Aty, *x_prev;
  c_int initialized;
  c_float *temp_m, *temp_n, *sigma, *sigma_inv;
  c_float sqrt_sigma_max;
  c_int nb_sigma_changed;
  c_float gamma;
  c_int gamma_maxed;
  c_float *Axys, *z, *pri_res, *pri_res_in, *yh, *Atyh, *df, *x0, *xx0, *dphi, *neg_dphi, *dphi_prev, *d;
  c_float tau;
  c_float *Qd, *Ad, *sqrt_sigma;
  c_float sqrt_delta, eta, beta;
  c_float *delta, *alpha, *temp_2m, *delta2, *delta_alpha;
  array_element *s;
  c_int *index_L, *index_P, *index_J;
  c_float eps_pri, eps_dua, eps_dua_in, eps_abs_in, eps_rel_in;
  c_float *delta_y, *Atdelta_y;
  c_float *delta_x, *Qdelta_x, *Adelta_x;
  c_float *D_temp, *E_temp;
  QPALMSolver   *solver;
  QPALMSettings *settings;
  QPALMScaling  *scaling;
  QPALMSolution *solution;
  QPALMInfo     *info;
  QPALMTimer    *timer;
} QPALMWorkspace;

/* ------------------------------------------------------------------------------------------------
 * Part 1d -- the public API (reference: include/qpalm.h:43-138, src/qpalm.c)
 * ---------------------------------------------------------------------------------------------- */
void            qpalm_set_default_settings(QPALMSettings *settings);                       /* qpalm.c:39  */
QPALMWorkspace* qpalm_setup(const QPALMData *data, const QPALMSettings *settings);         /* qpalm.c:73  */
void            qpalm_warm_start(QPALMWorkspace *work, c_float *x_ws, c_float *y_ws);      /* qpalm.c:322 */
void            qpalm_solve(QPALMWorkspace *work);                                         /* qpalm.c:401 */
void            qpalm_update_settings(QPALMWorkspace *work, const QPALMSettings *settings);/* qpalm.c:739 */
void            qpalm_update_bounds(QPALMWorkspace *work, const c_float *bmin, const c_float *bmax); /* :793 */
void            qpalm_update_q(QPALMWorkspace *work, const c_float *q);                    /* qpalm.c:827 */
void            qpalm_cleanup(QPALMWorkspace *work);                                       /* qpalm.c:874 */

/* host-side helpers the reference also exports and its tests link against */
c_int validate_data(const QPALMData *data);                                                /* validate.c:18 */
c_int validate_settings(const QPALMSettings *settings);                                    /* validate.c:43 */
void  update_status(QPALMInfo *info, c_int status_val);                                    /* util.c:61     */

/* ------------------------------------------------------------------------------------------------
 * Part 2 -- operator-level C ABI.  All pointers are HOST pointers; each call uploads its inputs,
 * runs the same device kernels the solver uses, and downloads the outputs.  Return 0 on success,
 * -(cudaError_t) on a CUDA failure, a positive code on invalid arguments.
 * ---------------------------------------------------------------------------------------------- */

/* Library / device probe.  Returns the number of usable CUDA devices (0 => every other call fails). */
int qpalm_b200_device_count(void);
const char *qpalm_b200_version(void);
/* Per-engine counters used by bench.py for the roofline (SURVEY.md 8(d)). */
typedef struct {
  int64_t kernel_launches;      /* kernels launched by this library since engine creation             */
  int64_t inner_iterations;     /* update_primal_iterate calls                                         */
  int64_t outer_iterations;
  int64_t refactorizations;     /* ldlcholQAtsigmaA / ldlchol(Q) equivalents                           */
  int64_t refactor_active_sum;  /* sum of |J| over refactorizations                                    */
  int64_t updown_calls;         /* rank-k update/downdate sweeps                                       */
  int64_t updown_rank_sum;      /* sum of k over them                                                  */
  int64_t spmv_calls;           /* Qd, Ad, A'yh products                                               */
  double  algorithmic_bytes;    /* SURVEY.md 8(d) byte model, accumulated over the executed steps      */
  double  dense_flops;          /* n^2|J| + n^3/3 per refactorization, 2n^2 per solve, 2kn^2 per updown*/
  double  device_ms_factor;     /* CUDA-event time spent in refactorizations                           */
  double  device_ms_updown;
  double  device_ms_total;      /* CUDA-event time of the whole qpalm_solve                            */
  int64_t sparse_factor_nnz;    /* entries of the supernodal factor (0: the dense Newton path is in use)  */
  int64_t sparse_supernodes;
  int64_t sparse_levels;        /* assembly-tree levels = launches-in-sequence of one factorization pass */
  int64_t sigma_update_calls;   /* ldlupdate_sigma_changed equivalents taken (rank updates after a sigma change) */
  int64_t sigma_update_rank_sum;
  int64_t kkt_factorizations;   /* > 0: the Newton steps went through the KKT path (kkt.cu); L S L' factorizations of the KKT matrix */
  int64_t kkt_refinement_steps; /* iterative-refinement corrections applied after KKT solves (newton.c:57-90)                 */
} QPALMB200Stats;
int qpalm_b200_get_stats(const QPALMWorkspace *work, QPALMB200Stats *out);
/* Selective per-kernel CUDA-event timing of the library's own launches (csrc/prof.cu): `patterns` is a comma-separated
 * list of kernel-name substrings ("*" = all, NULL/"" = off).  prof_report synchronises and writes one JSON object
 * {"kernel": {"launches": L, "ms": T}, ...} into buf (returns the needed size when buf is NULL) and resets the log. */
int qpalm_b200_prof_enable(const char *patterns);
int qpalm_b200_prof_report(char *buf, size_t buflen);
/* Debug: in-kernel phase clocks of the cluster-per-front factorization kernel (csrc/sparse.cu, mfc::k_mf_front), accumulated
 * while QPALM_B200_MF_CLOCKS is set; copies 16 counters out and clears them (tools/prof_config.py names them). */
int qpalm_b200_mf_clocks(unsigned long long *out16);

/* y = A x  (A m x n, CSC, stype 0)              -- replaces mat_vec,       solver_interface.c:252-262
 * y = A' x                                      -- replaces mat_tpose_vec, solver_interface.c:264-274
 * y = Q x  (Q n x n, CSC, lower triangle used)  -- replaces mat_vec on a stype=-1 matrix            */
int qpalm_b200_mat_vec(const solver_sparse *A, const c_float *x, c_float *y);
int qpalm_b200_mat_tpose_vec(const solver_sparse *A, const c_float *x, c_float *y);
/* column / row infinity norms -- replaces mat_inf_norm_cols/rows, solver_interface.c:276-314 */
int qpalm_b200_mat_inf_norm_cols(const solver_sparse *M, c_float *E);
int qpalm_b200_mat_inf_norm_rows(const solver_sparse *M, c_float *E);

/* Ruiz equilibration -- replaces scale_data, scaling.c:34-113.  In: unscaled A, Q(lower), q, bmin,
 * bmax and the iteration count.  Out: D[n], E[m], c and the scaled A->x, Q->x, q, bmin, bmax written
 * in place into the caller's arrays (pattern unchanged). */
int qpalm_b200_scale_data(solver_sparse *A, solver_sparse *Q, c_float *q, c_float *bmin, c_float *bmax,
                          c_int scaling_iters, c_float *D, c_float *E, c_float *c_out);

/* Residual step at a given iterate -- replaces compute_residuals (iteration.c:24-48) fused with
 * set_active_constraints / set_entering_leaving_constraints (newton.c:122-149).
 * In:  A (CSC), Ax, y, sigma, bmin, bmax (m);  Qx, q, x0 (n);  proximal flag, gamma;  active_old (m, 0/1).
 * Out: Axys, z, pri_res, yh (m); Atyh, df, dphi (n); active (m, 0/1); enter/leave lists with counts. */
int qpalm_b200_residuals_active_set(const solver_sparse *A,
        const c_float *Ax, const c_float *y, const c_float *sigma, const c_float *bmin, const c_float *bmax,
        const c_float *Qx, const c_float *q, const c_float *x0, c_int proximal, c_float gamma,
        const c_int *active_old,
        c_float *Axys, c_float *z, c_float *pri_res, c_float *yh, c_float *Atyh, c_float *df, c_float *dphi,
        c_int *active, c_int *nb_active, c_int *enter, c_int *nb_enter, c_int *leave, c_int *nb_leave);

/* Exact line search -- replaces exact_linesearch (linesearch.c:14-120) AFTER Qd (+d/gamma) and Ad
 * are formed.  In: eta = d'Qd, beta = d'df, Ad, Ax, y, sigma, sqrt_sigma, bmin, bmax (m).
 * Out: tau; optionally (may be NULL) the sorted breakpoints: sorted_s[nL], sorted_idx[nL], *nL. */
int qpalm_b200_linesearch(c_int m, c_float eta, c_float beta,
        const c_float *Ad, const c_float *Ax, const c_float *y, const c_float *sigma,
        const c_float *sqrt_sigma, const c_float *bmin, const c_float *bmax,
        c_float *tau, c_float *sorted_s, c_int *sorted_idx, c_int *nL);

/* Newton system -- replaces ldlcholQAtsigmaA / ldlchol + ldlsolveLD_neg_dphi
 * (solver_interface.c:319-405, 505-519):  solve (Q + A_J' Sigma_J A_J + beta I) d = rhs  with the
 * dense blocked Cholesky (FP64 DMMA trailing updates).  active may be NULL (no constraints active).
 * If L_out != NULL the n x n column-major lower Cholesky factor is returned. */
int qpalm_b200_newton_solve(const solver_sparse *Q, const solver_sparse *A, const c_float *sigma,
        const c_int *active, c_float beta, const c_float *rhs, c_float *d, c_float *L_out);

/* Rank-k update / downdate of a dense Cholesky factor -- replaces cholmod_updown as called from
 * ldlupdate_entering_constraints / ldldowndate_leaving_constraints (solver_interface.c:407-441).
 * L: n x n column-major lower factor (in/out);  W: n x k column-major;  update != 0 => L L' + W W'. */
int qpalm_b200_updown(c_int n, c_int k, c_float *L, const c_float *W, c_int update);

/* Sparse Newton system -- replaces, for problems whose Schur complement Q + A'A stays sparse, cholmod_analyze +
 * cholmod_factorize (ldlchol / ldlcholQAtsigmaA, solver_interface.c:319-405), cholmod_updown (:407-441) and cholmod_solve
 * (:505-519) with a supernodal multifrontal Cholesky (csrc/sparse.cu).
 * symbolic_*: the one-time HOST-side analysis (fill-reducing ordering, etree, supernodes, assembly-tree levels); no CUDA call,
 * usable without a GPU.  symbolic_array copies one structure array ("perm", "iperm", "sn_first", "sn_of_col", "rows_off",
 * "rowidx", "rel", "sn_parent", "child_ptr", "child_idx", "lvl_ptr", "lvl_sn", "panel_off", "upd_off") and returns its length.
 * sparse_newton: factor Q + A_J' Sigma_J A_J + beta I for J = active, then rank-update with the rows `enter` and rank-downdate
 * with the rows `leave` (each scaled by sqrt(sigma)), then d = (L L')^{-1} rhs.  L_out (n x n column-major, PERMUTED order) and
 * perm_out (perm[new] = old) are optional; rowsums_out[0] (optional) receives the Gershgorin bound of A_J' Sigma_J A_J. */
typedef struct QPALMB200Symbolic QPALMB200Symbolic;
QPALMB200Symbolic *qpalm_b200_symbolic_analyze(const solver_sparse *Q, const solver_sparse *A);
int   qpalm_b200_symbolic_info(const QPALMB200Symbolic *S, c_int out8[8], double *flops);
c_int qpalm_b200_symbolic_array(const QPALMB200Symbolic *S, const char *name, c_int *out, c_int cap);
void  qpalm_b200_symbolic_free(QPALMB200Symbolic *S);
int qpalm_b200_sparse_newton(const solver_sparse *Q, const solver_sparse *A, const c_float *sigma, const c_int *active,
        c_float beta, const c_float *rhs, c_float *d, c_float *L_out, c_int *perm_out, const c_int *enter, c_int nb_enter,
        const c_int *leave, c_int nb_leave, c_float *rowsums_out);

/* lambda_min estimate -- replaces lobpcg (nonconvex.c:29-168).  x0 is the (un-normalised) start
 * vector the reference draws with rand(); returns the under-estimate the reference returns. */
int qpalm_b200_lobpcg(const solver_sparse *Q, const c_float *x0, c_float *lambda_out, c_int *iters_out);

/* FP64 tensor-core (DMMA) SYRK micro-benchmark used for the tensor roofline denominator:
 * C(n x n lower) = W W' with W n x k; returns the average ms per call over `reps` calls. */
int qpalm_b200_bench_dsyrk(c_int n, c_int k, c_int reps, double *ms_out);
int qpalm_b200_bench_potrf(c_int n, c_int reps, double *ms_out);
/* one rank-k update or downdate of an n x n factor as the solver runs it (updown_gen.cu: generator-form passes, <= 32
 * columns each, each followed by the refresh of the inverted diagonal blocks), k >= 1: average ms per update or downdate */
int qpalm_b200_bench_updown(c_int n, c_int k, c_int reps, double *ms_out);
/* FP64 tensor-pipe (DMMA) issue-rate peak in TFLOP/s: register-resident mma.sync chains, no memory traffic. */
int qpalm_b200_bench_dmma_peak(double *tflops_out);
/* scalar FP64 FMA (DFMA) issue-rate peak in TFLOP/s, same method: the bound of the kernels that use plain fma() */
int qpalm_b200_bench_dfma_peak(double *tflops_out);
/* dense matrix-vector kernels at the solver's shapes (At is n x m): ms per A*x (column dots) and per A'*y (row sums) */
int qpalm_b200_bench_gemv(c_int n, c_int m, c_int reps, double *ms_cols_out, double *ms_rows_out);
/* sparse products through the solver's CSR / CSC kernels: out3 = ms per A x, A' y, Q x; nnz3 = stored entries each one streams */
int qpalm_b200_bench_spmv(const solver_sparse *A, const solver_sparse *Q, c_int reps, double *out3, c_int *nnz3);

/* ------------------------------------------------------------------------------------------------
 * Part 2b -- row-sharding of one large dense QP over the GPUs of a box (additive; SURVEY.md 8(e), BASELINE config 3).
 * One process per GPU.  Rank 0 makes a 128-byte NCCL id (shard_unique_id), the caller distributes it, every rank calls
 * shard_init and then the ordinary qpalm_setup / qpalm_solve with the SAME full problem data: the library keeps only its
 * block of constraint rows of A on the device and exchanges A d (allgather), A' yh and the Schur-complement SYRK partials
 * (allreduce) over NCCL.  Every rank returns the same full solution.  Sparse A: replicas only (no sharding).
 * ---------------------------------------------------------------------------------------------- */
int  qpalm_b200_shard_unique_id(char *out128);
int  qpalm_b200_shard_init(int rank, int world, const char *id128);
void qpalm_b200_shard_finalize(void);

/* ------------------------------------------------------------------------------------------------
 * Part 2c -- QPS front end (SURVEY.md 8(f2)): replaces interfaces/qps/src/qpalm_qps.c.
 * qps_read  = get_sizes_and_check_format + read_data (qpalm_qps.c:69-575): the returned QPALMData holds A with the
 *             reference's appended bound rows (one per column without an FR bound, below the constraint rows),
 *             Q as the QUADOBJ lower triangle (stype -1), q, c = -RHS(objective), bmin/bmax.  Free with qps_free.
 *             Returns 0 ok, 1 cannot open, 2 format error.
 * read_settings = read_settings (qpalm_qps.c:610-689): defaults, then "name value" pairs after five header lines.
 * qps_solve = main (qpalm_qps.c:692-831): read, qpalm_setup (device upload), qpalm_solve, copy the solution out.
 * ---------------------------------------------------------------------------------------------- */
int  qpalm_b200_qps_read(const char *path, QPALMData **data_out, char *name_out, size_t name_len);
void qpalm_b200_qps_free(QPALMData *data);
int  qpalm_b200_read_settings(const char *path, QPALMSettings *settings);
int  qpalm_b200_qps_solve(const char *qps_path, const char *settings_path, QPALMInfo *info_out,
                          c_float *x_out, c_float *y_out, size_t *n_io, size_t *m_io);

/* ------------------------------------------------------------------------------------------------
 * Part 3 -- batch entry point (additive).  `nb` QPs sharing Q, A (values and pattern) and settings
 * but with their own q, bmin, bmax.  Each instance's result equals what qpalm_setup + qpalm_solve
 * return for that instance alone; after qpalm_b200_batch_warm_start, what qpalm_setup +
 * qpalm_warm_start(x_ws[k], y_ws[k]) + qpalm_solve return for instance k alone.
 * q: nb x n, bmin/bmax: nb x m (row-major, one instance per row).
 * Outputs (host): x: nb x n, y: nb x m, info: nb entries.  One persistent CTA per instance in flight.
 * ---------------------------------------------------------------------------------------------- */
typedef struct QPALMB200Batch QPALMB200Batch;
QPALMB200Batch *qpalm_b200_batch_setup(const QPALMData *shared, const QPALMSettings *settings, c_int nb_max);
int  qpalm_b200_batch_solve(QPALMB200Batch *batch, c_int nb, const c_float *q, const c_float *bmin,
                            const c_float *bmax, c_float *x, c_float *y, QPALMInfo *info);
/* device-resident variant used by bench.py's kernel-only number: inputs already uploaded by
 * qpalm_b200_batch_upload; returns device milliseconds of the solve kernels only. */
int  qpalm_b200_batch_upload(QPALMB200Batch *batch, c_int nb, const c_float *q, const c_float *bmin, const c_float *bmax);
int  qpalm_b200_batch_solve_resident(QPALMB200Batch *batch, c_int nb, double *device_ms);
int  qpalm_b200_batch_download(QPALMB200Batch *batch, c_int nb, c_float *x, c_float *y, QPALMInfo *info);
/* Warm start of the NEXT batch solve, per instance (qpalm_warm_start, qpalm.c:322-399): x_ws nb x n, y_ws nb x m, host,
 * row-major, unscaled (what a solve returns).  Either may be NULL: that part starts cold.  Instances k < nb start from
 * row k; instances >= nb of the next solve start cold.  Consumed by the next qpalm_b200_batch_solve / _solve_resident,
 * like qpalm_solve resets `initialized`; (NULL, NULL) clears a pending warm start (nb is not read).  Returns 0, 1 for
 * invalid arguments (pending state unchanged), < 0 for a CUDA error (no warm start pending). */
int  qpalm_b200_batch_warm_start(QPALMB200Batch *batch, c_int nb, const c_float *x_ws, const c_float *y_ws);
/* totals of the last solve over instances 0..nb-1: out8 = {inner iterations, outer iterations, refactorisations,
 * sum of |J| over the refactorisations, engine (1 lock-step, 2 persistent), rank-k update sweeps, sum of their ranks,
 * downdates that lost definiteness (followed by a refactorisation)} -- inputs of the SURVEY 8(d) byte model */
int  qpalm_b200_batch_stats(QPALMB200Batch *batch, c_int nb, double *out8);
/* persistent engine, totals of the last solve over instances 0..nb-1: out2 = {rows of A streamed through the H SYRK, summed
 * over the refactorisations; refactorisations that rebuilt H from c Q} (zeros after a lock-step solve) */
int  qpalm_b200_batch_syrk_stats(QPALMB200Batch *batch, c_int nb, double *out2);
/* persistent engine, totals of the last solve over instances 0..nb-1, summed over the line searches: out2 = {breakpoints
 * with s > 0 (the ones the line search sorts); sorted breakpoints its walk read, up to and including the one that fixed
 * tau} (zeros after a lock-step solve) */
int  qpalm_b200_batch_linesearch_stats(QPALMB200Batch *batch, c_int nb, double *out2);
/* persistent engine, QPALM_B200_BATCH_PROF=1 at setup: per-instance SM-clock totals of 16 phases of the last solve */
int  qpalm_b200_batch_phase_profile(QPALMB200Batch *batch, c_int nb, long long *out);
long long qpalm_b200_batch_last_launches(const QPALMB200Batch *batch);   /* kernels launched by the last solve */
/* engine and CTA shape of the last solve: 0 lock-step, 3 or 4 persistent (the build with 3 or 4 CTAs per SM) */
int  qpalm_b200_batch_last_shape(const QPALMB200Batch *batch);
void qpalm_b200_batch_cleanup(QPALMB200Batch *batch);

/* Test probes of the persistent engine's in-CTA building blocks, run by separate kernels of the same build (shape 3: the
 * default build, shape 4: the 4-CTAs-per-SM build) with its CTA size, shared-memory plan and persistent work queue.
 * Newton-step probe, per instance b < nb (matrices n x n column-major, lower triangle used; 1 <= n <= 240):
 *   H = src + sum_{pos} w^2 a a' - sum_{neg} w^2 a a', src = H0[b] (H0: nb x n x n), or with from_q the one shared matrix
 *       H0 scaled by sscale (the solver's path without active rows; then npos = nneg = 0 and the factor reads H0 itself)
 *   L = chol(H + beta I), d_fused = (L L')^{-1} rhs[b] right after the factorisation
 *   then, nup > 0: rank update of L by the rows upd[0 .. nup), the first kpos entering (+), the rest leaving (-), in sweeps of 8
 *   d_after = (L L')^{-1} rhs[b] with the final L (separate forward and backward substitutions)
 * a = wts entry * column list entry of At (n x m, shared).  cnt: nb x 4 {npos, nneg, nup, kpos}; lists, wts: nb x 3m, per
 * instance the pos rows at [0, m), the neg rows at [m, 2m), the update rows at [2m, 3m).  Outputs H_out, L_out (nb x n x n,
 * lower triangles, zero above), d_fused, d_after (nb x n) and info (bit 0: a sweep lost definiteness, bit 1: the
 * factorisation met a non-positive pivot).  Returns 0, 1 for invalid arguments, < 0 for a CUDA error. */
int qpalm_b200_batchp_probe_newton(c_int shape, c_int nb, c_int n, c_int m, const c_float *At, const c_float *H0, c_int from_q,
        c_float sscale, const c_int *cnt, const c_int *lists, const c_float *wts, c_float beta, const c_float *rhs,
        c_float *H_out, c_float *L_out, c_float *d_fused, c_float *d_after, c_int *info);
/* The Newton-step probe, then 2 rounds more triangular solves per instance, so that the solves' mbarrier phase carries across
 * update sweeps, solves and instances: round r < rounds first updates L by the rows upd[0 .. nup), all entering (+) for even r and
 * all leaving (-) for odd r; every round r < 2 rounds then writes (L L')^{-1} ((r + 1) rhs[b]) to d_rounds (nb x 2 rounds x n). */
int qpalm_b200_batchp_probe_solves(c_int shape, c_int nb, c_int n, c_int m, const c_float *At, const c_float *H0, c_int from_q,
        c_float sscale, const c_int *cnt, const c_int *lists, const c_float *wts, c_float beta, const c_float *rhs,
        c_float *H_out, c_float *L_out, c_float *d_fused, c_float *d_after, c_int *info, c_int rounds, c_float *d_rounds);
/* the line search's in-CTA sort on nb independent arrays of N <= 2048 (key, val) pairs (nb x N each), in place: keys ascending
 * as unsigned integers, equal keys in their input order (the solver sorts (key, position) pairs) */
int qpalm_b200_batchp_probe_sort(c_int shape, c_int nb, c_int N, unsigned long long *keys, unsigned int *vals);

#ifdef __cplusplus
}
#endif
#endif /* QPALM_B200_H */
