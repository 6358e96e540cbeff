// kkt.cu -- the KKT factorization path of the semismooth Newton step (SURVEY.md 8 row f3).
//
// Reference (LADEL build only): FACTORIZE_KKT branch of newton_set_direction (src/newton.c:22-95), qpalm_form_kkt /
// qpalm_reform_kkt / kkt_solve (src/solver_interface.c:119-247), selection heuristic qpalm_set_factorization_method
// (src/solver_interface.c:20-70).  Instead of the Schur complement  Q + A_J' Sigma_J A_J + I/gamma  (whose pattern fills
// in when rows of A are long or overlap a lot), the step solves the quasi-definite augmented system
//
//        [ Q + I/gamma     A_J' ] [ d      ]   [ -dphi ]
//        [ A_J       -inv(Sigma_J) ] [ lambda ] = [   0   ]          (inactive rows: a decoupled -1 on the diagonal)
//
// B200 design: ONE symbolic analysis at setup of the static pattern with EVERY constraint row present (an inactive row
// only zeroes values), on the supernodal multifrontal machinery of sparse.cu run in its signed mode (L S L', pivot signs
// known a priori for a quasi-definite matrix).  A change of the active set or of sigma / gamma rewrites the values
// (k_kkt_values) and refactorises -- the reference's ladel_row_add / ladel_row_del are replaced by the refactorisation
// of the same matrix -- and every solve is followed by the reference's iterative refinement (newton.c:57-90).
#include "engine.cuh"
#include <vector>
#include <math.h>

namespace qb {

struct KktEngine {
  int n = 0, m = 0, N = 0;
  SparseChol *sp = nullptr;
  double *panels = nullptr;
  // K as a full symmetric CSR over the static pattern (int32), values rewritten per refactorisation
  int *Kp = nullptr, *Ki = nullptr;
  double *Kx = nullptr;
  long long nnzK = 0;
  // per entry: kind 0 = Q entry (src -> Q_csr.x, diag flag in krow), 1 = A entry of the top-right block (src -> A_csc.x, krow = row),
  // 2 = A entry of the bottom-left block (src -> A_csr.x, krow = row), 3 = constraint diagonal (krow = row)
  int *kind = nullptr, *src = nullptr, *krow = nullptr;
  double *rhs = nullptr, *sol = nullptr, *res = nullptr, *corr = nullptr;   // N each
  double *norms = nullptr, *norms_host = nullptr;                            // 2 doubles (device / pinned host)
  long long n_factor = 0, n_refine = 0;
};

__global__ void k_kkt_values(long long nnz, const int *__restrict__ kind, const int *__restrict__ src, const int *__restrict__ krow,
                             const double *__restrict__ Qx, const double *__restrict__ Acx, const double *__restrict__ Arx,
                             const int *__restrict__ active, const double *__restrict__ sigma_inv, double beta, double *Kx) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nnz) return;
  const int kd = kind[k];
  double v;
  if (kd == 0) v = Qx[src[k]] + (krow[k] ? beta : 0.0);
  else if (kd == 4) v = beta;                                   // structural diagonal of the (1,1) block that Q does not store
  else if (kd == 1) v = active[krow[k]] ? Acx[src[k]] : 0.0;
  else if (kd == 2) v = active[krow[k]] ? Arx[src[k]] : 0.0;
  else v = active[krow[k]] ? -sigma_inv[krow[k]] : -1.0;
  Kx[k] = v;
}

// rhs = [-dphi ; 0]
__global__ void k_kkt_rhs(int n, int N, const double *__restrict__ dphi, double *rhs) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N) rhs[i] = (i < n) ? dphi[i] * -1 : 0.0;
}
// res = rhs - K sol (K sol in `ks`), norms[0] = |res|inf, norms[1] = max(|K sol|inf, |rhs|inf)   (newton.c:57-66)
__global__ void __launch_bounds__(1024) k_kkt_residual(int N, const double *__restrict__ rhs, const double *__restrict__ ks, double *res, double *norms) {
  __shared__ double scratch[32];
  double r0 = 0.0, r1 = 0.0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const double r = rhs[i] - ks[i];
    res[i] = r;
    r0 = fmax(r0, fabs(r));
    r1 = fmax(r1, fmax(fabs(ks[i]), fabs(rhs[i])));
  }
  r0 = block_red<RED_MAX>(r0, scratch);
  __syncthreads();
  r1 = block_red<RED_MAX>(r1, scratch);
  if (threadIdx.x == 0) { norms[0] = r0; norms[1] = r1; }
}
__global__ void k_kkt_add(int N, const double *__restrict__ corr, double *sol) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N) sol[i] += corr[i];
}
__global__ void k_csr_spmv_plain(int rows, const int *__restrict__ p, const int *__restrict__ ci, const double *__restrict__ v,
                                 const double *__restrict__ x, double *y) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  double acc = 0.0;
  for (int k = p[row] + lane; k < p[row + 1]; k += 32) acc = fma(v[k], x[ci[k]], acc);
  acc = warp_sum(acc);
  if (lane == 0) y[row] = acc;
}

// the reference's switching criterion (src/solver_interface.c:20-66), restated on the caller's CSC inputs
bool kkt_heuristic_prefers_kkt(int n, int m, const long long *Ap, const long long *Ai, const long long *Qp, const long long *Qi) {
  if (m <= 0) return false;
  double nnz_kkt = (double)Qp[n] + n + (double)Ap[n] + m;
  for (int col = 1; col <= n; col++) {   // compensate for diagonal entries present in Q (last entry of an upper-stored column there;
    bool has_diag = false;               // here Q is lower-stored, so look for the diagonal anywhere in the column)
    for (long long k = Qp[col - 1]; k < Qp[col]; k++) if (Qi[k] == col - 1) { has_diag = true; break; }
    if (has_diag) nnz_kkt--;
  }
  double nnz_schur = nnz_kkt - (double)Ap[n] - m;
  std::vector<long long> rowcnt((size_t)m, 0);
  for (long long k = 0; k < Ap[n]; k++) rowcnt[Ai[k]]++;
  long long cmax = 0;
  for (int i = 0; i < m; i++) if (rowcnt[i] > cmax) cmax = rowcnt[i];
  for (int i = 0; i < m; i++) {
    const double c = (double)rowcnt[i];
    if (c + cmax <= n) nnz_schur += 0.5 * c * (c - 1);
    else nnz_schur += (n - cmax) * (c - (n - cmax + 1) / 2.0);
  }
  if (2 * cmax > n) nnz_schur += 0.5 * cmax * (cmax - 1) - (n - cmax) * (cmax - (n - cmax + 1) / 2.0);
  const double cap = (double)n * (n - 1) / 2;
  if (nnz_schur > cap) nnz_schur = cap;
  if (nnz_schur < 1) nnz_schur = 1;
  return (nnz_kkt * nnz_kkt) / (nnz_schur * nnz_schur) * n / (n + m) < 2;
}

int kkt_create(KktEngine **out, Engine *e, int n, int m, const long long *Ap, const long long *Ai, const long long *Qp, const long long *Qi) {
  *out = nullptr;
  if (e->A_dense || e->Q_dense || m <= 0) return 1;
  KktEngine *K = new KktEngine();
  K->n = n; K->m = m; K->N = n + m;
  const int N = n + m;
  // ---- lower-triangular pattern for the symbolic analysis (int64 CSC) ----
  std::vector<long long> Lp((size_t)N + 1, 0), Li;
  Li.reserve((size_t)Qp[n] + Ap[n] + N);
  std::vector<char> has_diag((size_t)n, 0);
  for (int j = 0; j < n; j++) {
    Lp[j] = (long long)Li.size();
    bool diag = false;
    for (long long k = Qp[j]; k < Qp[j + 1]; k++) if (Qi[k] == j) diag = true;
    has_diag[j] = diag;
    if (!diag) Li.push_back(j);                                   // the proximal term makes the diagonal structural
    for (long long k = Qp[j]; k < Qp[j + 1]; k++) if (Qi[k] >= j) Li.push_back(Qi[k]);
    for (long long k = Ap[j]; k < Ap[j + 1]; k++) Li.push_back(n + Ai[k]);
  }
  for (int i = 0; i < m; i++) { Lp[n + i] = (long long)Li.size(); Li.push_back(n + i); }
  Lp[N] = (long long)Li.size();
  if (int r = sparse_ldl_analyze(&K->sp, N, n, Lp.data(), Li.data(), e->stream)) { delete K; return r; }
  // ---- full symmetric CSR of K over the same pattern, with the source of every value ----
  // host copies of the engine's device index arrays (Q full symmetric CSR, A CSC / CSR) give the value positions
  std::vector<int> qp((size_t)n + 1), qi((size_t)e->Q_csr.nnz), acp((size_t)n + 1), aci((size_t)e->A_csc.nnz), arp((size_t)m + 1), arj((size_t)e->A_csr.nnz);
  QB_CUDA_TRY(cudaMemcpy(qp.data(), e->Q_csr.p, sizeof(int) * (n + 1), cudaMemcpyDeviceToHost));
  if (e->Q_csr.nnz) QB_CUDA_TRY(cudaMemcpy(qi.data(), e->Q_csr.i, sizeof(int) * (size_t)e->Q_csr.nnz, cudaMemcpyDeviceToHost));
  QB_CUDA_TRY(cudaMemcpy(acp.data(), e->A_csc.p, sizeof(int) * (n + 1), cudaMemcpyDeviceToHost));
  QB_CUDA_TRY(cudaMemcpy(aci.data(), e->A_csc.i, sizeof(int) * (size_t)e->A_csc.nnz, cudaMemcpyDeviceToHost));
  QB_CUDA_TRY(cudaMemcpy(arp.data(), e->A_csr.p, sizeof(int) * (m + 1), cudaMemcpyDeviceToHost));
  QB_CUDA_TRY(cudaMemcpy(arj.data(), e->A_csr.i, sizeof(int) * (size_t)e->A_csr.nnz, cudaMemcpyDeviceToHost));
  std::vector<int> kp((size_t)N + 1, 0), ki, kind, src, krow;
  const size_t est = (size_t)e->Q_csr.nnz + 2 * (size_t)e->A_csr.nnz + N;
  ki.reserve(est); kind.reserve(est); src.reserve(est); krow.reserve(est);
  for (int j = 0; j < n; j++) {
    kp[j] = (int)ki.size();
    if (!has_diag[j]) { ki.push_back(j); kind.push_back(4); src.push_back(0); krow.push_back(0); }
    for (int k = qp[j]; k < qp[j + 1]; k++) { ki.push_back(qi[k]); kind.push_back(0); src.push_back(k); krow.push_back(qi[k] == j ? 1 : 0); }
    for (int k = acp[j]; k < acp[j + 1]; k++) { ki.push_back(n + aci[k]); kind.push_back(1); src.push_back(k); krow.push_back(aci[k]); }
  }
  for (int i = 0; i < m; i++) {
    kp[n + i] = (int)ki.size();
    for (int k = arp[i]; k < arp[i + 1]; k++) { ki.push_back(arj[k]); kind.push_back(2); src.push_back(k); krow.push_back(i); }
    ki.push_back(n + i); kind.push_back(3); src.push_back(0); krow.push_back(i);
  }
  kp[N] = (int)ki.size();
  K->nnzK = (long long)ki.size();
  auto upi = [&](int **dst, const std::vector<int> &v) -> int {
    QB_CUDA_TRY(cudaMalloc((void **)dst, sizeof(int) * (v.size() + 2)));
    QB_CUDA_TRY(cudaMemcpy(*dst, v.data(), sizeof(int) * v.size(), cudaMemcpyHostToDevice));
    return 0;
  };
  int rc = 0;
  rc |= upi(&K->Kp, kp); rc |= upi(&K->Ki, ki); rc |= upi(&K->kind, kind); rc |= upi(&K->src, src); rc |= upi(&K->krow, krow);
  if (rc) { delete K; return rc; }
  QB_CUDA_TRY(cudaMalloc((void **)&K->Kx, sizeof(double) * (size_t)(K->nnzK + 2)));
  QB_CUDA_TRY(cudaMalloc((void **)&K->panels, sizeof(double) * sparse_chol_factor_doubles(K->sp)));
  for (double **v : {&K->rhs, &K->sol, &K->res, &K->corr}) {
    QB_CUDA_TRY(cudaMalloc((void **)v, sizeof(double) * (size_t)(N + 1)));
    QB_CUDA_TRY(cudaMemset(*v, 0, sizeof(double) * (size_t)(N + 1)));
  }
  QB_CUDA_TRY(cudaMalloc((void **)&K->norms, sizeof(double) * 2));
  QB_CUDA_TRY(cudaMallocHost((void **)&K->norms_host, sizeof(double) * 2));
  if (getenv("QPALM_B200_VERBOSE")) {
    const SparseCholInfo *I = sparse_chol_info(K->sp);
    fprintf(stderr, "[qpalm_b200] KKT Newton path: N=%d nnz(K)=%lld nnz(L)=%lld supernodes=%d levels=%d %.3g flop/factorization\n",
            N, K->nnzK, I->nnzL, I->nsuper, I->nlevels, I->flops);
  }
  *out = K;
  return 0;
}

void kkt_destroy(KktEngine *K) {
  if (!K) return;
  sparse_chol_destroy(K->sp);
  void *ptrs[] = {K->panels, K->Kp, K->Ki, K->Kx, K->kind, K->src, K->krow, K->rhs, K->sol, K->res, K->corr, K->norms};
  for (void *p : ptrs) if (p) cudaFree(p);
  if (K->norms_host) cudaFreeHost(K->norms_host);
  delete K;
}

long long kkt_factor_nnz(const KktEngine *K) { return K ? sparse_chol_info(K->sp)->nnzL : 0; }
long long kkt_factor_count(const KktEngine *K) { return K ? K->n_factor : 0; }
long long kkt_refine_count(const KktEngine *K) { return K ? K->n_refine : 0; }
void kkt_last_norms(const KktEngine *K, double out2[2]) { out2[0] = K->norms_host[0]; out2[1] = K->norms_host[1]; }

// values of K for the committed active set, then L S L'  (qpalm_form_kkt / qpalm_reform_kkt + ladel_factorize*)
int kkt_refactor(KktEngine *K, Engine *e, double beta) {
  QB_CUDA_TRY(cudaEventRecord(e->evs0, e->stream));
  QB_LAUNCH(k_kkt_values, (unsigned)cdivll(K->nnzK, 256), 256, 0, e->stream, K->nnzK, K->kind, K->src, K->krow, e->Q_csr.x, e->A_csc.x,
            e->A_csr.x, e->active, e->sigma_inv, beta, K->Kx);
  if (int r = sparse_chol_assemble(K->sp, e->stream, K->panels, true, K->Kp, K->Ki, K->Kx, nullptr, nullptr, nullptr, nullptr, nullptr,
                                   nullptr, nullptr, nullptr, 0.0)) return r;
  if (int r = sparse_chol_factor(K->sp, e->stream, K->panels, e->info_dev)) return r;
  QB_CUDA_TRY(cudaEventRecord(e->evs1, e->stream));
  K->n_factor++;
  e->n_refactor++;
  const SparseCholInfo *I = sparse_chol_info(K->sp);
  e->dense_flops += I->flops;
  e->alg_bytes += 12.0 * (double)I->nnzS + 2.0 * 8.0 * (double)I->nnzL;
  return 0;
}

// kkt_solve + iterative refinement (newton.c:55-90): d = first n entries of the solution of K z = [-dphi; 0]
int kkt_solve(KktEngine *K, Engine *e) {
  const int N = K->N, n = K->n;
  QB_LAUNCH(k_kkt_rhs, cdiv(N, 256), 256, 0, e->stream, n, N, e->dphi, K->rhs);
  if (int r = sparse_chol_solve(K->sp, e->stream, K->panels, K->rhs, K->sol, false)) return r;
  for (int it = 0; it <= 3 /* MAX_REFINEMENT_ITERATIONS */; it++) {
    QB_LAUNCH(k_csr_spmv_plain, cdiv(N, 8), 256, 0, e->stream, N, K->Kp, K->Ki, K->Kx, K->sol, K->corr);
    QB_LAUNCH(k_kkt_residual, 1, 1024, 0, e->stream, N, K->rhs, K->corr, K->res, K->norms);
    QB_CUDA_TRY(cudaMemcpyAsync(K->norms_host, K->norms, sizeof(double) * 2, cudaMemcpyDeviceToHost, e->stream));
    QB_CUDA_TRY(cudaStreamSynchronize(e->stream));
    const double res = K->norms_host[0], ref = K->norms_host[1];
    if (it == 3 || !(res > fmax(1e-10 * ref, 1e-12))) break;   // RELATIVE / ABSOLUTE_REFINEMENT_TOLERANCE (constants.h:101-102)
    if (int r = sparse_chol_solve(K->sp, e->stream, K->panels, K->res, K->corr, false)) return r;
    QB_LAUNCH(k_kkt_add, cdiv(N, 256), 256, 0, e->stream, N, K->corr, K->sol);
    K->n_refine++;
  }
  QB_CUDA_TRY(cudaMemcpyAsync(e->d, K->sol, sizeof(double) * (size_t)n, cudaMemcpyDeviceToDevice, e->stream));
  e->alg_bytes += 2.0 * 12.0 * (double)sparse_chol_info(K->sp)->nnzL;
  return 0;
}

}  // namespace qb
