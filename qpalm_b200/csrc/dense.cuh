// dense.cuh -- dense FP64 building blocks of the Newton system (Q + A_J' Sigma_J A_J + I/gamma) d = -dphi:
// DMMA (mma.sync m8n8k4 f64) NT-GEMM / SYRK, blocked right-looking Cholesky, blocked triangular
// solves and the rank-k update/downdate.  All matrices are column-major with a leading dimension that
// is a multiple of 128 (qb::kPanel); rows/columns beyond n are an identity pad.
#pragma once
#include "common.cuh"

namespace qb {

// C[M x N] = beta*C + alpha * A[M x K] * B[N x K]'      (A, B, C column-major; M, N % 128 == 0, K % 16 == 0)
// lower_only: only tiles with block-row >= block-col are computed (SYRK / Cholesky trailing update).
// C may alias A when N == 128 (in-place triangular solve of a panel against an inverted diagonal block).
int dgemm_nt(cudaStream_t s, int M, int N, int K, const double *A, int lda, const double *B, int ldb,
             double *C, int ldc, double alpha, double beta, bool lower_only);

// Batched variants (grid.z / grid.y = instance; element strides sA.. between instances; Kz: optional per-instance K,
// maskz: optional per-instance activity flags).  Kz entries must be multiples of 16 and at most K: the kernel runs Kz / 16
// k-tiles, dropping a remainder silently (the lock-step engine pads its row lists to a multiple of 16 with zero rows).
int dgemm_nt_batched(cudaStream_t s, int nb, int M, int N, int K, const int *Kz, const double *A, int lda, long long sA,
                     const double *B, int ldb, long long sB, double *C, int ldc, long long sC, double alpha, double beta,
                     bool lower_only, const int *maskz);
// tile rows (64 or 128) of the kernel this thread's last dgemm_nt_batched call launched, 0 if it launched none.  The 64-row
// kernel runs when the tiles with work number fewer than the SMs.
int dgemm_last_tile_rows();
int potrf_lower_batched(cudaStream_t s, int nb, int npad, double *L, int ld, long long sL, double *invdiag, long long sX,
                        int *info_dev, const int *mask);
int chol_solve_batched(cudaStream_t s, int nb, int npad, const double *L, int ld, long long sL, const double *invdiag,
                       long long sX, double *v, long long sV, const int *mask);

// In-place blocked Cholesky of the lower triangle of L (npad x npad, ld).  invdiag receives the inverses
// of the 128 x 128 diagonal blocks of the factor (npad/128 blocks, each 128 x 128 column-major, upper
// part zero).  *info_dev (device int) is set to 1 + (first non-positive pivot column) on failure.
int potrf_lower(cudaStream_t s, int npad, double *L, int ld, double *invdiag, int *info_dev);

// Recompute invdiag from an existing factor (after an update/downdate sweep).
int trtri_diag_blocks(cudaStream_t s, int npad, const double *L, int ld, double *invdiag);

// v <- (L L')^{-1} v, v of length npad (pad entries must be 0).
int chol_solve(cudaStream_t s, int npad, const double *L, int ld, const double *invdiag, double *v);
// cooperative grid of the one-launch dataflow solve of this thread's last chol_solve, 0 when it ran the per-block launches
int chol_solve_last_grid();
// releases the per-stream scratch chol_solve keeps (flag buffer of the one-launch dataflow solve); call before destroying s
void chol_solve_release(cudaStream_t s);

// L <- chol(L L' + sign * W W'), W npad x k (ldw), k <= 8 per call, destroys W.  coef/alpha are scratch
// (coef: 2 * 32 * 18 doubles, alpha: 8 doubles).  *info_dev set to nonzero if a downdate loses
// positive definiteness.
int chol_updown(cudaStream_t s, int npad, double *L, int ld, double *W, int ldw, int k, int sign,
                double *coef, int *info_dev);

// Generator-form pass (updown_gen.cu): L <- chol(L L' + W S W'), S = diag(+1 x kpos, -1 x (k - kpos)), k <= 32 per call, reached by
// ONE triangular solve with k right-hand sides (the only serial chain, npad / 128 steps) + fully parallel passes; W (npad x k, ldw)
// is only read.  invdiag = inverses of the diagonal blocks of the current L (input; refresh it afterwards with trtri_diag_blocks).
// Returns 0 when it ran, 1 when unavailable (no cooperative launch, or no room for its work space: use chol_updown), < 0 on a CUDA error.
int chol_updown_gen(cudaStream_t s, int npad, double *L, int ld, const double *invdiag, const double *W, int ldw, int k, int kpos,
                    int *info_dev);
int chol_updown_gen_max_rank();
void chol_updown_gen_release(cudaStream_t s);
// test hooks.  last_grid: the per-group cooperative grid (blockIdx.x extent) of k_fwd_multi in this thread's last pass, 0 when
// it launched none; *gmax (may be NULL) the limit it ran under (the resident CTAs / groups, or the cap).  set_grid_cap: caps
// this thread's limit at cap CTAs per group (cap <= 0: no cap, the default) so that tests can deal block rows to fewer CTAs.
// workspace: the device work space of stream s's last pass, What (npad x 32) | Z (npad x 32) | D (npad) with the column
// stride npad of that pass, or NULL.
int chol_updown_gen_last_grid(int *gmax);
void chol_updown_gen_set_grid_cap(int cap);
const double *chol_updown_gen_workspace(cudaStream_t s);

// L(lower) <- H(lower) + diag_add * I on the leading n x n block; pad block <- identity.
int copy_lower_add_diag(cudaStream_t s, int n, int npad, const double *H, double *L, int ld, double diag_add);

// out[i] = sum_j |S_ij| for the symmetric matrix given by its lower triangle (Gershgorin row sums)
int sym_abs_rowsums(cudaStream_t s, int n, const double *H, int ld, double *out);

}  // namespace qb
