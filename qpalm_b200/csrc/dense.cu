// dense.cu -- FP64 dense kernels for the Newton system of QPALM (sm_100a).
//
// Replaces, for the Schur-complement path of the reference (src/solver_interface.c:319-519):
//   cholmod_aat + cholmod_add      -> dgemm_nt(lower_only) on gathered, sqrt(sigma)-scaled rows of A
//   cholmod_analyze/factorize_p    -> potrf_lower  (blocked right-looking, DMMA trailing updates)
//   cholmod_solve(CHOLMOD_LDLt)    -> chol_solve   (blocked forward/backward substitution)
//   cholmod_updown                 -> chol_updown  (rank-k recurrence of t_cholmod_updown_numkr.c:289-376
//                                                   restated for L L' and panelised for the GPU)
#include "dense.cuh"
#include "chol32.cuh"
#include <vector>
#include <map>
#include <mutex>
#include <stdlib.h>

namespace qb {

long long g_kernel_launches = 0;

// ================================================================================================
// DMMA NT GEMM:  C = beta*C + alpha * A * B'
// CTA tile BM_ x 128 x 16, 8 consumer warps + 1 producer warp, a 4-stage ring of k-major shared tiles padded to BM_ + 4 / 132
// doubles (conflict-free 64-bit fragment loads: lane -> (k = lane & 3, row = lane >> 2) hits 16 distinct 8-byte banks per half warp).
// The tile movement is on the TMA engine: bulk asynchronous copies (cp.async.bulk, SASS UBLKCP) issued by the PRODUCER warp
// and completed on mbarriers (its predecessor issued 16 cp.async (LDGSTS) instructions per thread and stage; DESIGN.md
// section 4 has both rates).
//   * warps 0-7 only compute (no address arithmetic, no copy instructions, no __syncthreads in the main loop);
//   * warp 8 owns the pipeline: per k-tile it waits for the stage's `empty` barrier (one arrival per consumer warp), posts
//     the expected byte count on the `full` barrier and issues ONE bulk copy per lane: lanes 0-15 the 16 k-columns of the A
//     tile, lanes 16-31 those of the B tile (each a contiguous run of BM_ / BN doubles of the column-major operand, landing
//     in the padded k-major row the fragment loads expect).
// Every operand column start is 16-byte aligned (leading dimensions are multiples of 128, tile origins multiples of 64).
// ================================================================================================
namespace gemm {
constexpr int BM = 128, BN = 128, BK = 16;

__device__ __forceinline__ void dmma884(double &d0, double &d1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
      : "+d"(d0), "+d"(d1)
      : "d"(a), "d"(b));
}

constexpr int TSTAGES = 4;
template <int BM_> constexpr size_t smem_bytes_tma() { return sizeof(double) * TSTAGES * BK * ((BM_ + 4) + (BN + 4)) + 2 * TSTAGES * sizeof(unsigned long long); }

__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
  const unsigned a = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(a), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gmem_src, unsigned bytes, unsigned long long *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}

// BM_ = 128: CTA tile 128 x 128, warps 2 x 4, warp tile 64 x 32.  BM_ = 64: CTA tile 64 x 128, warps 1 x 8, warp tile
// 64 x 16 -- twice as many CTAs of half the work each, for the panel solves and in-block updates of the Cholesky chain
// whose 128-row grids fill less than one wave of the 148 SMs.
template <int BM_>
__global__ void __launch_bounds__(288, 1)
k_dgemm_nt_tma(int K, const double *A, int lda, const double *B, int ldb,
               double *C, int ldc, double alpha, double beta, int lower_only,
               long long sA, long long sB, long long sC, const int *Kz, const int *maskz) {
  constexpr int SROWA = BM_ + 4, SROWB = BN + 4;
  constexpr int WM = BM_ / 64, WN = 8 / WM, NF = BN / (8 * WN);
  const int bm = blockIdx.x, bn = blockIdx.y;
  if (lower_only && bn * BN >= (bm + 1) * BM_) return;
  if (maskz && !maskz[blockIdx.z]) return;
  if (Kz) K = Kz[blockIdx.z];
  if (K <= 0 && beta == 1.0) return;
  A += (size_t)blockIdx.z * sA; B += (size_t)blockIdx.z * sB; C += (size_t)blockIdx.z * sC;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  typedef double TileA[BK][SROWA];
  typedef double TileB[BK][SROWB];
  TileA *As = reinterpret_cast<TileA *>(smem_raw);
  TileB *Bs = reinterpret_cast<TileB *>(smem_raw + sizeof(double) * TSTAGES * BK * SROWA);
  unsigned long long *full = reinterpret_cast<unsigned long long *>(smem_raw + sizeof(double) * TSTAGES * BK * (SROWA + SROWB));
  unsigned long long *empty = full + TSTAGES;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int KT = K / BK;
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < TSTAGES; s++) { mbar_init(full + s, 1); mbar_init(empty + s, 8); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (warp == 8) {   // ---- producer ----
    const double *Ag = A + (size_t)bm * BM_, *Bg = B + (size_t)bn * BN;
    constexpr unsigned kBytes = sizeof(double) * BK * (BM_ + BN);
    for (int kt = 0; kt < KT; kt++) {
      const int st = kt % TSTAGES;
      if (kt >= TSTAGES) mbar_wait(empty + st, ((kt / TSTAGES) - 1) & 1);   // the consumers have drained this stage
      if (lane == 0) mbar_expect_tx(full + st, kBytes);
      __syncwarp();
      const int kk = lane & 15;
      if (lane < 16) bulk_g2s(&As[st][kk][0], Ag + (size_t)(kt * BK + kk) * lda, sizeof(double) * BM_, full + st);
      else bulk_g2s(&Bs[st][kk][0], Bg + (size_t)(kt * BK + kk) * ldb, sizeof(double) * BN, full + st);
    }
    return;
  }

  // ---- consumers ----
  const int wm = warp % WM, wn = warp / WM;
  double acc[8][NF][2];
#pragma unroll
  for (int i = 0; i < 8; i++)
#pragma unroll
    for (int j = 0; j < NF; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
  const int fr = lane >> 2, fk = lane & 3;
  for (int kt = 0; kt < KT; kt++) {
    const int st = kt % TSTAGES;
    mbar_wait(full + st, (kt / TSTAGES) & 1);
    double a[2][8], b[2][NF];
#pragma unroll
    for (int mb = 0; mb < 8; mb++) a[0][mb] = As[st][fk][wm * 64 + mb * 8 + fr];
#pragma unroll
    for (int nb = 0; nb < NF; nb++) b[0][nb] = Bs[st][fk][wn * (8 * NF) + nb * 8 + fr];
#pragma unroll
    for (int ks = 0; ks < 4; ks++) {
      const int cur = ks & 1, nxt = cur ^ 1;
      if (ks < 3) {
#pragma unroll
        for (int mb = 0; mb < 8; mb++) a[nxt][mb] = As[st][(ks + 1) * 4 + fk][wm * 64 + mb * 8 + fr];
#pragma unroll
        for (int nb = 0; nb < NF; nb++) b[nxt][nb] = Bs[st][(ks + 1) * 4 + fk][wn * (8 * NF) + nb * 8 + fr];
      }
#pragma unroll
      for (int mb = 0; mb < 8; mb++)
#pragma unroll
        for (int nb = 0; nb < NF; nb++) dmma884(acc[mb][nb][0], acc[mb][nb][1], a[cur][mb], b[cur][nb]);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(empty + st);   // this warp is done with the stage
  }
  // every bulk copy of this CTA has been waited for: C may alias A from here on
  const bool use_beta = (beta != 0.0);
#pragma unroll
  for (int mb = 0; mb < 8; mb++) {
    const int row = bm * BM_ + wm * 64 + mb * 8 + fr;
#pragma unroll
    for (int nb = 0; nb < NF; nb++) {
      const int col = bn * BN + wn * (8 * NF) + nb * 8 + 2 * fk;
      double *c0 = C + row + (size_t)col * ldc;
      double *c1 = c0 + ldc;
      double v0 = alpha * acc[mb][nb][0], v1 = alpha * acc[mb][nb][1];
      if (use_beta) { v0 += beta * (*c0); v1 += beta * (*c1); }
      *c0 = v0; *c1 = v1;
    }
  }
}
}  // namespace gemm

static int gemm_attr() {
  static bool attr_set = false;
  if (!attr_set) {
    QB_CUDA_TRY(cudaFuncSetAttribute(gemm::k_dgemm_nt_tma<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm::smem_bytes_tma<128>()));
    QB_CUDA_TRY(cudaFuncSetAttribute(gemm::k_dgemm_nt_tma<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm::smem_bytes_tma<64>()));
    attr_set = true;
  }
  return 0;
}

static thread_local int g_gemm_last_rows = 0;   // tile rows (64 or 128) of this thread's last dgemm_nt_batched launch
int dgemm_last_tile_rows() { return g_gemm_last_rows; }

int dgemm_nt_batched(cudaStream_t s, int nb, int M, int N, int K, const int *Kz, const double *A, int lda, long long sA,
                     const double *B, int ldb, long long sB, double *C, int ldc, long long sC, double alpha, double beta,
                     bool lower_only, const int *maskz) {
  g_gemm_last_rows = 0;
  if (M <= 0 || N <= 0 || nb <= 0) return 0;
  if ((M % gemm::BM) || (N % gemm::BN) || (K % gemm::BK)) {
    fprintf(stderr, "[qpalm_b200] dgemm_nt: bad shape M=%d N=%d K=%d\n", M, N, K);
    return 1;
  }
  if (int e = gemm_attr()) return e;
  // CTAs that do work with 128-row tiles; below one wave of the GPU the 64-row kernel doubles the parallelism
  const long long mt = M / gemm::BM, nt = N / gemm::BN;
  const long long tiles = (lower_only ? (nt <= mt ? nt * mt - nt * (nt - 1) / 2 : mt * (mt + 1) / 2) : mt * nt) * nb;
  static int num_sms = 0;
  if (!num_sms) { int dev = 0; QB_CUDA_TRY(cudaGetDevice(&dev)); QB_CUDA_TRY(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev)); }
  g_gemm_last_rows = tiles < num_sms ? 64 : gemm::BM;
  if (tiles < num_sms) {
    dim3 grid(M / 64, N / gemm::BN, nb);
    QB_LAUNCH(gemm::k_dgemm_nt_tma<64>, grid, 288, gemm::smem_bytes_tma<64>(), s, K, A, lda, B, ldb, C, ldc, alpha, beta,
              lower_only ? 1 : 0, sA, sB, sC, Kz, maskz);
  } else {
    dim3 grid(M / gemm::BM, N / gemm::BN, nb);
    QB_LAUNCH(gemm::k_dgemm_nt_tma<128>, grid, 288, gemm::smem_bytes_tma<128>(), s, K, A, lda, B, ldb, C, ldc, alpha, beta,
              lower_only ? 1 : 0, sA, sB, sC, Kz, maskz);
  }
  QB_CUDA_TRY(cudaGetLastError());
  return 0;
}

int dgemm_nt(cudaStream_t s, int M, int N, int K, const double *A, int lda, const double *B, int ldb,
             double *C, int ldc, double alpha, double beta, bool lower_only) {
  if (K <= 0) { fprintf(stderr, "[qpalm_b200] dgemm_nt: bad shape M=%d N=%d K=%d\n", M, N, K); return 1; }
  return dgemm_nt_batched(s, 1, M, N, K, nullptr, A, lda, 0, B, ldb, 0, C, ldc, 0, alpha, beta, lower_only, nullptr);
}

// ================================================================================================
// 128 x 128 diagonal block: Cholesky factor + inverse of the factor, one CTA, all in shared memory.
// ================================================================================================
namespace diag {
// 128 x 128 diagonal block: Cholesky factor + inverse of the factor, one CTA of 8 warps, everything in shared memory.
//
// Right-looking over four 32-column sub-panels.  Per sub-panel kb (rows/cols r0 = 32 kb ..):
//   S1  warp 0:      factor the 32 x 32 diagonal block in registers (lane = row; template-unrolled so every register
//                    index is static; one shuffle + one reciprocal + one FMA on the critical path per column), then
//                    invert it (lane = column of the inverse) into Xb (natural layout) and into the upper triangle
//                    of As (transposed), whose diagonal carries 1/L(c,c).
//       warps 1..7:  meanwhile form R = L(block row kb, cols < r0) * X(< r0, < r0) for the inverse of the whole block
//                    (only needs data that is final before S1) -> hidden under the serial factorization.
//   S2  all warps:   X(block row kb, cols < r0) = -Xbb * R;  L21 = A21 * Xbb'  (rows below the block) into the
//                    transposed panel buffer Pt.
//   S3  all warps:   trailing update A22 -= L21 L21' from Pt (4 x 4 register tiles, 128-bit shared loads) and
//                    copy of Pt back into As.
// The inverse X (lower triangular) lives transposed in the upper triangle of As: X(i,c) at As[c*DS + i].
constexpr int NB = 128, DS = 129, NT = 256, SB = 32, XS = 33, PS = 100;
constexpr size_t kSmemBytes = sizeof(double) * (NB * DS + SB * XS + (NB - SB) * XS + SB * PS + NB) + 16;

using chol32::fstep;

// one warp: in-register Cholesky of the 32 x 32 block at (base, base); strictly-lower part of L back into As,
// 1/L(j,j) onto the diagonal of As, L(j,j) into ldiag.
__device__ __forceinline__ void factor32_warp(double *As, double *ldiag, int base, int lane, int *info, int col0) {
  double a[SB];
#pragma unroll
  for (int c = 0; c < SB; c++) a[c] = (c <= lane) ? As[(base + lane) * DS + base + c] : 0.0;
  double dl = 0.0, dinv = 0.0;
  int badcol = -1;
  fstep<0>(a, lane, dl, dinv, badcol);
  if (badcol >= 0 && lane == 0 && info) atomicCAS(info, 0, col0 + base + badcol + 1);
#pragma unroll
  for (int c = 0; c < SB; c++) if (c < lane) As[(base + lane) * DS + base + c] = a[c];
  As[(base + lane) * DS + base + lane] = dinv;
  ldiag[base + lane] = dl;
}

// right-looking column sweep of X = inv(L_bb), lane = column of X: v[r] accumulates sum_t L(r,t) x(t) until row r
// is finalised; 31 - R independent FMAs per step, no lane-dependent branches
template <int R>
__device__ __forceinline__ void istep(const double *Lb, double (&v)[SB], const int lane) {
  const double rd = Lb[R * DS + R];         // 1 / L(R,R)
  double xr = (R == lane) ? rd : -v[R] * rd;
  xr = (R < lane) ? 0.0 : xr;
  v[R] = xr;
#pragma unroll
  for (int q = R + 1; q < SB; q++) v[q] = fma(Lb[q * DS + R], xr, v[q]);
  if constexpr (R + 1 < SB) istep<R + 1>(Lb, v, lane);
}

// one warp: Xbb = inv(L_bb).  Natural layout into Xb (zeros above the diagonal), transposed into the upper
// triangle of the As block.
__device__ __forceinline__ void inv32_warp(double *As, double *Xb, int base, int lane) {
  double v[SB];
#pragma unroll
  for (int r = 0; r < SB; r++) v[r] = 0.0;
  istep<0>(As + base * DS + base, v, lane);
#pragma unroll
  for (int r = 0; r < SB; r++) {
    Xb[r * XS + lane] = v[r];
    if (r > lane) As[(base + lane) * DS + base + r] = v[r];
  }
}

// acc[a][b] += sum_{u0 <= u < u1} P[a*ps + u] * Q[b*qs + u]
template <int TR, int TC>
__device__ __forceinline__ void dot_tile(const double *P, int ps, const double *Q, int qs, int u0, int u1,
                                         double (&acc)[TR][TC]) {
#pragma unroll 4
  for (int u = u0; u < u1; u++) {
    double p[TR], q[TC];
#pragma unroll
    for (int a = 0; a < TR; a++) p[a] = P[a * ps + u];
#pragma unroll
    for (int b = 0; b < TC; b++) q[b] = Q[b * qs + u];
#pragma unroll
    for (int a = 0; a < TR; a++)
#pragma unroll
      for (int b = 0; b < TC; b++) acc[a][b] = fma(p[a], q[b], acc[a][b]);
  }
}

// Thread tiles are 2 rows x 4 columns with the two rows half a panel apart and the lanes of a warp running along the
// rows: row operands (stride DS or XS, both odd) then fall into distinct banks and the column operand is a broadcast.

// Rt(c, r) = sum_{u = c}^{r0 - 1} L(r0 + r, u) X(u, c),  r < 32, c < r0
__device__ __forceinline__ void inv_offdiag_R(const double *As, double *Rt, int r0, int t, int nthr) {
  const int ntiles = 16 * (r0 >> 2);
  for (int tile = t; tile < ntiles; tile += nthr) {
    const int tr = tile & 15, c0 = 4 * (tile >> 4);
    double acc[2][4] = {};
    const double *P = As + (r0 + tr) * DS, *Q = As + c0 * DS;
    // triangular head: X(u, c0 + b) exists for u >= c0 + b (the diagonal of As holds X(c,c))
#pragma unroll
    for (int uu = 0; uu < 4; uu++) {
      const int u = c0 + uu;
      const double p0 = P[u], p1 = P[16 * DS + u];
#pragma unroll
      for (int b = 0; b <= uu; b++) {
        const double q = Q[b * DS + u];
        acc[0][b] = fma(p0, q, acc[0][b]);
        acc[1][b] = fma(p1, q, acc[1][b]);
      }
    }
    dot_tile<2, 4>(P, 16 * DS, Q, DS, c0 + 4, r0, acc);
#pragma unroll
    for (int a = 0; a < 2; a++)
#pragma unroll
      for (int b = 0; b < 4; b++) Rt[(c0 + b) * XS + tr + 16 * a] = acc[a][b];
  }
}

// X(r0 + r, c) = - sum_{u <= r} Xbb(r, u) Rt(c, u), stored transposed at As[c*DS + r0 + r]
__device__ __forceinline__ void inv_offdiag_X(double *As, const double *Xb, const double *Rt, int r0, int t, int nthr) {
  const int ntiles = 16 * (r0 >> 2);
  for (int tile = t; tile < ntiles; tile += nthr) {
    const int tr = tile & 15, c0 = 4 * (tile >> 4);
    double acc[2][4] = {};
    dot_tile<2, 4>(Xb + tr * XS, 16 * XS, Rt + c0 * XS, XS, 0, tr + 17, acc);   // Xb is zero above its diagonal
#pragma unroll
    for (int a = 0; a < 2; a++)
#pragma unroll
      for (int b = 0; b < 4; b++) As[(c0 + b) * DS + r0 + tr + 16 * a] = -acc[a][b];
  }
}

// position of panel row i (relative to the first trailing row) inside one Pt column: rows 4t, 4t+1 of all 4-row groups
// first, rows 4t+2, 4t+3 after them, so that the 128-bit loads of consecutive groups are consecutive
__device__ __forceinline__ int pt_pos(int i) { return ((i >> 1) & 1) * 48 + ((i >> 2) << 1) + (i & 1); }

// Pt(c, i - r1) = sum_{u <= c} A(i, base + u) Xbb(c, u) for rows i >= r1 = base + 32 (the new L21, transposed)
__device__ __forceinline__ void panel_solve(const double *As, const double *Xb, double *Pt, int base, int t, int nthr) {
  const int r1 = base + SB, half = (NB - r1) >> 1, ntiles = half * 8;
  for (int tile = t; tile < ntiles; tile += nthr) {
    const int tc = tile / half, tr = tile - tc * half, c0 = 4 * tc;
    double acc[2][4] = {};
    dot_tile<2, 4>(As + (r1 + tr) * DS + base, half * DS, Xb + c0 * XS, XS, 0, c0 + 4, acc);
#pragma unroll
    for (int a = 0; a < 2; a++)
#pragma unroll
      for (int b = 0; b < 4; b++) Pt[(c0 + b) * PS + pt_pos(tr + a * half)] = acc[a][b];
  }
}

// A(i, k) -= sum_u Pt(u, i - r1) Pt(u, k - r1) for r1 <= k <= i < 128, and L21 copied from Pt into As
__device__ __forceinline__ void trailing_update(double *As, const double *Pt, int base, int t, int nthr) {
  const int r1 = base + SB, nrow = NB - r1, nt = nrow >> 2, ntiles = nt * (nt + 1) / 2;
  for (int tile = t; tile < ntiles; tile += nthr) {
    int ti = (int)((sqrtf(8.0f * (float)tile + 1.0f) - 1.0f) * 0.5f);
    while (ti * (ti + 1) / 2 > tile) ti--;
    while ((ti + 1) * (ti + 2) / 2 <= tile) ti++;
    const int tk = tile - ti * (ti + 1) / 2;
    double acc[4][4] = {};
#pragma unroll 4
    for (int u = 0; u < SB; u++) {
      const double2 pa = *reinterpret_cast<const double2 *>(Pt + u * PS + 2 * ti);
      const double2 pb = *reinterpret_cast<const double2 *>(Pt + u * PS + 48 + 2 * ti);
      const double2 qa = *reinterpret_cast<const double2 *>(Pt + u * PS + 2 * tk);
      const double2 qb = *reinterpret_cast<const double2 *>(Pt + u * PS + 48 + 2 * tk);
      const double p[4] = {pa.x, pa.y, pb.x, pb.y}, q[4] = {qa.x, qa.y, qb.x, qb.y};
#pragma unroll
      for (int a = 0; a < 4; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) acc[a][b] = fma(p[a], q[b], acc[a][b]);
    }
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
      for (int b = 0; b < 4; b++) {
        const int i = r1 + 4 * ti + a, k = r1 + 4 * tk + b;
        if (k <= i) As[i * DS + k] -= acc[a][b];
      }
  }
  for (int idx = t; idx < nrow * SB; idx += nthr) {
    const int u = idx / nrow, i = idx - u * nrow;
    As[(r1 + i) * DS + base + u] = Pt[u * PS + pt_pos(i)];
  }
}

template <bool PROF>
__device__ __forceinline__ void diag_body(double *Lg, int ld, double *Xg, int *info, int col0, int factor, int block_stride,
                                          long long strideL, long long strideX, const int *mask, long long *clk) {
  if (mask && !mask[blockIdx.y]) return;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double *As = reinterpret_cast<double *>(smem_raw);
  double *Pt = As + NB * DS;              // 16-byte aligned (NB*DS is even)
  double *Xb = Pt + SB * PS;
  double *Rt = Xb + SB * XS;
  double *ldiag = Rt + (NB - SB) * XS;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int nclk = 0;
#define DIAG_TICK() do { if (PROF && tid == 0) clk[nclk++] = clock64(); } while (0)
  Lg += (size_t)blockIdx.y * strideL + (size_t)blockIdx.x * block_stride * (size_t)(ld + 1);
  Xg += (size_t)blockIdx.y * strideX + (size_t)blockIdx.x * NB * NB;
  if (info) info += blockIdx.y;
  col0 += blockIdx.x * block_stride;
  DIAG_TICK();
#pragma unroll 1
  for (int it = 0; it < NB * NB / NT; it += 32) {     // 32 independent loads in flight per thread
    double t[32];
#pragma unroll
    for (int q = 0; q < 32; q++) {
      const int idx = tid + (it + q) * NT, i = idx & (NB - 1), k = idx >> 7;
      t[q] = (k <= i) ? Lg[i + (size_t)ld * k] : 0.0;
    }
#pragma unroll
    for (int q = 0; q < 32; q++) {
      const int idx = tid + (it + q) * NT, i = idx & (NB - 1), k = idx >> 7;
      if (k <= i) As[i * DS + k] = t[q];
    }
  }
  __syncthreads();
  if (!factor) {
    // Inverse only (after an update pass): nothing here waits for a factorization, so the four 32 x 32 diagonal inverses run
    // side by side on warps 0-3 (one per SM sub-partition; Xb of blocks 1-3 in the idle panel buffer Pt), then the off-diagonal
    // block rows with all threads.  Same operations per entry as the interleaved loop below: identical bits, 40 -> 15 us.
    if (tid < NB) { const double d = As[tid * DS + tid]; ldiag[tid] = d; As[tid * DS + tid] = 1.0 / d; }
    __syncthreads();
    if (warp < 4) inv32_warp(As, warp == 0 ? Xb : Pt + (warp - 1) * SB * XS, warp * SB, lane);
    __syncthreads();
#pragma unroll 1
    for (int kb = 1; kb < 4; kb++) {
      inv_offdiag_R(As, Rt, kb * SB, tid, NT);
      __syncthreads();
      inv_offdiag_X(As, Pt + (kb - 1) * SB * XS, Rt, kb * SB, tid, NT);
      __syncthreads();
    }
    for (int idx = tid; idx < NB * NB; idx += NT) {
      const int i = idx & (NB - 1), c = idx >> 7;
      Xg[i + (size_t)NB * c] = (c <= i) ? As[c * DS + i] : 0.0;
    }
    return;
  }
  DIAG_TICK();
#pragma unroll 1
  for (int kb = 0; kb < 4; kb++) {
    const int base = kb * SB;
    if (warp == 0) {
      if (factor) { factor32_warp(As, ldiag, base, lane, info, col0); __syncwarp(); }
      DIAG_TICK();
      inv32_warp(As, Xb, base, lane);
      DIAG_TICK();
    } else if (kb > 0 && warp != 4) {
      // warp 4 shares warp 0's SM sub-partition (issue port, FP64 unit): keep it idle while warp 0 runs the serial chain
      inv_offdiag_R(As, Rt, base, tid - 32 - (warp > 4 ? 32 : 0), NT - 64);
    }
    __syncthreads();
    DIAG_TICK();
    if (kb > 0) inv_offdiag_X(As, Xb, Rt, base, tid, NT);
    if (factor && kb < 3) {
      panel_solve(As, Xb, Pt, base, tid, NT);
      __syncthreads();
      DIAG_TICK();
      trailing_update(As, Pt, base, tid, NT);
    }
    __syncthreads();
    DIAG_TICK();
  }
  if (factor) {
    for (int idx = tid; idx < NB * NB; idx += NT) {
      const int i = idx & (NB - 1), k = idx >> 7;
      if (k <= i) Lg[i + (size_t)ld * k] = (k == i) ? ldiag[i] : As[i * DS + k];
    }
  }
  for (int idx = tid; idx < NB * NB; idx += NT) {
    const int i = idx & (NB - 1), c = idx >> 7;
    Xg[i + (size_t)NB * c] = (c <= i) ? As[c * DS + i] : 0.0;
  }
  DIAG_TICK();
#undef DIAG_TICK
}

// factor == 1: the block (lower) is factorised in place, then inverted.  factor == 0: the block already
// holds a Cholesky factor (after an update/downdate sweep) and only the inverse is formed.
// grid.x: diagonal block index (block_stride columns apart), grid.y: batch instance.
__global__ void __launch_bounds__(NT, 1)
k_diag_block(double *Lg, int ld, double *Xg, int *info, int col0, int factor, int block_stride,
             long long strideL, long long strideX, const int *mask) {
  diag_body<false>(Lg, ld, Xg, info, col0, factor, block_stride, strideL, strideX, mask, nullptr);
}
// instrumented twin (tools/microbench.py): thread 0 records clock64() at every phase boundary
__global__ void __launch_bounds__(NT, 1)
k_diag_block_prof(double *Lg, int ld, double *Xg, int factor, long long *clk) {
  diag_body<true>(Lg, ld, Xg, nullptr, 0, factor, 0, 0, 0, nullptr, clk);
}
}  // namespace diag

static int diag_attr() {
  static bool set = false;
  if (!set) {
    QB_CUDA_TRY(cudaFuncSetAttribute(diag::k_diag_block, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)diag::kSmemBytes));
    set = true;
  }
  return 0;
}

// phase clocks of one 128 x 128 factor+inverse (out: up to 32 clock64 samples, returns the count)
int diag_block_phase_clocks(long long *out32) {
  QB_CUDA_TRY(cudaFuncSetAttribute(diag::k_diag_block_prof, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)diag::kSmemBytes));
  const int n = diag::NB;
  std::vector<double> A((size_t)n * n);
  for (int j = 0; j < n; j++) for (int i = 0; i < n; i++) A[i + (size_t)n * j] = (i == j) ? n + 1.0 : 1.0 / (1.0 + abs(i - j));
  double *dA = nullptr, *dX = nullptr; long long *dc = nullptr;
  QB_CUDA_TRY(cudaMalloc(&dA, sizeof(double) * n * n));
  QB_CUDA_TRY(cudaMalloc(&dX, sizeof(double) * n * n));
  QB_CUDA_TRY(cudaMalloc(&dc, sizeof(long long) * 32));
  for (int rep = 0; rep < 2; rep++) {
    QB_CUDA_TRY(cudaMemcpy(dA, A.data(), sizeof(double) * n * n, cudaMemcpyHostToDevice));
    QB_CUDA_TRY(cudaMemset(dc, 0, sizeof(long long) * 32));
    diag::k_diag_block_prof<<<1, diag::NT, diag::kSmemBytes>>>(dA, n, dX, 1, dc);
    QB_CUDA_TRY(cudaDeviceSynchronize());
  }
  QB_CUDA_TRY(cudaMemcpy(out32, dc, sizeof(long long) * 32, cudaMemcpyDeviceToHost));
  cudaFree(dA); cudaFree(dX); cudaFree(dc);
  return 0;
}

// Two-level right-looking blocked Cholesky.  Inner panels are 128 wide (diagonal block factor+inverse in one
// CTA, panel solve as an in-place DMMA GEMM against the inverted block); their rank-128 updates are applied
// only inside the current 512-wide outer block.  Everything to the right of the outer block receives ONE
// rank-512 DMMA update per outer block, which amortises the C-tile read-modify-write of the trailing matrix
// four times better than rank-128 updates.
static int outer_block() {   // 512 by default; QPALM_B200_KOUTER=256|1024 for A/B measurements
  static const int v = [] { const char *e = getenv("QPALM_B200_KOUTER"); const int k = e ? atoi(e) : 512; return (k == 256 || k == 1024) ? k : 512; }();
  return v;
}

// Look-ahead (single matrix, npad > 2 * kOuter): the panel chain of an outer block (diagonal-block kernel on one SM,
// panel solves on npad/128 SMs at most) is latency-bound and leaves most of the GPU idle, while the rank-512 update of
// everything to the right is throughput-bound.  The update is therefore split: the part that lands on the NEXT outer
// block's columns is applied first, and the panel chain of that block then runs on a high-priority stream while the
// rest of the update fills the remaining SMs from the caller's stream.  CTAs of the high-priority stream are placed
// as soon as any SM frees up (an update CTA lasts < 100 us), so the chain is not starved by the queued update.
namespace {
struct LookAhead {
  cudaStream_t hi = nullptr, mid = nullptr;
  cudaEvent_t ev_in = nullptr, ev_chain = nullptr, ev_rest = nullptr, ev_panels = nullptr, ev_slabs = nullptr;
  int device = -1;
  int init() {
    int dev = 0;
    QB_CUDA_TRY(cudaGetDevice(&dev));
    if (hi && dev == device) return 0;
    int lo_p = 0, hi_p = 0;
    QB_CUDA_TRY(cudaDeviceGetStreamPriorityRange(&lo_p, &hi_p));
    QB_CUDA_TRY(cudaStreamCreateWithPriority(&hi, cudaStreamNonBlocking, hi_p));
    QB_CUDA_TRY(cudaStreamCreateWithPriority(&mid, cudaStreamNonBlocking, hi_p));
    QB_CUDA_TRY(cudaEventCreateWithFlags(&ev_panels, cudaEventDisableTiming));
    QB_CUDA_TRY(cudaEventCreateWithFlags(&ev_slabs, cudaEventDisableTiming));
    QB_CUDA_TRY(cudaEventCreateWithFlags(&ev_in, cudaEventDisableTiming));
    QB_CUDA_TRY(cudaEventCreateWithFlags(&ev_chain, cudaEventDisableTiming));
    QB_CUDA_TRY(cudaEventCreateWithFlags(&ev_rest, cudaEventDisableTiming));
    device = dev;
    return 0;
  }
};
thread_local LookAhead g_la;
}  // namespace

int potrf_lower_batched(cudaStream_t s, int nb, int npad, double *L, int ld, long long sL, double *invdiag, long long sX,
                        int *info_dev, const int *mask) {
  if (int e = diag_attr()) return e;
  const int kOuter = outer_block();
  static const bool la_env_off = getenv("QPALM_B200_NO_LOOKAHEAD") != nullptr;
  const bool la = (nb == 1 && !mask && npad > 2 * kOuter && !la_env_off);
  cudaStream_t sc = s;          // stream of the panel chain
  bool rest_pending = false;    // a "rest" update is in flight on s
  bool slabs_pending = false;   // the update of column slabs 1.. of the current outer block is in flight on g_la.mid
  if (la) {
    if (int e = g_la.init()) return e;
    sc = g_la.hi;
    QB_CUDA_TRY(cudaEventRecord(g_la.ev_in, s));
    QB_CUDA_TRY(cudaStreamWaitEvent(sc, g_la.ev_in, 0));
    QB_CUDA_TRY(cudaStreamWaitEvent(g_la.mid, g_la.ev_in, 0));
  }
  for (int J0 = 0; J0 < npad; J0 += kOuter) {
    const int Jend = (J0 + kOuter < npad) ? J0 + kOuter : npad;
    for (int j0 = J0; j0 < Jend; j0 += kPanel) {
      double *Ljj = L + j0 + (size_t)j0 * ld;
      double *Xp = invdiag + (size_t)(j0 / kPanel) * kPanel * kPanel;
      QB_LAUNCH(diag::k_diag_block, dim3(1, nb), diag::NT, diag::kSmemBytes, sc, Ljj, ld, Xp, info_dev, j0, 1, 0, sL, sX, mask);
      const int rem = npad - j0 - kPanel;
      if (rem <= 0) continue;
      double *L21 = Ljj + kPanel;
      // L21 <- A21 * inv(L11)'   (in place, one 128-wide tile column)
      if (int e = dgemm_nt_batched(sc, nb, rem, kPanel, kPanel, nullptr, L21, ld, sL, Xp, kPanel, sX, L21, ld, sL, 1.0, 0.0, false, mask)) return e;
      // rank-128 update of the remaining columns of THIS outer block (all rows below)
      const int wcols = Jend - (j0 + kPanel);
      if (wcols > 0) {
        // those columns also receive the previous outer block's update from the side stream: wait for it once
        if (slabs_pending) { QB_CUDA_TRY(cudaStreamWaitEvent(sc, g_la.ev_slabs, 0)); slabs_pending = false; }
        double *Cin = L + (j0 + kPanel) + (size_t)(j0 + kPanel) * ld;
        if (int e = dgemm_nt_batched(sc, nb, rem, wcols, kPanel, nullptr, L21, ld, sL, L21, ld, sL, Cin, ld, sL, -1.0, 1.0, true, mask)) return e;
      }
    }
    if (slabs_pending) { QB_CUDA_TRY(cudaStreamWaitEvent(sc, g_la.ev_slabs, 0)); slabs_pending = false; }
    // rank-(Jend-J0) update of everything to the right of the outer block
    const int rem = npad - Jend;
    if (rem > 0) {
      const double *P = L + Jend + (size_t)J0 * ld;
      double *A22 = L + Jend + (size_t)Jend * ld;
      const int K = Jend - J0;
      if (la && rem > kOuter) {
        // The next outer block's columns first.  Only its FIRST 128-column slab sits on the panel chain; slabs 1.. run on a
        // second high-priority stream under the next diagonal block + panel solve (they are needed by the first in-block
        // update only).  Both wait for the previous "rest" update, which wrote the same columns.
        QB_CUDA_TRY(cudaEventRecord(g_la.ev_panels, sc));
        if (rest_pending) {
          QB_CUDA_TRY(cudaStreamWaitEvent(sc, g_la.ev_rest, 0));
          QB_CUDA_TRY(cudaStreamWaitEvent(g_la.mid, g_la.ev_rest, 0));
        }
        if (int e = dgemm_nt_batched(sc, 1, rem, kPanel, K, nullptr, P, ld, 0, P, ld, 0, A22, ld, 0, -1.0, 1.0, true, nullptr)) return e;
        QB_CUDA_TRY(cudaStreamWaitEvent(g_la.mid, g_la.ev_panels, 0));
        if (int e = dgemm_nt_batched(g_la.mid, 1, rem - kPanel, kOuter - kPanel, K, nullptr, P + kPanel, ld, 0, P + kPanel, ld, 0,
                                     A22 + (size_t)kPanel * (ld + 1), ld, 0, -1.0, 1.0, true, nullptr)) return e;
        QB_CUDA_TRY(cudaEventRecord(g_la.ev_slabs, g_la.mid));
        slabs_pending = true;
        // the rest, on the caller's stream, concurrent with the next block's panel chain (needs the finished panels only)
        QB_CUDA_TRY(cudaStreamWaitEvent(s, g_la.ev_panels, 0));
        const double *P2 = P + kOuter;
        double *A33 = A22 + (size_t)kOuter * (ld + 1);
        if (int e = dgemm_nt_batched(s, 1, rem - kOuter, rem - kOuter, K, nullptr, P2, ld, 0, P2, ld, 0, A33, ld, 0, -1.0, 1.0, true, nullptr)) return e;
        QB_CUDA_TRY(cudaEventRecord(g_la.ev_rest, s));
        rest_pending = true;
      } else {
        if (rest_pending) { QB_CUDA_TRY(cudaStreamWaitEvent(sc, g_la.ev_rest, 0)); rest_pending = false; }
        if (int e = dgemm_nt_batched(sc, nb, rem, rem, K, nullptr, P, ld, sL, P, ld, sL, A22, ld, sL, -1.0, 1.0, true, mask)) return e;
      }
    }
  }
  if (la) {
    QB_CUDA_TRY(cudaEventRecord(g_la.ev_chain, sc));
    QB_CUDA_TRY(cudaStreamWaitEvent(s, g_la.ev_chain, 0));
  }
  QB_CUDA_TRY(cudaGetLastError());
  return 0;
}

int potrf_lower(cudaStream_t s, int npad, double *L, int ld, double *invdiag, int *info_dev) {
  return potrf_lower_batched(s, 1, npad, L, ld, 0, invdiag, 0, info_dev, nullptr);
}

int trtri_diag_blocks(cudaStream_t s, int npad, const double *L, int ld, double *invdiag) {
  if (int e = diag_attr()) return e;
  const int nblk = npad / kPanel;
  QB_LAUNCH(diag::k_diag_block, nblk, diag::NT, diag::kSmemBytes, s, const_cast<double *>(L), ld, invdiag,
            (int *)nullptr, 0, 0, kPanel, 0LL, 0LL, (const int *)nullptr);
  QB_CUDA_TRY(cudaGetLastError());
  return 0;
}

// ================================================================================================
// blocked triangular solves.  One launch per 128-column block; the CTA that owns the next diagonal
// block also applies that block's inverse, so the following launch finds its x-block ready.
// ================================================================================================
namespace trsv {
constexpr int NB = 128, NT = 256;

// y(0..127) = X * v  (X lower, col-major 128x128) ; result written to out[], all NT threads call.
__device__ void apply_inv_lower(const double *__restrict__ X, const double *v_s, double *out, double *scratch) {
  const int r = threadIdx.x & (NB - 1), h = threadIdx.x >> 7;  // h in {0,1}: column halves
  double acc = 0.0;
  const int c0 = h * 64, c1 = c0 + 64;
#pragma unroll 8
  for (int c = c0; c < c1; c++) acc = fma(X[r + NB * c], v_s[c], acc);
  scratch[h * NB + r] = acc;
  __syncthreads();
  if (h == 0) out[r] = scratch[r] + scratch[NB + r];
}
// y(c) = sum_i X(i,c) v(i)  (X' * v)
__device__ void apply_inv_lower_t(const double *__restrict__ X, const double *v_s, double *out) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int c = warp; c < NB; c += NT / 32) {
    double acc = 0.0;
#pragma unroll
    for (int q = 0; q < 4; q++) acc = fma(X[lane + 32 * q + NB * c], v_s[lane + 32 * q], acc);
    acc = warp_sum(acc);
    if (lane == 0) out[c] = acc;
  }
}

__global__ void __launch_bounds__(NT) k_first_fwd(const double *invdiag0, double *v, long long sX, long long sV, const int *mask) {
  if (mask && !mask[blockIdx.y]) return;
  invdiag0 += (size_t)blockIdx.y * sX; v += (size_t)blockIdx.y * sV;
  __shared__ double vs[NB], scratch[2 * NB];
  if (threadIdx.x < NB) vs[threadIdx.x] = v[threadIdx.x];
  __syncthreads();
  apply_inv_lower(invdiag0, vs, v, scratch);
}

// step b of the forward solve: rows of blocks > b get rhs -= L(rows, block b) * x_b; CTA 0 (block b+1)
// then forms x_{b+1} = inv(L_{b+1,b+1}) rhs_{b+1}.
__global__ void __launch_bounds__(NT) k_fwd_step(const double *__restrict__ L, int ld, const double *invdiag,
                                                 double *v, int b, long long sL, long long sX, long long sV, const int *mask) {
  if (mask && !mask[blockIdx.y]) return;
  L += (size_t)blockIdx.y * sL; invdiag += (size_t)blockIdx.y * sX; v += (size_t)blockIdx.y * sV;
  __shared__ double xs[NB], scratch[2 * NB], rs[NB];
  const int j0 = b * NB, r0 = (b + 1 + blockIdx.x) * NB;
  const int tid = threadIdx.x, r = tid & (NB - 1), h = tid >> 7;
  if (tid < NB) xs[tid] = v[j0 + tid];
  __syncthreads();
  const double *Lp = L + (size_t)(r0 + r) + (size_t)(j0 + h * 64) * ld;
  double acc = 0.0;
#pragma unroll 8
  for (int c = 0; c < 64; c++) acc = fma(Lp[(size_t)c * ld], xs[h * 64 + c], acc);
  scratch[h * NB + r] = acc;
  __syncthreads();
  if (h == 0) {
    const double nv = v[r0 + r] - (scratch[r] + scratch[NB + r]);
    if (blockIdx.x == 0) rs[r] = nv; else v[r0 + r] = nv;
  }
  if (blockIdx.x == 0) {
    __syncthreads();
    apply_inv_lower(invdiag + (size_t)(b + 1) * NB * NB, rs, v + r0, scratch);
  }
}

__global__ void __launch_bounds__(NT) k_first_bwd(const double *invdiag_last, double *v_last, long long sX, long long sV, const int *mask) {
  if (mask && !mask[blockIdx.y]) return;
  invdiag_last += (size_t)blockIdx.y * sX; v_last += (size_t)blockIdx.y * sV;
  __shared__ double vs[NB];
  if (threadIdx.x < NB) vs[threadIdx.x] = v_last[threadIdx.x];
  __syncthreads();
  apply_inv_lower_t(invdiag_last, vs, v_last);
}

// step b of the backward solve (b descending): columns of blocks < b get z -= L(block b rows, cols)' d_b;
// the CTA that owns block b-1 then forms d_{b-1} = inv(L_{b-1,b-1})' z_{b-1}.
__global__ void __launch_bounds__(NT) k_bwd_step(const double *__restrict__ L, int ld, const double *invdiag,
                                                 double *v, int b, long long sL, long long sX, long long sV, const int *mask) {
  if (mask && !mask[blockIdx.y]) return;
  L += (size_t)blockIdx.y * sL; invdiag += (size_t)blockIdx.y * sX; v += (size_t)blockIdx.y * sV;
  __shared__ double ds[NB], zs[NB];
  const int i0 = b * NB, c0 = blockIdx.x * NB;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid < NB) ds[tid] = v[i0 + tid];
  __syncthreads();
  const bool next_diag = ((int)blockIdx.x == b - 1);
  for (int cc = warp * 16; cc < warp * 16 + 16; cc += 4) {
    double acc[4] = {0, 0, 0, 0};
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const double dv = ds[lane + 32 * q];
#pragma unroll
      for (int u = 0; u < 4; u++)
        acc[u] = fma(L[(size_t)(i0 + lane + 32 * q) + (size_t)(c0 + cc + u) * ld], dv, acc[u]);
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const double sacc = warp_sum(acc[u]);
      if (lane == 0) {
        const double nv = v[c0 + cc + u] - sacc;
        if (next_diag) zs[cc + u] = nv; else v[c0 + cc + u] = nv;
      }
    }
  }
  if (next_diag) {
    __syncthreads();
    apply_inv_lower_t(invdiag + (size_t)(b - 1) * NB * NB, zs, v + c0);
  }
}
}  // namespace trsv

// ================================================================================================
// Dataflow triangular solves (single matrix): ONE cooperative launch for forward + backward substitution.
// CTA c owns the 128-row blocks c, c + G, ... : forward it accumulates  t_i = b_i - sum_{j<i} L_ij y_j  tile by tile,
// consuming y_j as soon as its owner has published it (tagged 16-byte packets in global memory, see pk_store), then forms
// y_i = inv(L_ii) t_i and publishes it; backward likewise over the block columns in descending order.  The tile of the
// next step is loaded into registers BEFORE the CTA waits for the packets, so the critical path per block is one L2 round
// trip + two 128 x 128 matrix-vector products from registers / shared memory (measured 3.7 us per block step at n = 8000),
// instead of one kernel launch per block (about 22 us).  The cooperative launch guarantees that all CTAs are co-resident, which the spin-waits need.
// ================================================================================================
namespace flow {
constexpr int NB = 128, NT = 256;
constexpr size_t kSmemBytes = sizeof(double) * (NB * NB + 6 * NB);

__device__ __forceinline__ int ld_acquire(const int *p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release(int *p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// all threads of the CTA return once *f == epoch
__device__ __forceinline__ void wait_flag(const int *f, int epoch) {
  if (threadIdx.x == 0) while (ld_acquire(f) != epoch) {}
  __syncthreads();
}
// publish after the CTA's global writes
__device__ __forceinline__ void publish(int *f, int epoch) {
  __syncthreads();
  if (threadIdx.x == 0) { __threadfence(); st_release(f, epoch); }
}
// Solution blocks travel between CTAs as TAGGED PACKETS: one 16-byte store {lo32, epoch, hi32, epoch} per double, the reader
// spins on its own packet until both tags carry the launch's epoch (tear-proof at 8-byte granularity -- the layout of NCCL's LL
// protocol).  Value and "it is there" arrive in ONE L2 round trip and the producer needs neither __threadfence() nor a separate
// flag store; the first version (fence -> flag -> acquire poll -> dependent load of the values) paid three on the chain of every
// block.  Measured effect: 66 -> 60 us per solve at n = 1000, 477 -> 469 us at n = 8000 (the step is bound elsewhere there).  Epoch-stamped, so nothing is cleared between launches.
__device__ __forceinline__ void pk_store(uint4 *pk, double v, int epoch) {
  const long long b = __double_as_longlong(v);
  asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %2};" ::"l"(pk), "r"((unsigned)(b & 0xffffffffll)), "r"((unsigned)epoch),
               "r"((unsigned)((unsigned long long)b >> 32)) : "memory");
}
__device__ __forceinline__ double pk_wait(const uint4 *pk, int epoch) {
  unsigned lo, t0, hi, t1;
  do {
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(lo), "=r"(t0), "=r"(hi), "=r"(t1) : "l"(pk) : "memory");
  } while (t0 != (unsigned)epoch || t1 != (unsigned)epoch);
  return __longlong_as_double((long long)(((unsigned long long)hi << 32) | lo));
}
__device__ __forceinline__ void load_block_to_smem(double *Xs, const double *Xg) {
  const double2 *src = reinterpret_cast<const double2 *>(Xg);
  double2 *dst = reinterpret_cast<double2 *>(Xs);
#pragma unroll 8
  for (int idx = threadIdx.x; idx < NB * NB / 2; idx += NT) dst[idx] = __ldcg(src + idx);
}

__global__ void __launch_bounds__(NT, 1)
k_solve_flow(const double *__restrict__ L, int ld, const double *__restrict__ X, double *v, int nblk, uint4 *packets, int epoch) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double *Xs = reinterpret_cast<double *>(smem_raw);   // inverse of the current diagonal block, column-major
  double *xs = Xs + NB * NB;                           // incoming solution block
  double *scratch = xs + NB;                           // 2 * NB partial sums
  double *rs = scratch + 2 * NB;                       // right-hand side of the diagonal solve
  uint4 *pk_f = packets, *pk_b = packets + (size_t)nblk * NB;   // forward (y) and backward (x) blocks
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, r = tid & (NB - 1), h = tid >> 7;
  const int G = gridDim.x;

  // ---------------- forward: L y = b ----------------
  for (int i = blockIdx.x; i < nblk; i += G) {
    load_block_to_smem(Xs, X + (size_t)i * NB * NB);
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    for (int j = 0; j < i; j++) {
      const double *Lp = L + (size_t)(i * NB + r) + (size_t)(j * NB + h * 64) * ld;
      double t[64];
#pragma unroll
      for (int c = 0; c < 64; c++) t[c] = Lp[(size_t)c * ld];        // in flight while waiting for y_j
      __syncthreads();   // the previous step's readers of xs are done
      if (tid < NB) xs[tid] = pk_wait(pk_f + (size_t)j * NB + tid, epoch);
      __syncthreads();
#pragma unroll
      for (int c = 0; c < 64; c += 4) {
        a0 = fma(t[c], xs[h * 64 + c], a0);
        a1 = fma(t[c + 1], xs[h * 64 + c + 1], a1);
        a2 = fma(t[c + 2], xs[h * 64 + c + 2], a2);
        a3 = fma(t[c + 3], xs[h * 64 + c + 3], a3);
      }
    }
    scratch[h * NB + r] = (a0 + a1) + (a2 + a3);
    __syncthreads();
    if (h == 0) rs[r] = __ldcg(v + (size_t)i * NB + r) - (scratch[r] + scratch[NB + r]);
    __syncthreads();
    {   // y_i = inv(L_ii) rs   (Xs lower triangular, zeros above)
      double b0 = 0.0, b1 = 0.0, b2 = 0.0, b3 = 0.0;
      const int c0 = h * 64;
#pragma unroll
      for (int c = 0; c < 64; c += 4) {
        b0 = fma(Xs[r + NB * (c0 + c)], rs[c0 + c], b0);
        b1 = fma(Xs[r + NB * (c0 + c + 1)], rs[c0 + c + 1], b1);
        b2 = fma(Xs[r + NB * (c0 + c + 2)], rs[c0 + c + 2], b2);
        b3 = fma(Xs[r + NB * (c0 + c + 3)], rs[c0 + c + 3], b3);
      }
      scratch[h * NB + r] = (b0 + b1) + (b2 + b3);
      __syncthreads();
      if (h == 0) {
        const double yv = scratch[r] + scratch[NB + r];
        v[(size_t)i * NB + r] = yv;                       // for this CTA's own backward step
        pk_store(pk_f + (size_t)i * NB + r, yv, epoch);    // for the CTAs below
      }
    }
    __syncthreads();   // scratch / rs / Xs are reused by the next block of this CTA
  }

  // ---------------- backward: L' x = y ----------------
  const int last = blockIdx.x + ((nblk - 1 - blockIdx.x) / G) * G;      // this CTA's highest block
  for (int j = last; j >= 0; j -= G) {
    __syncthreads();
    load_block_to_smem(Xs, X + (size_t)j * NB * NB);
    double acc[16];
#pragma unroll
    for (int u = 0; u < 16; u++) acc[u] = 0.0;
    for (int i = nblk - 1; i > j; i--) {
      const double *Lp = L + (size_t)(i * NB + lane) + (size_t)(j * NB + warp * 16) * ld;
      double t[16][4];
#pragma unroll
      for (int u = 0; u < 16; u++)
#pragma unroll
        for (int q = 0; q < 4; q++) t[u][q] = Lp[(size_t)u * ld + 32 * q];
      __syncthreads();   // the previous step's readers of xs are done
      if (tid < NB) xs[tid] = pk_wait(pk_b + (size_t)i * NB + tid, epoch);
      __syncthreads();
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const double dv = xs[lane + 32 * q];
#pragma unroll
        for (int u = 0; u < 16; u++) acc[u] = fma(t[u][q], dv, acc[u]);
      }
    }
    // y_j was written to v by THIS CTA in its forward pass (CTA barriers since then order it for every thread here)
#pragma unroll
    for (int u = 0; u < 16; u++) {
      const double sacc = warp_sum(acc[u]);
      if (lane == 0) rs[warp * 16 + u] = __ldcg(v + (size_t)j * NB + warp * 16 + u) - sacc;
    }
    __syncthreads();
    // x_j = inv(L_jj)' rs : column c of Xs dotted with rs
    for (int c = warp; c < NB; c += NT / 32) {
      double a = 0.0;
#pragma unroll
      for (int q = 0; q < 4; q++) a = fma(Xs[lane + 32 * q + NB * c], rs[lane + 32 * q], a);
      a = warp_sum(a);
      if (lane == 0) { v[(size_t)j * NB + c] = a; pk_store(pk_b + (size_t)j * NB + c, a, epoch); }
    }
  }
}

struct FlowState { uint4 *flags = nullptr; int cap = 0; int epoch = 0; int max_grid = 0; };   // flags: the packet ring, 2 * nblk * NB packets
static std::mutex g_flow_mu;
static std::map<cudaStream_t, FlowState> g_flow;
}  // namespace flow

static thread_local int g_solve_last_grid = 0;   // cooperative grid of this thread's last chol_solve, 0: per-block launches
int chol_solve_last_grid() { return g_solve_last_grid; }

// returns 0 when the dataflow solve ran, 1 when it is not available (caller falls back to the per-block launches), < 0 on error
static int chol_solve_flow(cudaStream_t s, int npad, const double *L, int ld, const double *invdiag, double *v) {
  static const bool off = getenv("QPALM_B200_NO_FLOW_SOLVE") != nullptr;
  if (off) return 1;
  const int nblk = npad / kPanel;
  flow::FlowState st;
  {
    std::lock_guard<std::mutex> lk(flow::g_flow_mu);
    flow::FlowState &ref = flow::g_flow[s];
    if (ref.max_grid == 0) {
      int dev = 0, coop = 0, sms = 0, per_sm = 0;
      QB_CUDA_TRY(cudaGetDevice(&dev));
      QB_CUDA_TRY(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
      QB_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
      QB_CUDA_TRY(cudaFuncSetAttribute(flow::k_solve_flow, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)flow::kSmemBytes));
      QB_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, flow::k_solve_flow, flow::NT, flow::kSmemBytes));
      ref.max_grid = coop ? sms * per_sm : -1;
    }
    if (ref.max_grid <= 0) return 1;
    if (ref.cap < 2 * nblk) {
      if (ref.flags) QB_CUDA_TRY(cudaFree(ref.flags));
      ref.cap = 2 * nblk + 64;
      QB_CUDA_TRY(cudaMalloc(&ref.flags, sizeof(uint4) * (size_t)ref.cap * flow::NB));
      QB_CUDA_TRY(cudaMemsetAsync(ref.flags, 0, sizeof(uint4) * (size_t)ref.cap * flow::NB, s));
      ref.epoch = 0;
    }
    ref.epoch++;
    st = ref;
  }
  int grid = nblk < st.max_grid ? nblk : st.max_grid;
  int nblk_arg = nblk, ld_arg = ld, epoch = st.epoch;
  uint4 *flags = st.flags;
  void *args[] = {(void *)&L, (void *)&ld_arg, (void *)&invdiag, (void *)&v, (void *)&nblk_arg, (void *)&flags, (void *)&epoch};
  const bool prof = g_prof_on && prof_begin("flow::k_solve_flow", s);
  const cudaError_t err = cudaLaunchCooperativeKernel((const void *)flow::k_solve_flow, dim3(grid), dim3(flow::NT), args, flow::kSmemBytes, s);
  if (prof) prof_end(s);
  if (err != cudaSuccess) {
    // e.g. a partitioned GPU (MPS / MIG slice) that cannot co-schedule the grid: remember it and use the per-block launches
    (void)cudaGetLastError();
    std::lock_guard<std::mutex> lk(flow::g_flow_mu);
    flow::g_flow[s].max_grid = -1;
    return 1;
  }
  ++g_kernel_launches;
  g_solve_last_grid = grid;
  return 0;
}

// frees the per-stream flag buffer of the dataflow solves (call before destroying the stream)
void chol_solve_release(cudaStream_t s) {
  std::lock_guard<std::mutex> lk(flow::g_flow_mu);
  auto it = flow::g_flow.find(s);
  if (it == flow::g_flow.end()) return;
  if (it->second.flags) cudaFree(it->second.flags);
  flow::g_flow.erase(it);
}

int chol_solve_batched(cudaStream_t s, int nb, int npad, const double *L, int ld, long long sL, const double *invdiag,
                       long long sX, double *v, long long sV, const int *mask) {
  const int nblk = npad / kPanel;
  QB_LAUNCH(trsv::k_first_fwd, dim3(1, nb), trsv::NT, 0, s, invdiag, v, sX, sV, mask);
  for (int b = 0; b + 1 < nblk; b++)
    QB_LAUNCH(trsv::k_fwd_step, dim3(nblk - 1 - b, nb), trsv::NT, 0, s, L, ld, invdiag, v, b, sL, sX, sV, mask);
  QB_LAUNCH(trsv::k_first_bwd, dim3(1, nb), trsv::NT, 0, s, invdiag + (size_t)(nblk - 1) * kPanel * kPanel,
            v + (size_t)(nblk - 1) * kPanel, sX, sV, mask);
  for (int b = nblk - 1; b >= 1; b--)
    QB_LAUNCH(trsv::k_bwd_step, dim3(b, nb), trsv::NT, 0, s, L, ld, invdiag, v, b, sL, sX, sV, mask);
  QB_CUDA_TRY(cudaGetLastError());
  return 0;
}
int chol_solve(cudaStream_t s, int npad, const double *L, int ld, const double *invdiag, double *v) {
  g_solve_last_grid = 0;
  if (npad > 2 * kPanel) {
    const int rc = chol_solve_flow(s, npad, L, ld, invdiag, v);
    if (rc <= 0) return -rc;
  }
  return chol_solve_batched(s, 1, npad, L, ld, 0, invdiag, 0, v, 0, nullptr);
}

// ================================================================================================
// rank-k update / downdate, k <= 8 per sweep.
//
// CHOLMOD's kernel (Modify/t_cholmod_updown_numkr.c:289-376) walks the columns j of a unit-lower
// L D L' factor; per column and per rank vector r it forms (alpha_r, gamma_r) from w_r[j] and d_j and
// then, for every row i below j:   w_r[i] -= w_r[j] * L[i][j];  L[i][j] -= gamma_r * w_r[i].
// Here the factor is L L' (d_j = l_jj^2, unit column = column / l_jj) and the sweep is panelised in
// 32-column panels: the data-dependent scalar recurrence of a panel only needs the panel's 32 x 32
// diagonal block and its 32 rows of W ("phase 1", one warp, registers + shuffles); every row below is
// then transformed independently with the 32 x (2 + 2k) coefficients of the panel ("phase 2", one
// thread per row, coalesced column-major accesses).  Phase 1 of panel p+1 is executed by the phase-2
// CTA that owns those rows, so a sweep costs one launch per panel.
// ================================================================================================
namespace updown {
constexpr int PB = 32, KMAX = 8, CO = 2 + 2 * KMAX, NT = 128;

// one warp; lane = row of the diagonal block.  Reads/writes L block and W rows in global memory.
__device__ void phase1(double *Lg, int ld, double *Wg, int ldw, int k, int sign, int j0,
                       double *alpha_state, double *coef_out, int *info) {
  const int lane = threadIdx.x & 31;
  double lrow[PB], w[KMAX], alpha[KMAX];
#pragma unroll
  for (int j = 0; j < PB; j++) lrow[j] = (j <= lane) ? Lg[(size_t)(j0 + lane) + (size_t)(j0 + j) * ld] : 0.0;
#pragma unroll
  for (int r = 0; r < KMAX; r++) {
    w[r] = (r < k) ? Wg[(size_t)(j0 + lane) + (size_t)r * ldw] : 0.0;
    alpha[r] = (r < k) ? alpha_state[r] : 1.0;
  }
  const double sg = (double)sign;
  bool bad = false;
#pragma unroll
  for (int j = 0; j < PB; j++) {
    const double ljj = __shfl_sync(0xffffffffu, lrow[j], j);
    const double winv = 1.0 / ljj;
    double dj = ljj * ljj;
    double t = lrow[j] * winv;  // unit-column entry of this lane's row
#pragma unroll
    for (int r = 0; r < KMAX; r++) {
      if (r < k) {
        const double wj = __shfl_sync(0xffffffffu, w[r], j);
        const double a = alpha[r] + sg * (wj * wj) / dj;
        dj *= a;
        const double gam = -sg * wj / dj;
        dj /= alpha[r];
        alpha[r] = a;
        if (lane > j) { w[r] -= wj * t; t -= gam * w[r]; }
        if (lane == 0) { coef_out[j * CO + 2 + r] = wj; coef_out[j * CO + 2 + KMAX + r] = gam; }
      }
    }
    const double lnew = sqrt(dj);
    if (!(dj > 0.0)) bad = true;
    if (lane > j) lrow[j] = t * lnew;
    else if (lane == j) lrow[j] = lnew;
    if (lane == 0) { coef_out[j * CO + 0] = winv; coef_out[j * CO + 1] = lnew; }
  }
#pragma unroll
  for (int j = 0; j < PB; j++)
    if (j <= lane) Lg[(size_t)(j0 + lane) + (size_t)(j0 + j) * ld] = lrow[j];
#pragma unroll
  for (int r = 0; r < KMAX; r++)
    if (r < k) {
      Wg[(size_t)(j0 + lane) + (size_t)r * ldw] = 0.0;
      if (lane == 0) alpha_state[r] = alpha[r];
    }
  if (bad && lane == 0 && info) atomicExch(info, 1);
}

__global__ void __launch_bounds__(32) k_first(double *L, int ld, double *W, int ldw, int k, int sign,
                                               double *alpha_state, double *coef, int *info) {
  if (threadIdx.x < KMAX) alpha_state[threadIdx.x] = 1.0;
  __syncwarp();
  phase1(L, ld, W, ldw, k, sign, 0, alpha_state, coef, info);
}

// panel p (columns j0..j0+31): rows i >= j0+32.  coef_in: coefficients of panel p; CTA 0 afterwards
// runs phase 1 of panel p+1 (rows j0+32..j0+63 are the first 32 rows it owns) into coef_out.
__global__ void __launch_bounds__(NT) k_panel(double *L, int ld, double *W, int ldw, int k, int sign, int j0,
                                              int npad, double *alpha_state, const double *coef_in,
                                              double *coef_out, int *info) {
  __shared__ double cs[PB * CO];
  for (int i = threadIdx.x; i < PB * CO; i += NT) cs[i] = coef_in[i];
  __syncthreads();
  const int i = j0 + PB + blockIdx.x * NT + threadIdx.x;
  if (i < npad) {
    double w[KMAX];
#pragma unroll
    for (int r = 0; r < KMAX; r++) w[r] = (r < k) ? W[(size_t)i + (size_t)r * ldw] : 0.0;
    double *Lp = L + (size_t)i + (size_t)j0 * ld;
#pragma unroll 4
    for (int j = 0; j < PB; j++) {
      double t = Lp[(size_t)j * ld] * cs[j * CO + 0];
#pragma unroll
      for (int r = 0; r < KMAX; r++) {
        if (r < k) { w[r] -= cs[j * CO + 2 + r] * t; t -= cs[j * CO + 2 + KMAX + r] * w[r]; }
      }
      Lp[(size_t)j * ld] = t * cs[j * CO + 1];
    }
#pragma unroll
    for (int r = 0; r < KMAX; r++)
      if (r < k) W[(size_t)i + (size_t)r * ldw] = w[r];
  }
  if (blockIdx.x == 0 && j0 + PB < npad) {
    __syncthreads();  // this CTA's own global writes (rows j0+32..j0+63) are visible to its warp 0
    if (threadIdx.x < 32) phase1(L, ld, W, ldw, k, sign, j0 + PB, alpha_state, coef_out, info);
  }
}
}  // namespace updown

int chol_updown(cudaStream_t s, int npad, double *L, int ld, double *W, int ldw, int k, int sign,
                double *coef, int *info_dev) {
  using namespace updown;
  if (k <= 0) return 0;
  if (k > KMAX) return 1;
  double *alpha_state = coef + 2 * PB * CO;
  QB_LAUNCH(k_first, 1, 32, 0, s, L, ld, W, ldw, k, sign, alpha_state, coef, info_dev);
  const int npanels = npad / PB;
  for (int p = 0; p < npanels; p++) {
    const int j0 = p * PB;
    const int rows = npad - j0 - PB;
    if (rows <= 0) break;
    double *cin = coef + (size_t)(p & 1) * PB * CO, *cout = coef + (size_t)((p + 1) & 1) * PB * CO;
    QB_LAUNCH(k_panel, cdiv(rows, NT), NT, 0, s, L, ld, W, ldw, k, sign, j0, npad, alpha_state, cin, cout,
              info_dev);
  }
  QB_CUDA_TRY(cudaGetLastError());
  return 0;
}

// ================================================================================================
// small helpers
// ================================================================================================
__global__ void k_copy_lower_add_diag(int n, int npad, const double *__restrict__ H, double *__restrict__ L,
                                      int ld, double diag_add) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int j = blockIdx.y;
  if (i >= npad || i < j) return;
  double v;
  if (i < n && j < n) v = H[(size_t)i + (size_t)j * ld] + ((i == j) ? diag_add : 0.0);
  else v = (i == j) ? 1.0 : 0.0;
  L[(size_t)i + (size_t)j * ld] = v;
}
int copy_lower_add_diag(cudaStream_t s, int n, int npad, const double *H, double *L, int ld, double diag_add) {
  dim3 grid(cdiv(npad, 256), npad);
  QB_LAUNCH(k_copy_lower_add_diag, grid, 256, 0, s, n, npad, H, L, ld, diag_add);
  QB_CUDA_TRY(cudaGetLastError());
  return 0;
}

// row i of the symmetric matrix: entries (i, j<=i) from row i of the lower triangle, (i, j>i) from column i
__global__ void k_sym_abs_rowsums(int n, const double *__restrict__ H, int ld, double *out) {
  __shared__ double scratch[32];
  const int i = blockIdx.x;
  double acc = 0.0;
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    const double v = (j <= i) ? H[(size_t)i + (size_t)j * ld] : H[(size_t)j + (size_t)i * ld];
    acc += fabs(v);
  }
  acc = block_red<RED_SUM>(acc, scratch);
  if (threadIdx.x == 0) out[i] = acc;
}
int sym_abs_rowsums(cudaStream_t s, int n, const double *H, int ld, double *out) {
  QB_LAUNCH(k_sym_abs_rowsums, n, 256, 0, s, n, H, ld, out);
  QB_CUDA_TRY(cudaGetLastError());
  return 0;
}

}  // namespace qb
