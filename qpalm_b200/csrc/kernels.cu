// kernels.cu -- sparse/dense matrix-vector products, fused vector steps, reductions, the line search
// (breakpoints -> stable LSD radix sort -> prefix scan -> root select) and Ruiz scaling kernels.
//
// Element-wise arithmetic follows the operation order of the reference loops exactly and this file is
// compiled with -fmad=false, so Axys, z, the active set, alpha, delta and the breakpoints s = alpha/delta
// are bit-identical to the reference at identical inputs (SURVEY.md 8(a) rows a3-a5, a12).
#include "engine.cuh"
#include <vector>
#include <chrono>
#include <thread>
#include <mutex>
#include <math.h>
#include <string.h>

namespace qb {

constexpr int kRedBlocks = 512;   // max grid of a reducing kernel; partials are [S_COUNT][kRedBlocks]
constexpr int kRedThreads = 256;
constexpr double kInfty = 1e20;

__constant__ int c_slot_op[S_COUNT];

static int red_grid(int len) { int g = cdiv(len, kRedThreads); return g < 1 ? 1 : (g > kRedBlocks ? kRedBlocks : g); }

// ------------------------------------------------------------------------------------------------
// allocation / transfers
// ------------------------------------------------------------------------------------------------
int dev_alloc(void **p, size_t bytes) {
  if (bytes == 0) bytes = 8;
  QB_CUDA_TRY(cudaMalloc(p, bytes));
  QB_CUDA_TRY(cudaMemset(*p, 0, bytes));
  return 0;
}
// carve from the engine's zero-filled slab; falls back to an individual allocation when the slab is exhausted
static int arena_alloc(Engine *e, void **p, size_t bytes) {
  if (bytes == 0) bytes = 8;
  const size_t need = (bytes + 255) & ~(size_t)255;
  if (e->arena && e->arena_off + need <= e->arena_cap) { *p = e->arena + e->arena_off; e->arena_off += need; return 0; }
  return dev_alloc(p, bytes);
}
static bool in_arena(const Engine *e, const void *p) {
  return e->arena && (const char *)p >= e->arena && (const char *)p < e->arena + e->arena_cap;
}
int upload(Engine *e, double *dst, const double *src, int len) {
  if (len > 0) QB_CUDA_TRY(cudaMemcpyAsync(dst, src, sizeof(double) * (size_t)len, cudaMemcpyHostToDevice, e->stream));
  return 0;
}
int download(Engine *e, double *dst, const double *src, int len) {
  if (len > 0) QB_CUDA_TRY(cudaMemcpyAsync(dst, src, sizeof(double) * (size_t)len, cudaMemcpyDeviceToHost, e->stream));
  QB_CUDA_TRY(cudaStreamSynchronize(e->stream));
  return 0;
}
__global__ void k_widen(const int *src, long long *dst, int len) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < len) dst[i] = src[i];
}
int download_int(Engine *e, long long *dst, const int *src, int len) {
  if (len <= 0) return 0;
  long long *tmp = nullptr;
  QB_CUDA_TRY(cudaMalloc(&tmp, sizeof(long long) * (size_t)len));
  QB_LAUNCH(k_widen, cdiv(len, 256), 256, 0, e->stream, src, tmp, len);
  QB_CUDA_TRY(cudaMemcpyAsync(dst, tmp, sizeof(long long) * (size_t)len, cudaMemcpyDeviceToHost, e->stream));
  QB_CUDA_TRY(cudaStreamSynchronize(e->stream));
  cudaFree(tmp);
  return 0;
}
int sync_scalars(Engine *e) {
  QB_CUDA_TRY(cudaMemcpyAsync(e->scal_host, e->scal_dev, sizeof(double) * S_COUNT, cudaMemcpyDeviceToHost, e->stream));
  // the factorization status rides along (first non-positive pivot of the last Cholesky / L S L', 0 = fine)
  QB_CUDA_TRY(cudaMemcpyAsync(e->info_host, e->info_dev, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
  QB_CUDA_TRY(cudaStreamSynchronize(e->stream));
  return 0;
}

// ------------------------------------------------------------------------------------------------
// plain vector kernels
// ------------------------------------------------------------------------------------------------
__global__ void k_copy(const double *__restrict__ s, double *__restrict__ d, int len) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < len; i += gridDim.x * blockDim.x) d[i] = s[i];
}
__global__ void k_set(double *d, double v, int len) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < len; i += gridDim.x * blockDim.x) d[i] = v;
}
__global__ void k_seti(int *d, int v, int len) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < len; i += gridDim.x * blockDim.x) d[i] = v;
}
__global__ void k_copyi(const int *s, int *d, int len) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < len; i += gridDim.x * blockDim.x) d[i] = s[i];
}
__global__ void k_axpy(double a, const double *__restrict__ x, double *y, int len) {   // y = y + a*x
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < len; i += gridDim.x * blockDim.x) y[i] = y[i] + a * x[i];
}
__global__ void k_scale(double a, double *x, int len) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < len; i += gridDim.x * blockDim.x) x[i] *= a;
}
__global__ void k_ewprod(const double *a, const double *b, double *c, int len) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < len; i += gridDim.x * blockDim.x) c[i] = a[i] * b[i];
}
static int vgrid(int len) { int g = cdiv(len, 256); return g < 1 ? 1 : (g > 2048 ? 2048 : g); }
int vec_copy(Engine *e, const double *src, double *dst, int len) { if (len > 0) QB_LAUNCH(k_copy, vgrid(len), 256, 0, e->stream, src, dst, len); return 0; }
int vec_set(Engine *e, double *dst, double v, int len) { if (len > 0) QB_LAUNCH(k_set, vgrid(len), 256, 0, e->stream, dst, v, len); return 0; }
int vec_axpy(Engine *e, double a, const double *x, double *y, int len) { if (len > 0) QB_LAUNCH(k_axpy, vgrid(len), 256, 0, e->stream, a, x, y, len); return 0; }
int vec_scale(Engine *e, double a, double *x, int len) { if (len > 0) QB_LAUNCH(k_scale, vgrid(len), 256, 0, e->stream, a, x, len); return 0; }
int vec_ewprod(Engine *e, const double *a, const double *b, double *c, int len) { if (len > 0) QB_LAUNCH(k_ewprod, vgrid(len), 256, 0, e->stream, a, b, c, len); return 0; }
static int ivec_set(Engine *e, int *dst, int v, int len) { if (len > 0) QB_LAUNCH(k_seti, vgrid(len), 256, 0, e->stream, dst, v, len); return 0; }
static int ivec_copy(Engine *e, const int *s, int *d, int len) { if (len > 0) QB_LAUNCH(k_copyi, vgrid(len), 256, 0, e->stream, s, d, len); return 0; }

// ------------------------------------------------------------------------------------------------
// reductions: every reducing kernel writes partials[slot * kRedBlocks + blockIdx.x]; k_finalize folds
// the first `nblocks` partials of each requested slot (fixed order) into scal[slot].
// ------------------------------------------------------------------------------------------------
struct SlotList { int n; int slot[24]; };

__device__ __forceinline__ void write_partial(double *partials, int slot, double v) {
  partials[slot * kRedBlocks + blockIdx.x] = v;
}
template <int OP>
__device__ __forceinline__ void block_partial(double v, double *scratch, double *partials, int slot) {
  v = block_red<OP>(v, scratch);
  if (threadIdx.x == 0) write_partial(partials, slot, v);
}
__global__ void k_finalize(SlotList sl, const double *__restrict__ partials, int nblocks, double *scal) {
  __shared__ double scratch[32];
  const int slot = sl.slot[blockIdx.x];
  const int op = c_slot_op[slot];
  double ident = (op == RED_SUM) ? 0.0 : (op == RED_MAX ? -1.0e300 : 1.0e300);
  double v = ident;
  for (int i = threadIdx.x; i < nblocks; i += blockDim.x) {
    const double p = partials[slot * kRedBlocks + i];
    v = (op == RED_SUM) ? v + p : (op == RED_MAX ? fmax(v, p) : fmin(v, p));
  }
  if (op == RED_SUM) v = block_red<RED_SUM>(v, scratch);
  else if (op == RED_MAX) v = block_red<RED_MAX>(v, scratch);
  else v = block_red<RED_MIN>(v, scratch);
  if (threadIdx.x == 0) scal[slot] = v;
}
static int finalize(Engine *e, std::initializer_list<int> slots, int nblocks) {
  SlotList sl; sl.n = 0;
  for (int s : slots) sl.slot[sl.n++] = s;
  QB_LAUNCH(k_finalize, sl.n, 256, 0, e->stream, sl, e->partials, nblocks, e->scal_dev);
  return 0;
}
int init_slot_ops() {
  int ops[S_COUNT];
  for (int i = 0; i < S_COUNT; i++) ops[i] = RED_SUM;
  const int maxs[] = {S_PRI_RES, S_PRI_RES_RAW, S_NORM_AX, S_NORM_Z, S_NORM_EDY, S_ADX_MAX, S_DUA_RES, S_DUA2_RES,
                      S_NORM_QX, S_NORM_Q, S_NORM_ATYH, S_NORM_ATDY, S_NORM_DDX, S_TMP4, S_TMP5, S_LMAX};
  for (int s : maxs) ops[s] = RED_MAX;
  ops[S_ADX_MIN] = RED_MIN;
  QB_CUDA_TRY(cudaMemcpyToSymbol(c_slot_op, ops, sizeof(ops)));
  return 0;
}

// ------------------------------------------------------------------------------------------------
// matrix-vector products
// ------------------------------------------------------------------------------------------------
// CSR gather: one warp per row (also serves A'y through the CSC arrays and Q through its full CSR)
__global__ void __launch_bounds__(256) k_csr_spmv(int rows, const int *__restrict__ p, const int *__restrict__ ci,
                                                  const double *__restrict__ v, const double *__restrict__ x, double *y) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int b = p[row], en = p[row + 1];
  // 128-bit value loads / 64-bit index loads on even-aligned pairs (the arrays carry two elements of padding, the first and
  // last pair of a row are masked); two accumulators per lane, fixed order
  double acc0 = 0.0, acc1 = 0.0;
  for (int k = (b & ~1) + 2 * lane; k < en; k += 64) {
    const double2 vv = *reinterpret_cast<const double2 *>(v + k);
    const int2 cc = *reinterpret_cast<const int2 *>(ci + k);
    if (k >= b) acc0 = fma(vv.x, __ldg(x + cc.x), acc0);
    if (k + 1 < en) acc1 = fma(vv.y, __ldg(x + cc.y), acc1);
  }
  const double acc = warp_sum(acc0 + acc1);
  if (lane == 0) y[row] = acc;
}
// dense, column dots: y[k] = sum_i M[i + ld*k] x[i]; one warp per column, 4 independent accumulators
__global__ void __launch_bounds__(256) k_gemv_cols(int len, int ncols, int ld, const double *__restrict__ M,
                                                   const double *__restrict__ x, double *y) {
  const int lane = threadIdx.x & 31;
  const int col = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (col >= ncols) return;
  const double *c = M + (size_t)col * ld;
  double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
  int i = lane;
  for (; i + 96 < len; i += 128) {
    a0 = fma(c[i], __ldg(x + i), a0);
    a1 = fma(c[i + 32], __ldg(x + i + 32), a1);
    a2 = fma(c[i + 64], __ldg(x + i + 64), a2);
    a3 = fma(c[i + 96], __ldg(x + i + 96), a3);
  }
  for (; i < len; i += 32) a0 = fma(c[i], __ldg(x + i), a0);
  double acc = warp_sum((a0 + a1) + (a2 + a3));
  if (lane == 0) y[col] = acc;
}
// dense, row sums: partial[s][i] = sum_{k in split s} M[i + ld*k] x[k]; 128 rows per CTA
__global__ void __launch_bounds__(128) k_gemv_rows(int nrows, int ncols, int ld, const double *__restrict__ M,
                                                   const double *__restrict__ x, double *partial, int cols_per_split) {
  const int i = blockIdx.x * 128 + threadIdx.x;
  const int k0 = blockIdx.y * cols_per_split;
  const int k1 = min(ncols, k0 + cols_per_split);
  if (i >= nrows) return;
  const double *r = M + i;
  double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
  int k = k0;
  for (; k + 3 < k1; k += 4) {
    a0 = fma(r[(size_t)k * ld], __ldg(x + k), a0);
    a1 = fma(r[(size_t)(k + 1) * ld], __ldg(x + k + 1), a1);
    a2 = fma(r[(size_t)(k + 2) * ld], __ldg(x + k + 2), a2);
    a3 = fma(r[(size_t)(k + 3) * ld], __ldg(x + k + 3), a3);
  }
  for (; k < k1; k++) a0 = fma(r[(size_t)k * ld], __ldg(x + k), a0);
  partial[(size_t)blockIdx.y * nrows + i] = (a0 + a1) + (a2 + a3);
}
__global__ void k_sum_splits(int nrows, int splits, const double *__restrict__ partial, double *y) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nrows) return;
  double acc = 0.0;
  for (int s = 0; s < splits; s++) acc += partial[(size_t)s * nrows + i];
  y[i] = acc;
}
static int gemv_rows(Engine *e, int nrows, int ncols, int ld, const double *M, const double *x, double *y) {
  int splits = e->gemv_splits;
  if (splits > ncols) splits = ncols < 1 ? 1 : ncols;
  const int cps = cdiv(ncols, splits);
  splits = cdiv(ncols, cps);
  dim3 grid(cdiv(nrows, 128), splits);
  QB_LAUNCH(k_gemv_rows, grid, 128, 0, e->stream, nrows, ncols, ld, M, x, e->gemv_partials, cps);
  QB_LAUNCH(k_sum_splits, cdiv(nrows, 256), 256, 0, e->stream, nrows, splits, e->gemv_partials, y);
  return 0;
}
int spmv_A(Engine *e, const double *x, double *y) {
  if (e->m == 0) return 0;
  e->n_spmv++;
  if (e->A_dense) {
    if (e->m_loc > 0) QB_LAUNCH(k_gemv_cols, cdiv(e->m_loc, 8), 256, 0, e->stream, e->n, e->m_loc, e->n, e->At, x, y + e->m_lo);
    if (e->sh_world > 1) return shard_allgather(y, (size_t)e->m_cap, e->stream);   // every rank ends with the full A x
  } else QB_LAUNCH(k_csr_spmv, cdiv(e->m, 8), 256, 0, e->stream, e->m, e->A_csr.p, e->A_csr.i, e->A_csr.x, x, y);
  return 0;
}
int spmv_At(Engine *e, const double *x, double *y) {
  e->n_spmv++;
  if (e->m == 0) return vec_set(e, y, 0.0, e->n);
  if (e->A_dense) {
    if (e->m_loc > 0) { if (int r = gemv_rows(e, e->n, e->m_loc, e->n, e->At, x + e->m_lo, y)) return r; }
    else if (int r = vec_set(e, y, 0.0, e->n)) return r;
    if (e->sh_world > 1) return shard_allreduce(y, y, (size_t)e->n, false, e->stream);   // sum of the per-rank partials
    return 0;
  }
  QB_LAUNCH(k_csr_spmv, cdiv(e->n, 8), 256, 0, e->stream, e->n, e->A_csc.p, e->A_csc.i, e->A_csc.x, x, y);
  return 0;
}
int spmv_Q(Engine *e, const double *x, double *y) {
  e->n_spmv++;
  if (e->Q_dense) QB_LAUNCH(k_gemv_cols, cdiv(e->n, 8), 256, 0, e->stream, e->n, e->n, e->n, e->Qd, x, y);
  else QB_LAUNCH(k_csr_spmv, cdiv(e->n, 8), 256, 0, e->stream, e->n, e->Q_csr.p, e->Q_csr.i, e->Q_csr.x, x, y);
  return 0;
}

// ------------------------------------------------------------------------------------------------
// residual step: compute_residuals (iteration.c:24-48) fused with the candidate active set
// (newton.c:122-149) and every reduction of check_termination (termination.c:44-240)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kRedThreads)
k_res_m(int m, int scaling, const double *__restrict__ Ax, const double *__restrict__ y,
        const double *__restrict__ sigma, const double *__restrict__ sigma_inv,
        const double *__restrict__ bmin, const double *__restrict__ bmax,
        const double *__restrict__ E, const double *__restrict__ Einv, const double *__restrict__ Ad,
        const int *__restrict__ active_old,
        double *Axys, double *z, double *pri_res, double *yh, double *delta_y, int *active_cand,
        double *partials) {
  __shared__ double scratch[32];
  double r_pri = 0, r_raw = 0, r_ax = 0, r_z = 0, r_edy = 0, oob = 0, adx_max = -1.0e300, adx_min = 1.0e300;
  double n_act = 0, n_ent = 0, n_lea = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
    const double ax = Ax[i], yi = y[i], lo = bmin[i], hi = bmax[i];
    double t = yi * sigma_inv[i];
    const double axys = ax + t;
    const double zi = fmax(lo, fmin(axys, hi));
    const double pr = ax - zi;
    t = pr * sigma[i];
    const double yhi = yi + t;
    Axys[i] = axys; z[i] = zi; pri_res[i] = pr; yh[i] = yhi;
    const int act = (axys <= lo) || (axys >= hi);
    const int old = active_old[i];
    active_cand[i] = act;
    n_act += act; n_ent += (act && !old); n_lea += (!act && old);
    const double ei = scaling ? E[i] : 1.0, einv = scaling ? Einv[i] : 1.0;
    r_pri = fmax(r_pri, fabs(einv * pr)); r_raw = fmax(r_raw, fabs(pr));
    r_ax = fmax(r_ax, fabs(einv * ax)); r_z = fmax(r_z, fabs(einv * zi));
    const double dy = yhi - yi;
    delta_y[i] = dy;
    r_edy = fmax(r_edy, fabs(ei * dy));
    const bool hi_fin = hi < ei * kInfty, lo_fin = lo > -ei * kInfty;
    oob += hi_fin ? hi * fmax(dy, 0.0) : 0.0;
    oob += lo_fin ? lo * fmin(dy, 0.0) : 0.0;
    const double adx = einv * Ad[i];
    if (hi_fin) adx_max = fmax(adx_max, adx);
    if (lo_fin) adx_min = fmin(adx_min, adx);
  }
  block_partial<RED_MAX>(r_pri, scratch, partials, S_PRI_RES);
  block_partial<RED_MAX>(r_raw, scratch, partials, S_PRI_RES_RAW);
  block_partial<RED_MAX>(r_ax, scratch, partials, S_NORM_AX);
  block_partial<RED_MAX>(r_z, scratch, partials, S_NORM_Z);
  block_partial<RED_MAX>(r_edy, scratch, partials, S_NORM_EDY);
  block_partial<RED_SUM>(oob, scratch, partials, S_OOB);
  block_partial<RED_MAX>(adx_max, scratch, partials, S_ADX_MAX);
  block_partial<RED_MIN>(adx_min, scratch, partials, S_ADX_MIN);
  block_partial<RED_SUM>(n_act, scratch, partials, S_NB_ACTIVE);
  block_partial<RED_SUM>(n_ent, scratch, partials, S_NB_ENTER);
  block_partial<RED_SUM>(n_lea, scratch, partials, S_NB_LEAVE);
}

__global__ void __launch_bounds__(kRedThreads)
k_res_n(int n, int scaling, int proximal, double neg_inv_gamma, const double *__restrict__ tau_ptr, double inv_gamma,
        const double *__restrict__ Qx, const double *__restrict__ q, const double *__restrict__ x0,
        const double *__restrict__ x, const double *__restrict__ x_prev, const double *__restrict__ Atyh,
        const double *__restrict__ Aty, const double *__restrict__ D, const double *__restrict__ Dinv,
        const double *__restrict__ Qd, const double *__restrict__ d,
        double *df, double *dphi, double *delta_x, double *partials) {
  __shared__ double scratch[32];
  double r_dua = 0, r_dua2 = 0, r_qx = 0, r_q = 0, r_atyh = 0, r_atdy = 0, r_ddx = 0, dxdx = 0, dxqdx = 0, qdx = 0;
  const double neg_tau_over_gamma = -(*tau_ptr) * inv_gamma;   // -work->tau/work->gamma (termination.c:228)
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
    const double qx = Qx[j], qj = q[j], xj = x[j], at = Atyh[j];
    double dfj = qx + qj;
    if (proximal) dfj = dfj + neg_inv_gamma * x0[j];
    const double dp = dfj + at;
    df[j] = dfj; dphi[j] = dp;
    const double dinv = scaling ? Dinv[j] : 1.0;
    if (proximal) {
      const double xx0 = xj - x0[j];
      const double t = dp + neg_inv_gamma * xx0;
      r_dua = fmax(r_dua, fabs(dinv * t));
    } else r_dua = fmax(r_dua, fabs(dinv * dp));
    r_dua2 = fmax(r_dua2, fabs(dinv * dp));
    r_qx = fmax(r_qx, fabs(dinv * qx)); r_q = fmax(r_q, fabs(dinv * qj)); r_atyh = fmax(r_atyh, fabs(dinv * at));
    const double atdy = at - Aty[j];
    r_atdy = fmax(r_atdy, fabs(dinv * atdy));
    const double dx = xj - x_prev[j];
    delta_x[j] = dx;
    const double ddx = scaling ? D[j] * dx : dx;
    r_ddx = fmax(r_ddx, fabs(ddx));
    dxdx += ddx * ddx;
    if (proximal) { const double t2 = Qd[j] + neg_tau_over_gamma * d[j]; dxqdx += dx * t2; }
    else dxqdx += Qd[j] * dx;
    qdx += qj * dx;
  }
  block_partial<RED_MAX>(r_dua, scratch, partials, S_DUA_RES);
  block_partial<RED_MAX>(r_dua2, scratch, partials, S_DUA2_RES);
  block_partial<RED_MAX>(r_qx, scratch, partials, S_NORM_QX);
  block_partial<RED_MAX>(r_q, scratch, partials, S_NORM_Q);
  block_partial<RED_MAX>(r_atyh, scratch, partials, S_NORM_ATYH);
  block_partial<RED_MAX>(r_atdy, scratch, partials, S_NORM_ATDY);
  block_partial<RED_MAX>(r_ddx, scratch, partials, S_NORM_DDX);
  block_partial<RED_SUM>(dxdx, scratch, partials, S_DXDX);
  block_partial<RED_SUM>(dxqdx, scratch, partials, S_DXQDX);
  block_partial<RED_SUM>(qdx, scratch, partials, S_QDX);
}

int step_residuals(Engine *e, bool proximal, double gamma, double /*tau unused: read on device*/) {
  const int gm = red_grid(e->m), gn = red_grid(e->n);
  if (e->m > 0) {
    QB_LAUNCH(k_res_m, gm, kRedThreads, 0, e->stream, e->m, e->scaling, e->Ax, e->y, e->sigma, e->sigma_inv, e->bmin,
              e->bmax, e->E, e->Einv, e->Ad, e->active_old, e->Axys, e->z, e->pri_res, e->yh, e->delta_y,
              e->active_cand, e->partials);
    finalize(e, {S_PRI_RES, S_PRI_RES_RAW, S_NORM_AX, S_NORM_Z, S_NORM_EDY, S_OOB, S_ADX_MAX, S_ADX_MIN, S_NB_ACTIVE,
                 S_NB_ENTER, S_NB_LEAVE}, gm);
  }
  if (int r = spmv_At(e, e->yh, e->Atyh)) return r;
  QB_LAUNCH(k_res_n, gn, kRedThreads, 0, e->stream, e->n, e->scaling, proximal ? 1 : 0, -1 / gamma,
            e->scal_dev + S_TAU, 1 / gamma, e->Qx, e->q, e->x0, e->x, e->x_prev, e->Atyh, e->Aty, e->D, e->Dinv,
            e->Qdv, e->d, e->df, e->dphi, e->delta_x, e->partials);
  finalize(e, {S_DUA_RES, S_DUA2_RES, S_NORM_QX, S_NORM_Q, S_NORM_ATYH, S_NORM_ATDY, S_NORM_DDX, S_DXDX, S_DXQDX, S_QDX}, gn);
  QB_CUDA_TRY(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// ordered index lists (single CTA, chunked ballot scan: ascending row order is part of the contract,
// it defines the column order of the update matrix -- SURVEY.md 8(a) row a5)
// ------------------------------------------------------------------------------------------------
constexpr int kListThreads = 1024;

// mode 0: commit the candidate active set (active <- cand) and list enter = cand & !old, leave = !cand & old
// mode 1: difference between the current (active, sigma) and the (activeH, sigmaH) H was assembled for:
//         pos: rows whose weight grew (scale sqrt(dw)), neg: rows whose weight shrank (scale sqrt(-dw));
//         from_scratch: the record is ignored (all active rows go to pos with scale sqrt_sigma).
//         The record is then updated.
__global__ void __launch_bounds__(kListThreads)
k_build_lists(int m, int mode, int from_scratch, const int *__restrict__ cand, int *active, const int *__restrict__ old,
              const double *__restrict__ sigma, const double *__restrict__ sqrt_sigma, int *activeH, double *sigmaH,
              int *list0, int *list1, double *w0, double *w1, double *scal) {
  __shared__ int warp_cnt0[32], warp_cnt1[32];
  __shared__ int base0, base1;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) { base0 = 0; base1 = 0; }
  __syncthreads();
  for (int start = 0; start < m; start += kListThreads) {
    const int i = start + tid;
    bool p0 = false, p1 = false;
    double s0 = 0.0, s1 = 0.0;
    if (i < m) {
      if (mode == 0) {
        const int c = cand[i], o = old[i];
        active[i] = c;
        p0 = c && !o; p1 = !c && o;
      } else {
        const int a = active[i];
        const double wn = a ? sigma[i] : 0.0;
        const double wh = (from_scratch || !activeH[i]) ? 0.0 : sigmaH[i];
        const double dw = wn - wh;
        if (dw > 0.0) { p0 = true; s0 = (wh == 0.0) ? sqrt_sigma[i] : sqrt(dw); }
        else if (dw < 0.0) { p1 = true; s1 = sqrt(-dw); }
        activeH[i] = a; sigmaH[i] = sigma[i];
      }
    }
    const unsigned b0 = __ballot_sync(0xffffffffu, p0), b1 = __ballot_sync(0xffffffffu, p1);
    if (lane == 0) { warp_cnt0[warp] = __popc(b0); warp_cnt1[warp] = __popc(b1); }
    __syncthreads();
    int off0 = base0, off1 = base1;
    for (int w = 0; w < warp; w++) { off0 += warp_cnt0[w]; off1 += warp_cnt1[w]; }
    const unsigned lt = (1u << lane) - 1u;
    if (p0) { const int pos = off0 + __popc(b0 & lt); list0[pos] = i; if (mode == 1) w0[pos] = s0; }
    if (p1) { const int pos = off1 + __popc(b1 & lt); list1[pos] = i; if (mode == 1) w1[pos] = s1; }
    __syncthreads();
    if (tid == 0) {
      int t0 = 0, t1 = 0;
      for (int w = 0; w < 32; w++) { t0 += warp_cnt0[w]; t1 += warp_cnt1[w]; }
      base0 += t0; base1 += t1;
    }
    __syncthreads();
  }
  if (tid == 0) { scal[S_TMP0] = (double)base0; scal[S_TMP1] = (double)base1; }
}

int step_compact_lists(Engine *e) {
  if (e->m == 0) return 0;
  QB_LAUNCH(k_build_lists, 1, kListThreads, 0, e->stream, e->m, 0, 0, e->active_cand, e->active, e->active_old,
            e->sigma, e->sqrt_sigma, e->activeH, e->sigmaH, e->enter, e->leave, e->w_pos, e->w_neg, e->scal_dev);
  return 0;
}
int step_commit_active(Engine *e) { return ivec_copy(e, e->active, e->active_old, e->m); }

// ------------------------------------------------------------------------------------------------
// gather of scaled rows of A into the dense panel W (n x kpad, column c = scale * A(list[c], :)')
// -- the columns cholmod_submatrix extracts from At_sqrt_sigma (solver_interface.c:417,435,493)
// ------------------------------------------------------------------------------------------------
__global__ void k_gather_dense(int n, int npad, const double *__restrict__ At, const int *__restrict__ list,
                               const double *__restrict__ scale, int scale_by_row, int cnt, double *W, int ldw, int m_lo, int m_loc) {
  const int c = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npad) return;
  double v = 0.0;
  if (c < cnt && i < n) {
    const int row = list[c], loc = row - m_lo;   // rows owned by another rank contribute a zero column here
    if (loc >= 0 && loc < m_loc) v = At[(size_t)i + (size_t)n * loc] * (scale_by_row ? scale[row] : scale[c]);
  }
  W[(size_t)i + (size_t)ldw * c] = v;
}
__global__ void k_gather_csr(int npad, const int *__restrict__ p, const int *__restrict__ ci, const double *__restrict__ x,
                             const int *__restrict__ list, const double *__restrict__ scale, int scale_by_row, int cnt,
                             double *W, int ldw) {
  const int c = blockIdx.x;
  double *col = W + (size_t)ldw * c;
  for (int i = threadIdx.x; i < npad; i += blockDim.x) col[i] = 0.0;
  __syncthreads();
  if (c < cnt) {
    const int row = list[c];
    const double s = scale_by_row ? scale[row] : scale[c];
    for (int k = p[row] + threadIdx.x; k < p[row + 1]; k += blockDim.x) col[ci[k]] = x[k] * s;
  }
}
static int gather_rows(Engine *e, const int *list, const double *scale, bool scale_by_row, int cnt, int kpad, int col0 = 0) {
  if (kpad <= 0) return 0;
  double *W = e->W + (size_t)e->ld * col0;
  if (e->A_dense) {
    dim3 grid(cdiv(e->npad, 256), kpad);
    QB_LAUNCH(k_gather_dense, grid, 256, 0, e->stream, e->n, e->npad, e->At, list, scale, scale_by_row ? 1 : 0, cnt, W, e->ld, e->m_lo, e->m_loc);
  } else {
    QB_LAUNCH(k_gather_csr, kpad, 256, 0, e->stream, e->npad, e->A_csr.p, e->A_csr.i, e->A_csr.x, list, scale,
              scale_by_row ? 1 : 0, cnt, W, e->ld);
  }
  return 0;
}

int gather_rows_public(Engine *e, const int *list, const double *scale, bool scale_by_row, int cnt, int kpad) {
  return gather_rows(e, list, scale, scale_by_row, cnt, kpad);
}

// dst(lower) <- Q ; everything else in the lower triangle <- 0
__global__ void k_init_lower_from_dense(int n, int npad, const double *__restrict__ Q, double *dst, int ld) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
  if (i >= npad || i < j) return;
  dst[(size_t)i + (size_t)j * ld] = (i < n && j < n) ? Q[(size_t)i + (size_t)j * n] : 0.0;
}
__global__ void k_scatter_csr_lower(int n, const int *__restrict__ p, const int *__restrict__ ci, const double *__restrict__ x,
                                    double *dst, int ld) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n) return;
  for (int k = p[row] + lane; k < p[row + 1]; k += 32) {
    const int col = ci[k];
    if (col <= row) dst[(size_t)row + (size_t)col * ld] = x[k];
  }
}
__global__ void k_add_diag_pad(int n, int npad, double *L, int ld, double beta) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npad) return;
  double *p = L + (size_t)i * (ld + 1);
  *p = (i < n) ? (*p + beta) : 1.0;
}
// partial: dst is this rank's term of a sum over ranks (the H record of a row-sharded problem) -- Q enters on rank 0 only
static int init_lower_from_Q(Engine *e, double *dst, bool partial = false) {
  if (partial && e->sh_world > 1 && e->sh_rank != 0) {
    QB_CUDA_TRY(cudaMemsetAsync(dst, 0, sizeof(double) * (size_t)e->ld * e->npad, e->stream));
    return 0;
  }
  if (e->Q_dense) {
    dim3 grid(cdiv(e->npad, 256), e->npad);
    QB_LAUNCH(k_init_lower_from_dense, grid, 256, 0, e->stream, e->n, e->npad, e->Qd, dst, e->ld);
  } else {
    QB_CUDA_TRY(cudaMemsetAsync(dst, 0, sizeof(double) * (size_t)e->ld * e->npad, e->stream));
    QB_LAUNCH(k_scatter_csr_lower, cdiv(e->n, 8), 256, 0, e->stream, e->n, e->Q_csr.p, e->Q_csr.i, e->Q_csr.x, dst, e->ld);
  }
  return 0;
}

// accumulate  dst(lower) += sign * sum_c W_c W_c'  over a list, in chunks of e->wcols columns
static int syrk_list(Engine *e, double *dst, const int *list, const double *scale, bool scale_by_row, int cnt, double sign) {
  for (int off = 0; off < cnt; off += e->wcols) {
    const int k = (cnt - off < e->wcols) ? cnt - off : e->wcols;
    const int kpad = round_up(k, 16);
    if (int r = gather_rows(e, list + off, scale_by_row ? scale : scale + off, scale_by_row, k, kpad)) return r;
    if (int r = dgemm_nt(e->stream, e->npad, e->npad, kpad, e->W, e->ld, e->W, e->ld, dst, e->ld, sign, 1.0, true)) return r;
    e->dense_flops += (double)e->n * e->n * k;
  }
  return 0;
}

// ldlcholQAtsigmaA / ldlchol(Q)  (solver_interface.c:319-405): assemble H (incrementally when cheaper),
// L <- chol(H + beta I)
// sparse problems: H is assembled straight into the supernodal panels (always from scratch: the assembly is
// O(sum_active nnz_row^2), negligible next to the factorization) and factorized level by level (sparse.cu)
static int sparse_refactor(Engine *e, bool with_constraints, double beta, int nb_active) {
  QB_CUDA_TRY(cudaEventRecord(e->evs0, e->stream));
  const bool wc = with_constraints && e->m > 0;
  if (int r = sparse_chol_assemble(e->sp, e->stream, e->spL, true, e->Q_csr.p, e->Q_csr.i, e->Q_csr.x, e->A_csc.p, e->A_csc.i,
                                   e->A_csc.x, e->A_csr.p, e->A_csr.i, e->A_csr.x, wc ? e->active : nullptr, e->sigma, beta)) return r;
  if (int r = sparse_chol_factor(e->sp, e->stream, e->spL, e->info_dev)) return r;
  QB_CUDA_TRY(cudaEventRecord(e->evs1, e->stream));
  const SparseCholInfo *I = sparse_chol_info(e->sp);
  e->n_refactor++; e->refactor_active_sum += wc ? nb_active : 0;
  e->dense_flops += I->flops;
  e->alg_bytes += 12.0 * (double)I->nnzS + 2.0 * 8.0 * (double)I->nnzL;   // SURVEY 8(d): B_H + B_L (read H, write + read L)
  return 0;
}

int step_newton_refactor(Engine *e, bool with_constraints, bool from_scratch, double beta, int nb_active) {
  if (e->sp) return sparse_refactor(e, with_constraints, beta, nb_active);
  QB_CUDA_TRY(cudaEventRecord(e->evs0, e->stream));
  if (!with_constraints || e->m == 0) {
    if (int r = init_lower_from_Q(e, e->L)) return r;
    QB_LAUNCH(k_add_diag_pad, cdiv(e->npad, 256), 256, 0, e->stream, e->n, e->npad, e->L, e->ld, beta);
    nb_active = 0;
  } else {
    if (!e->H_valid) from_scratch = true;
    for (int attempt = 0; attempt < 2; attempt++) {
      QB_LAUNCH(k_build_lists, 1, kListThreads, 0, e->stream, e->m, 1, from_scratch ? 1 : 0, e->active_cand, e->active,
                e->active_old, e->sigma, e->sqrt_sigma, e->activeH, e->sigmaH, e->list_pos, e->list_neg, e->w_pos,
                e->w_neg, e->scal_dev);
      if (int r = sync_scalars(e)) return r;
      const int npos = (int)e->scal_host[S_TMP0], nneg = (int)e->scal_host[S_TMP1];
      if (!from_scratch && npos + nneg > nb_active) {
        // cheaper to rebuild; the record now equals the current state, so force the full list
        from_scratch = true;
        continue;
      }
      if (from_scratch) { if (int r = init_lower_from_Q(e, e->H, true)) return r; }
      if (int r = syrk_list(e, e->H, e->list_pos, e->w_pos, false, npos, 1.0)) return r;
      if (int r = syrk_list(e, e->H, e->list_neg, e->w_neg, false, nneg, -1.0)) return r;
      break;
    }
    e->H_valid = true;
    if (e->sh_world > 1) {   // L <- sum over ranks of the H partials, then + beta I (and the identity pad)
      if (int r = shard_allreduce(e->H, e->L, (size_t)e->ld * e->npad, false, e->stream)) return r;
      QB_LAUNCH(k_add_diag_pad, cdiv(e->npad, 256), 256, 0, e->stream, e->n, e->npad, e->L, e->ld, beta);
    } else if (int r = copy_lower_add_diag(e->stream, e->n, e->npad, e->H, e->L, e->ld, beta)) return r;
  }
  if (int r = potrf_lower(e->stream, e->npad, e->L, e->ld, e->invdiag, e->info_dev)) return r;
  QB_CUDA_TRY(cudaEventRecord(e->evs1, e->stream));
  e->n_refactor++; e->refactor_active_sum += nb_active;
  e->dense_flops += (double)e->n * e->n * e->n / 3.0;
  e->alg_bytes += 8.0 * (double)nb_active * e->n + 2.0 * 8.0 * (double)e->n * (e->n + 1) / 2;
  return 0;
}

// generator-form passes (updown_gen.cu) serve factors of at least two 128-column blocks; below that the per-panel kernels of
// dense.cu cost a handful of launches.  <= 32 columns per pass, entering and leaving rows share a pass; the inverted diagonal
// blocks are refreshed after every pass (the next pass's triangular solve needs them, and so do the Newton solves)
bool use_updown_gen(const Engine *e) {
  return !e->sp && e->npad >= 256 && e->updown_gen_ok;
}
static int updown_gen_lists(Engine *e, const int *pos, const double *pos_scale, bool pos_by_row, int npos,
                            const int *neg, const double *neg_scale, bool neg_by_row, int nneg) {
  const int KMAX = chol_updown_gen_max_rank();
  int ip = 0, in = 0;
  while (ip < npos || in < nneg) {
    const int kp = (npos - ip < KMAX) ? npos - ip : KMAX;
    const int kn = (nneg - in < KMAX - kp) ? nneg - in : KMAX - kp;
    if (int r = gather_rows(e, pos + ip, pos_by_row ? pos_scale : pos_scale + ip, pos_by_row, kp, kp, 0)) return r;
    if (int r = gather_rows(e, neg + in, neg_by_row ? neg_scale : neg_scale + in, neg_by_row, kn, kn, kp)) return r;
    // row-sharded problem: every rank gathered the rows it owns (zero columns for the others); the sum over ranks is the full
    // n x k block, and every rank then runs the same pass on its replica of L
    if (e->sh_world > 1) { if (int r = shard_allreduce(e->W, e->W, (size_t)e->ld * (kp + kn), false, e->stream)) return r; }
    const int rc = chol_updown_gen(e->stream, e->npad, e->L, e->ld, e->invdiag, e->W, e->ld, kp + kn, kp, e->info_dev);
    // 1: unavailable -- it fails on the first pass or never, so nothing has been applied and the caller can fall back to the
    // per-panel kernels; < 0: CUDA error
    if (rc) return (rc == 1 && ip == 0 && in == 0) ? 1 : (rc < 0 ? rc : -999);
    if (int r = trtri_diag_blocks(e->stream, e->npad, e->L, e->ld, e->invdiag)) return r;
    e->n_updown++; e->updown_rank_sum += kp + kn;
    e->dense_flops += 2.0 * (kp + kn) * (double)e->n * e->n;
    e->alg_bytes += 3.0 * 8.0 * (double)e->n * (e->n + 1) / 2;
    ip += kp; in += kn;
  }
  return 0;
}

// ldlupdate_entering_constraints / ldldowndate_leaving_constraints (solver_interface.c:407-441)
int step_newton_updown(Engine *e, int nb_enter, int nb_leave) {
  QB_CUDA_TRY(cudaEventRecord(e->evs0, e->stream));
  if (use_updown_gen(e)) {
    const int rc = updown_gen_lists(e, e->enter, e->sqrt_sigma, true, nb_enter, e->leave, e->sqrt_sigma, true, nb_leave);
    if (rc < 0) return rc;
    if (rc == 0) { QB_CUDA_TRY(cudaEventRecord(e->evs1, e->stream)); return 0; }
    e->updown_gen_ok = false;   // unavailable on this device / partition: per-panel kernels from now on
  }
  for (int pass = 0; pass < 2; pass++) {
    const int *list = pass == 0 ? e->enter : e->leave;
    const int cnt = pass == 0 ? nb_enter : nb_leave;
    for (int off = 0; off < cnt; off += 8) {
      const int k = cnt - off < 8 ? cnt - off : 8;
      if (e->sp) {
        if (int r = sparse_chol_updown(e->sp, e->stream, e->spL, e->A_csr.p, e->A_csr.i, e->A_csr.x, list + off, e->sqrt_sigma,
                                       true, k, pass == 0 ? +1 : -1, e->info_dev)) return r;
        e->n_updown++; e->updown_rank_sum += k;
        e->alg_bytes += 2.0 * 12.0 * (double)sparse_chol_info(e->sp)->nnzL;
        continue;
      }
      if (int r = gather_rows(e, list + off, e->sqrt_sigma, true, k, 8)) return r;
      if (e->sh_world > 1) { if (int r = shard_allreduce(e->W, e->W, (size_t)e->ld * 8, false, e->stream)) return r; }   // as in updown_gen_lists
      if (int r = chol_updown(e->stream, e->npad, e->L, e->ld, e->W, e->ld, k, pass == 0 ? +1 : -1, e->ud_coef, e->info_dev)) return r;
      e->n_updown++; e->updown_rank_sum += k;
      e->dense_flops += 2.0 * k * (double)e->n * e->n;
      e->alg_bytes += 2.0 * 8.0 * (double)e->n * (e->n + 1) / 2;
    }
  }
  if (!e->sp) { if (int r = trtri_diag_blocks(e->stream, e->npad, e->L, e->ld, e->invdiag)) return r; }
  QB_CUDA_TRY(cudaEventRecord(e->evs1, e->stream));
  return 0;
}

// ldlupdate_sigma_changed (solver_interface.c:443-503): rank-k update with sqrt(sigma_new - sigma_old) * a_j
int sigma_changed_update(Engine *e, int nb_changed) {
  QB_CUDA_TRY(cudaEventRecord(e->evs0, e->stream));
  if (use_updown_gen(e)) {
    const int rc = updown_gen_lists(e, e->changed, e->w_pos, false, nb_changed, nullptr, nullptr, false, 0);
    if (rc < 0) return rc;
    if (rc == 0) { QB_CUDA_TRY(cudaEventRecord(e->evs1, e->stream)); return 0; }
    e->updown_gen_ok = false;
  }
  for (int off = 0; off < nb_changed; off += 8) {
    const int k = nb_changed - off < 8 ? nb_changed - off : 8;
    if (e->sp) {
      if (int r = sparse_chol_updown(e->sp, e->stream, e->spL, e->A_csr.p, e->A_csr.i, e->A_csr.x, e->changed + off, e->w_pos + off,
                                     false, k, +1, e->info_dev)) return r;
      e->n_updown++; e->updown_rank_sum += k;
      continue;
    }
    if (int r = gather_rows(e, e->changed + off, e->w_pos + off, false, k, 8)) return r;
    if (e->sh_world > 1) { if (int r = shard_allreduce(e->W, e->W, (size_t)e->ld * 8, false, e->stream)) return r; }
    if (int r = chol_updown(e->stream, e->npad, e->L, e->ld, e->W, e->ld, k, +1, e->ud_coef, e->info_dev)) return r;
    e->n_updown++; e->updown_rank_sum += k;
    e->dense_flops += 2.0 * k * (double)e->n * e->n;
  }
  if (!e->sp) { if (int r = trtri_diag_blocks(e->stream, e->npad, e->L, e->ld, e->invdiag)) return r; }
  QB_CUDA_TRY(cudaEventRecord(e->evs1, e->stream));
  return 0;
}

__global__ void k_neg_to_pad(int n, int npad, const double *__restrict__ src, double *dst) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < npad) dst[i] = (i < n) ? src[i] * -1 : 0.0;
}
// ldlsolveLD_neg_dphi (solver_interface.c:505-519)
int step_newton_solve(Engine *e) {
  if (e->sp) {
    e->alg_bytes += 2.0 * 12.0 * (double)sparse_chol_info(e->sp)->nnzL;
    e->dense_flops += 4.0 * (double)sparse_chol_info(e->sp)->nnzL;
    return sparse_chol_solve(e->sp, e->stream, e->spL, e->dphi, e->d, true);
  }
  QB_LAUNCH(k_neg_to_pad, cdiv(e->npad, 256), 256, 0, e->stream, e->n, e->npad, e->dphi, e->vpad);
  if (int r = chol_solve(e->stream, e->npad, e->L, e->ld, e->invdiag, e->vpad)) return r;
  e->dense_flops += 2.0 * (double)e->n * e->n;
  e->alg_bytes += 2.0 * 8.0 * (double)e->n * (e->n + 1) / 2;
  return vec_copy(e, e->vpad, e->d, e->n);
}

// ================================================================================================
// exact line search (linesearch.c:14-120): breakpoints -> stable LSD radix sort -> scan -> select
// ================================================================================================
__global__ void __launch_bounds__(kRedThreads)
k_ls_build(int m, const double *__restrict__ Ad, const double *__restrict__ Ax, const double *__restrict__ y,
           const double *__restrict__ sigma, const double *__restrict__ sqrt_sigma, const double *__restrict__ bmin,
           const double *__restrict__ bmax, unsigned long long *key, unsigned int *val, double *da, double *db,
           double *partials) {
  __shared__ double scratch[32];
  double a_part = 0, b_part = 0, n_l = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
    const double ss = sqrt_sigma[i], sg = sigma[i], ax = Ax[i], yi = y[i];
    const double t = ss * Ad[i];
    double dl[2], al[2];
    dl[1] = t; dl[0] = t * -1;
    double u = ax - bmin[i]; u = sg * u; u = yi + u; al[0] = u / ss;
    u = bmax[i] - ax; u = sg * u; u = u - yi; al[1] = u / ss;
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int idx = i + h * m;
      const double s = al[h] / dl[h];
      const bool inL = s > 0, inP = dl[h] > 0;
      key[idx] = inL ? (unsigned long long)__double_as_longlong(s) : ~0ull;
      val[idx] = (unsigned int)idx;
      const double d2 = dl[h] * dl[h], dalp = dl[h] * al[h];
      da[idx] = inP ? d2 : -d2;
      db[idx] = inP ? -dalp : dalp;
      if ((int)inL + (int)inP == 1) { a_part += d2; b_part += dalp; }
      n_l += inL;
    }
  }
  block_partial<RED_SUM>(a_part, scratch, partials, S_LS_A);
  block_partial<RED_SUM>(b_part, scratch, partials, S_LS_B);
  block_partial<RED_SUM>(n_l, scratch, partials, S_NL);
}

// ---- stable LSD radix sort, 8 bits per pass, tiles of 2048 keys ------------------------------------
namespace rsort {
constexpr int NT = 512, ROUNDS = 4, TILE = NT * ROUNDS, NW = NT / 32;

__global__ void __launch_bounds__(NT) k_hist(const unsigned long long *__restrict__ keys, int N, int shift,
                                             unsigned int *hist, int ntiles) {
  __shared__ unsigned int h[256];
  if (threadIdx.x < 256) h[threadIdx.x] = 0;
  __syncthreads();
  const int base = blockIdx.x * TILE;
#pragma unroll
  for (int r = 0; r < ROUNDS; r++) {
    const int e = base + r * NT + threadIdx.x;
    if (e < N) atomicAdd(&h[(unsigned)(keys[e] >> shift) & 255u], 1u);
  }
  __syncthreads();
  if (threadIdx.x < 256) hist[threadIdx.x * ntiles + blockIdx.x] = h[threadIdx.x];
}
// exclusive scan of hist[0 .. total) in place (digit-major, tile-minor), one CTA: every warp scans one contiguous
// segment with a running carry (coalesced, no CTA barriers inside the loop), the 32 segment totals are combined once and
// added back in a second sweep over the warp's own writes.  (The round-1 version walked the array in 1024-entry chunks
// with three CTA barriers per chunk: 82 us at 2m = 717k against ~10 us for this form.)
__global__ void __launch_bounds__(1024) k_scan(unsigned int *hist, int total) {
  __shared__ unsigned int wtot[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int seg = ((total + 31) / 32 + 31) & ~31;          // per-warp segment, a multiple of 32
  const int begin = warp * seg, end = min(begin + seg, total);
  unsigned int carry = 0;
  for (int i0 = begin; i0 < begin + seg; i0 += 32) {
    const int i = i0 + lane;
    const unsigned int v = (i < end) ? hist[i] : 0u;
    unsigned int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
    if (i < end) hist[i] = carry + inc - v;
    carry += __shfl_sync(0xffffffffu, inc, 31);
  }
  if (lane == 0) wtot[warp] = carry;
  __syncthreads();
  unsigned int off = 0;
  for (int w = 0; w < warp; w++) off += wtot[w];
  if (off)
    for (int i = begin + lane; i < end; i += 32) hist[i] += off;
}
__global__ void __launch_bounds__(NT) k_scatter(const unsigned long long *__restrict__ kin, const unsigned int *__restrict__ vin,
                                                unsigned long long *kout, unsigned int *vout, int N, int shift,
                                                const unsigned int *__restrict__ hist, int ntiles) {
  __shared__ unsigned int warp_cnt[NW][256];
  __shared__ unsigned int running[256];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid < 256) running[tid] = hist[tid * ntiles + blockIdx.x];
  const int base = blockIdx.x * TILE;
  for (int r = 0; r < ROUNDS; r++) {
    for (int i = tid; i < NW * 256; i += NT) (&warp_cnt[0][0])[i] = 0;
    __syncthreads();
    const int e = base + r * NT + tid;
    const bool valid = e < N;
    unsigned long long k = 0; unsigned int v = 0; unsigned int dg = 0x10000u + lane;
    if (valid) { k = kin[e]; v = vin[e]; dg = (unsigned)(k >> shift) & 255u; }
    const unsigned peers = __match_any_sync(0xffffffffu, dg);
    const unsigned lt = (1u << lane) - 1u;
    const int rank = __popc(peers & lt);
    if (valid && rank == 0) warp_cnt[warp][dg] = __popc(peers);
    __syncthreads();
    if (valid) {
      unsigned int off = running[dg];
      for (int w = 0; w < warp; w++) off += warp_cnt[w][dg];
      const unsigned int pos = off + rank;
      kout[pos] = k; vout[pos] = v;
    }
    __syncthreads();
    if (tid < 256) {
      unsigned int t = 0;
#pragma unroll
      for (int w = 0; w < NW; w++) t += warp_cnt[w][tid];
      running[tid] += t;
    }
    __syncthreads();
  }
}
}  // namespace rsort

// sorts (ls_key[0], ls_val[0]) of length N; result ends in buffer index 0 (8 passes, even count)
static int radix_sort_pairs(Engine *e, int N) {
  const int ntiles = cdiv(N, rsort::TILE);
  int cur = 0;
  for (int pass = 0; pass < 8; pass++) {
    const int shift = pass * 8;
    QB_LAUNCH(rsort::k_hist, ntiles, rsort::NT, 0, e->stream, e->ls_key[cur], N, shift, e->rs_hist, ntiles);
    QB_LAUNCH(rsort::k_scan, 1, 1024, 0, e->stream, e->rs_hist, 256 * ntiles);
    QB_LAUNCH(rsort::k_scatter, ntiles, rsort::NT, 0, e->stream, e->ls_key[cur], e->ls_val[cur], e->ls_key[cur ^ 1],
              e->ls_val[cur ^ 1], N, shift, e->rs_hist, ntiles);
    cur ^= 1;
  }
  return 0;
}

// walk of linesearch.c:89-119 as a chunked exclusive scan with early exit (one CTA)
__global__ void __launch_bounds__(1024)
k_ls_select(const unsigned long long *__restrict__ key, const unsigned int *__restrict__ val,
            const double *__restrict__ da, const double *__restrict__ db, double *scal) {
  __shared__ double wa[32], wb[32];
  __shared__ double carry_a, carry_b;
  __shared__ int found;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nL = (int)scal[S_NL];
  if (tid == 0) { carry_a = scal[S_ETA] + scal[S_LS_A]; carry_b = scal[S_BETA] - scal[S_LS_B]; found = 0x7fffffff; }
  __syncthreads();
  for (int start = 0; start < nL; start += 1024) {
    const int i = start + tid;
    double ta = 0.0, tb = 0.0, s = 0.0;
    if (i < nL) { const unsigned int idx = val[i]; ta = da[idx]; tb = db[idx]; s = __longlong_as_double((long long)key[i]); }
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
      if (i == found) scal[S_TAU] = -b_i / a_i;
      return;
    }
    if (tid == 1023) { carry_a += oa + ia; carry_b += ob + ib; }
    __syncthreads();
  }
  if (tid == 0) scal[S_TAU] = -carry_b / carry_a;
}

// ---- 2m <= LS1_MAX: stable LSD radix sort + breakpoint walk in ONE single-CTA launch -----------------------------------
// The multi-launch sort above costs 24 launches per line search (hist / scan / scatter x 8 passes) whatever the size; for
// 2m = 4000 (BASELINE config 1) they are 1272 of the 2567 launches of a solve and ~10 ms of its 48 ms.  Here the (key, index)
// pairs live in shared memory (two ping-pong buffers, 24 bytes per pair), every pass is histogram -> 256-bin exclusive scan ->
// ordered scatter in rounds of 1024 elements (per-warp digit counts from __match_any_sync, an exclusive scan of each digit's
// counts over the 32 warps, then one read per element), passes whose digit is the same for all keys are skipped, and the walk
// of linesearch.c:89-119 (k_ls_select's chunked scan) runs on the sorted pairs without leaving the CTA.  Same stable order
// (ties by ascending original index) and the same arithmetic in the walk as the multi-launch path: results are bit-identical.
namespace ls1 {
constexpr int NT = 1024, NW = NT / 32, LS1_MAX = 8192;
constexpr size_t smem_bytes(int N) { return (size_t)N * 24 + 2 * 256 * NW + 4 * (256 + 256) + 64; }

__global__ void __launch_bounds__(NT, 1)
k_sort_select(unsigned long long *key_g, unsigned int *val_g, int N, const double *__restrict__ da, const double *__restrict__ db, double *scal) {
  extern __shared__ __align__(16) unsigned char sm_raw[];
  unsigned long long *k0 = reinterpret_cast<unsigned long long *>(sm_raw), *k1 = k0 + N;
  unsigned int *v0 = reinterpret_cast<unsigned int *>(k1 + N), *v1 = v0 + N;
  unsigned int *hist = v1 + N, *running = hist + 256;
  unsigned short *wcnt = reinterpret_cast<unsigned short *>(running + 256);   // [NW][256]: per-warp digit counts, then their exclusive scan over the warps (< 1024)
  __shared__ double wa[32], wb[32];
  __shared__ double carry_a, carry_b;
  __shared__ int found;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < N; i += NT) { k0[i] = key_g[i]; v0[i] = val_g[i]; }
  __syncthreads();
  unsigned long long *kin = k0, *kout = k1;
  unsigned int *vin = v0, *vout = v1;
  for (int pass = 0; pass < 8; pass++) {
    const int shift = pass * 8;
    if (tid < 256) hist[tid] = 0;
    __syncthreads();
    for (int i = tid; i < N; i += NT) atomicAdd(&hist[(unsigned)(kin[i] >> shift) & 255u], 1u);
    __syncthreads();
    if (hist[(unsigned)(kin[0] >> shift) & 255u] == (unsigned)N) { __syncthreads(); continue; }   // one digit for all keys
    if (warp == 0) {   // exclusive scan of the 256 bins
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
    for (int start = 0; start < N; start += NT) {
      for (int i = tid; i < NW * 256 / 2; i += NT) reinterpret_cast<unsigned int *>(wcnt)[i] = 0;
      __syncthreads();
      const int e = start + tid;
      const bool valid = e < N;
      unsigned long long k = 0; unsigned int v = 0; unsigned int dg = 0x10000u + lane;
      if (valid) { k = kin[e]; v = vin[e]; dg = (unsigned)(k >> shift) & 255u; }
      const unsigned peers = __match_any_sync(0xffffffffu, dg);
      const int rank = __popc(peers & ((1u << lane) - 1u));
      if (valid && rank == 0) wcnt[warp * 256 + dg] = (unsigned short)__popc(peers);
      __syncthreads();
      if (tid < 256) {   // digit tid: exclusive scan of its counts over the warps (in place), then advance the running offset
        unsigned int acc = 0;
#pragma unroll 8
        for (int w = 0; w < NW; w++) { const unsigned int c = wcnt[w * 256 + tid]; wcnt[w * 256 + tid] = (unsigned short)acc; acc += c; }
        hist[tid] = acc;   // this round's total of the digit (hist is free after the scan)
      }
      __syncthreads();
      if (valid) {
        const unsigned int pos = running[dg] + wcnt[warp * 256 + dg] + rank;
        kout[pos] = k; vout[pos] = v;
      }
      __syncthreads();
      if (tid < 256) running[tid] += hist[tid];
      __syncthreads();
    }
    unsigned long long *tk = kin; kin = kout; kout = tk;
    unsigned int *tv = vin; vin = vout; vout = tv;
  }
  __syncthreads();
  for (int i = tid; i < N; i += NT) { key_g[i] = kin[i]; val_g[i] = vin[i]; }   // the operator ABI returns the sorted pairs
  // ---- the walk (k_ls_select on the shared-memory pairs) ----
  const int nL = (int)scal[S_NL];
  if (tid == 0) { carry_a = scal[S_ETA] + scal[S_LS_A]; carry_b = scal[S_BETA] - scal[S_LS_B]; found = 0x7fffffff; }
  __syncthreads();
  for (int start = 0; start < nL; start += NT) {
    const int i = start + tid;
    double ta = 0.0, tb = 0.0, sv = 0.0;
    if (i < nL) { const unsigned int idx = vin[i]; ta = da[idx]; tb = db[idx]; sv = __longlong_as_double((long long)kin[i]); }
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
    if (i < nL && (a_i * sv + b_i > 0)) atomicMin(&found, i);
    __syncthreads();
    if (found != 0x7fffffff) {
      if (i == found) scal[S_TAU] = -b_i / a_i;
      return;
    }
    if (tid == NT - 1) { carry_a += oa + ia; carry_b += ob + ib; }
    __syncthreads();
  }
  if (tid == 0) scal[S_TAU] = -carry_b / carry_a;
}
}  // namespace ls1

int linesearch_device(Engine *e, int m, const double *Ad, const double *Ax, const double *y, const double *sigma,
                      const double *sqrt_sigma, const double *bmin, const double *bmax) {
  if (m == 0) {
    QB_CUDA_TRY(cudaMemsetAsync(e->scal_dev + S_LS_A, 0, sizeof(double) * 2, e->stream));
    QB_CUDA_TRY(cudaMemsetAsync(e->scal_dev + S_NL, 0, sizeof(double), e->stream));
  } else {
    const int g = red_grid(m);
    QB_LAUNCH(k_ls_build, g, kRedThreads, 0, e->stream, m, Ad, Ax, y, sigma, sqrt_sigma, bmin, bmax, e->ls_key[0],
              e->ls_val[0], e->ls_da, e->ls_db, e->partials);
    finalize(e, {S_LS_A, S_LS_B, S_NL}, g);
    static const bool multi_launch = getenv("QPALM_B200_LS_MULTI") != nullptr;   // A/B and parity runs of the multi-launch path
    if (2 * m <= ls1::LS1_MAX && !multi_launch) {
      static bool attr_set = false;
      if (!attr_set) {
        QB_CUDA_TRY(cudaFuncSetAttribute(ls1::k_sort_select, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ls1::smem_bytes(ls1::LS1_MAX)));
        attr_set = true;
      }
      QB_LAUNCH(ls1::k_sort_select, 1, ls1::NT, ls1::smem_bytes(2 * m), e->stream, e->ls_key[0], e->ls_val[0], 2 * m, e->ls_da, e->ls_db, e->scal_dev);
      QB_CUDA_TRY(cudaGetLastError());
      return 0;
    }
    if (int r = radix_sort_pairs(e, 2 * m)) return r;
  }
  QB_LAUNCH(k_ls_select, 1, 1024, 0, e->stream, e->ls_key[0], e->ls_val[0], e->ls_da, e->ls_db, e->scal_dev);
  QB_CUDA_TRY(cudaGetLastError());
  return 0;
}

__global__ void __launch_bounds__(kRedThreads)
k_ls_dots(int n, int proximal, double inv_gamma, const double *__restrict__ d, double *Qd, const double *__restrict__ df,
          double *partials) {
  __shared__ double scratch[32];
  double eta = 0, beta = 0;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
    double qd = Qd[j];
    const double dj = d[j];
    if (proximal) { qd = qd + inv_gamma * dj; Qd[j] = qd; }
    eta += dj * qd; beta += dj * df[j];
  }
  block_partial<RED_SUM>(eta, scratch, partials, S_ETA);
  block_partial<RED_SUM>(beta, scratch, partials, S_BETA);
}
int step_linesearch(Engine *e, bool proximal, double gamma) {
  if (int r = spmv_Q(e, e->d, e->Qdv)) return r;
  if (int r = spmv_A(e, e->d, e->Ad)) return r;
  const int g = red_grid(e->n);
  QB_LAUNCH(k_ls_dots, g, kRedThreads, 0, e->stream, e->n, proximal ? 1 : 0, 1 / gamma, e->d, e->Qdv, e->df, e->partials);
  finalize(e, {S_ETA, S_BETA}, g);
  return linesearch_device(e, e->m, e->Ad, e->Ax, e->y, e->sigma, e->sqrt_sigma, e->bmin, e->bmax);
}

// update_primal_iterate tail (iteration.c:219-228), tau read from the device scalar block
__global__ void k_update_iterate(int n, int m, const double *__restrict__ scal, double *x, double *x_prev,
                                 const double *__restrict__ d, double *Qd, double *Qx, double *Ad, double *Ax) {
  const double tau = scal[S_TAU];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    const double xi = x[i];
    x_prev[i] = xi;
    x[i] = xi + tau * d[i];
    const double qd = Qd[i] * tau;
    Qd[i] = qd; Qx[i] = Qx[i] + qd;
  }
  if (i < m) {
    const double ad = Ad[i] * tau;
    Ad[i] = ad; Ax[i] = Ax[i] + ad;
  }
}
int step_update_iterate(Engine *e) {
  const int len = e->n > e->m ? e->n : e->m;
  QB_LAUNCH(k_update_iterate, cdiv(len, 256), 256, 0, e->stream, e->n, e->m, e->scal_dev, e->x, e->x_prev, e->d, e->Qdv,
            e->Qx, e->Ad, e->Ax);
  return 0;
}

// update_sigma (iteration.c:86-131); the per-row factor of At_scale goes to sig_fac, the changed rows
// (ascending) to e->changed with their update scale sqrt_sigma_new * sqrt(1 - 1/f^2) in w_pos
__global__ void __launch_bounds__(kListThreads)
k_update_sigma(int m, double theta, double delta, double sigma_max, double sqrt_sigma_max,
               const double *__restrict__ pri_res, const double *__restrict__ pri_res_in, const int *__restrict__ active,
               double *sigma, double *sigma_inv, double *sqrt_sigma, double *sig_fac, int *changed, double *wchg, double *scal) {
  __shared__ int warp_cnt[32];
  __shared__ int base;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const double nrm = scal[S_PRI_RES_RAW];
  if (tid == 0) base = 0;
  __syncthreads();
  for (int start = 0; start < m; start += kListThreads) {
    const int k = start + tid;
    bool chg = false; double fac = 1.0, ssn = 0.0;
    if (k < m) {
      const double pr = fabs(pri_res[k]);
      if ((pr > theta * fabs(pri_res_in[k])) && active[k]) {
        double mult = fmax(1.0, delta * pr / (nrm + 1e-6));
        const double st = mult * sigma[k];
        if (st <= sigma_max) {
          chg = (sigma[k] != st);
          sigma[k] = st; sigma_inv[k] = 1.0 / st;
          mult = sqrt(mult);
          ssn = mult * sqrt_sigma[k]; sqrt_sigma[k] = ssn; fac = mult;
        } else {
          chg = (sigma[k] != sigma_max);
          sigma[k] = sigma_max; sigma_inv[k] = 1.0 / sigma_max;
          fac = sqrt_sigma_max / sqrt_sigma[k];
          ssn = sqrt_sigma_max; sqrt_sigma[k] = ssn;
        }
      }
      sig_fac[k] = fac;
    }
    const unsigned b = __ballot_sync(0xffffffffu, chg);
    if (lane == 0) warp_cnt[warp] = __popc(b);
    __syncthreads();
    int off = base;
    for (int w = 0; w < warp; w++) off += warp_cnt[w];
    if (chg) {
      const int pos = off + __popc(b & ((1u << lane) - 1u));
      changed[pos] = k;
      double f2 = fac * fac; f2 = sqrt(1 - 1 / f2);     // solver_interface.c:457-461
      wchg[pos] = ssn * f2;
    }
    __syncthreads();
    if (tid == 0) { int t = 0; for (int w = 0; w < 32; w++) t += warp_cnt[w]; base += t; }
    __syncthreads();
  }
  if (tid == 0) scal[S_NB_SIGMA_CHANGED] = (double)base;
}
int step_update_sigma(Engine *e, double theta, double delta, double sigma_max, double sqrt_sigma_max) {
  if (e->m == 0) return 0;
  QB_LAUNCH(k_update_sigma, 1, kListThreads, 0, e->stream, e->m, theta, delta, sigma_max, sqrt_sigma_max, e->pri_res,
            e->pri_res_in, e->active, e->sigma, e->sigma_inv, e->sqrt_sigma, e->sig_fac, e->changed, e->w_pos, e->scal_dev);
  return 0;
}

__global__ void __launch_bounds__(kRedThreads)
k_objective(int n, int proximal, double inv_gamma, const double *__restrict__ Qx, const double *__restrict__ x,
            const double *__restrict__ q, double *partials) {
  __shared__ double scratch[32];
  double obj = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    if (proximal) obj += (0.5 * (Qx[i] - inv_gamma * x[i]) + q[i]) * x[i];
    else obj += (0.5 * Qx[i] + q[i]) * x[i];
  }
  block_partial<RED_SUM>(obj, scratch, partials, S_OBJ);
}
int step_objective(Engine *e, bool proximal, double gamma) {
  const int g = red_grid(e->n);
  QB_LAUNCH(k_objective, g, kRedThreads, 0, e->stream, e->n, proximal ? 1 : 0, 1 / gamma, e->Qx, e->x, e->q, e->partials);
  finalize(e, {S_OBJ}, g);
  return 0;
}

// initialize_sigma (iteration.c:50-84): f = x'Qx/2 + q'x, dist2 = |Ax - clip(Ax)|^2  -> one scalar sigma
__global__ void __launch_bounds__(kRedThreads)
k_init_sigma_red(int n, int m, const double *__restrict__ x, const double *__restrict__ Qx, const double *__restrict__ q,
                 const double *__restrict__ Ax, const double *__restrict__ bmin, const double *__restrict__ bmax, double *partials) {
  __shared__ double scratch[32];
  double xqx = 0, qx = 0, d2 = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) { xqx += x[i] * Qx[i]; qx += q[i] * x[i]; }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
    const double t = Ax[i] - fmax(bmin[i], fmin(Ax[i], bmax[i]));
    d2 += t * t;
  }
  block_partial<RED_SUM>(xqx, scratch, partials, S_TMP0);
  block_partial<RED_SUM>(qx, scratch, partials, S_TMP1);
  block_partial<RED_SUM>(d2, scratch, partials, S_TMP2);
}
__global__ void k_fill_sigma(int m, double s, double *sigma, double *sigma_inv, double *sqrt_sigma) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m) { sigma[i] = s; sigma_inv[i] = 1.0 / s; sqrt_sigma[i] = sqrt(s); }
}
int initialize_sigma(Engine *e, double sigma_init) {
  const int len = e->n > e->m ? e->n : e->m;
  const int g = red_grid(len);
  QB_LAUNCH(k_init_sigma_red, g, kRedThreads, 0, e->stream, e->n, e->m, e->x, e->Qx, e->q, e->Ax, e->bmin, e->bmax, e->partials);
  finalize(e, {S_TMP0, S_TMP1, S_TMP2}, g);
  if (int r = sync_scalars(e)) return r;
  const double f = 0.5 * e->scal_host[S_TMP0] + e->scal_host[S_TMP1], dist2 = e->scal_host[S_TMP2];
  const double af = f < 0 ? -f : f;
  double s = sigma_init * (af > 1 ? af : 1) / ((0.5 * dist2) > 1 ? (0.5 * dist2) : 1);
  s = s < 1e4 ? s : 1e4;
  s = s > 1e-4 ? s : 1e-4;
  if (e->m > 0) QB_LAUNCH(k_fill_sigma, cdiv(e->m, 256), 256, 0, e->stream, e->m, s, e->sigma, e->sigma_inv, e->sqrt_sigma);
  e->H_valid = false;
  return 0;
}

// boost_gamma's Gershgorin bound of A_J' Sigma_J A_J (iteration.c:159-211, nonconvex.c:185-210).
// Uses L as scratch: the caller must refactorise afterwards.
__global__ void __launch_bounds__(kRedThreads) k_max_reduce(int n, const double *__restrict__ v, double *partials, int slot) {
  __shared__ double scratch[32];
  double mx = -1.0e300;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) mx = fmax(mx, v[i]);
  block_partial<RED_MAX>(mx, scratch, partials, slot);
}
// KKT path without the Schur structure: upper bound of the Gershgorin bound, row j: sum_{r in J} sigma_r |A_rj| |A_r|_1
// (>= sum_c |sum_r sigma_r A_rj A_rc|; boost_gamma only needs a bound on lambda_max, iteration.c:166-176)
__global__ void k_kkt_gershgorin_rows(int m, const int *__restrict__ rp, const double *__restrict__ rx, const int *__restrict__ active,
                                      const double *__restrict__ sigma, double *row_w) {
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= m) return;
  double s = 0.0;
  if (active[r]) for (int k = rp[r] + lane; k < rp[r + 1]; k += 32) s += fabs(rx[k]);
  s = warp_sum(s);
  if (lane == 0) row_w[r] = active[r] ? sigma[r] * s : 0.0;
}
__global__ void k_kkt_gershgorin_cols(int n, const int *__restrict__ cp, const int *__restrict__ ci, const double *__restrict__ cx,
                                      const double *__restrict__ row_w, double *out) {
  const int lane = threadIdx.x & 31;
  const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (j >= n) return;
  double s = 0.0;
  for (int k = cp[j] + lane; k < cp[j + 1]; k += 32) s += fabs(cx[k]) * row_w[ci[k]];
  s = warp_sum(s);
  if (lane == 0) out[j] = s;
}

int step_gershgorin_AtSA(Engine *e, double *ub_host) {
  if (e->kkt && !e->sp) {
    QB_LAUNCH(k_kkt_gershgorin_rows, cdiv(e->m, 8), 256, 0, e->stream, e->m, e->A_csr.p, e->A_csr.x, e->active, e->sigma, e->tmp_m);
    QB_LAUNCH(k_kkt_gershgorin_cols, cdiv(e->n, 8), 256, 0, e->stream, e->n, e->A_csc.p, e->A_csc.i, e->A_csc.x, e->tmp_m, e->tmp_n);
    const int g = red_grid(e->n);
    QB_LAUNCH(k_max_reduce, g, kRedThreads, 0, e->stream, e->n, e->tmp_n, e->partials, S_TMP4);
    finalize(e, {S_TMP4}, g);
    if (int r = sync_scalars(e)) return r;
    *ub_host = e->scal_host[S_TMP4];
    return 0;
  }
  if (e->sp) {   // A_J' Sigma_J A_J assembled into the factor's panels (the caller refactorises afterwards)
    if (int r = sparse_chol_assemble(e->sp, e->stream, e->spL, false, e->Q_csr.p, e->Q_csr.i, e->Q_csr.x, e->A_csc.p, e->A_csc.i,
                                     e->A_csc.x, e->A_csr.p, e->A_csr.i, e->A_csr.x, e->active, e->sigma, 0.0)) return r;
    if (int r = sparse_chol_abs_rowsums(e->sp, e->stream, e->spL, e->tmp_n)) return r;
    const int g = red_grid(e->n);
    QB_LAUNCH(k_max_reduce, g, kRedThreads, 0, e->stream, e->n, e->tmp_n, e->partials, S_TMP4);
    finalize(e, {S_TMP4}, g);
    if (int r = sync_scalars(e)) return r;
    *ub_host = e->scal_host[S_TMP4];
    return 0;
  }
  QB_CUDA_TRY(cudaMemsetAsync(e->L, 0, sizeof(double) * (size_t)e->ld * e->npad, e->stream));
  // temporary lists of the committed active set; the H record is left untouched (separate scratch arrays)
  QB_LAUNCH(k_build_lists, 1, kListThreads, 0, e->stream, e->m, 1, 1, e->active_cand, e->active, e->active_old, e->sigma,
            e->sqrt_sigma, (int *)e->ls_val[1], e->ls_da, e->list_pos, e->list_neg, e->w_pos, e->w_neg, e->scal_dev);
  if (int r = sync_scalars(e)) return r;
  const int npos = (int)e->scal_host[S_TMP0];
  if (int r = syrk_list(e, e->L, e->list_pos, e->w_pos, false, npos, 1.0)) return r;
  if (e->sh_world > 1) { if (int r = shard_allreduce(e->L, e->L, (size_t)e->ld * e->npad, false, e->stream)) return r; }
  if (int r = sym_abs_rowsums(e->stream, e->n, e->L, e->ld, e->tmp_n)) return r;
  const int g = red_grid(e->n);
  QB_LAUNCH(k_max_reduce, g, kRedThreads, 0, e->stream, e->n, e->tmp_n, e->partials, S_TMP4);
  finalize(e, {S_TMP4}, g);
  if (int r = sync_scalars(e)) return r;
  *ub_host = e->scal_host[S_TMP4];
  return 0;
}

// dual objective (iteration.c:272-299): -(1/2)(A'y+q)' Q^-1 (A'y+q) - sum_i (y_i>0 ? y_i bmax_i : y_i bmin_i)
__global__ void k_add_to_pad(int n, int npad, const double *__restrict__ a, const double *__restrict__ b, double *out, double *keep) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < npad) { const double v = (i < n) ? a[i] + 1.0 * b[i] : 0.0; out[i] = v; if (i < n) keep[i] = v; }
}
__global__ void __launch_bounds__(kRedThreads)
k_dual_obj(int n, int m, const double *__restrict__ rhs, const double *__restrict__ sol, const double *__restrict__ y,
           const double *__restrict__ bmin, const double *__restrict__ bmax, double *partials) {
  __shared__ double scratch[32];
  double dot = 0, sup = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) dot += rhs[i] * sol[i];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) sup += y[i] > 0 ? y[i] * bmax[i] : y[i] * bmin[i];
  block_partial<RED_SUM>(dot, scratch, partials, S_TMP0);
  block_partial<RED_SUM>(sup, scratch, partials, S_TMP1);
}
int factor_Q_for_dual(Engine *e) {
  if (e->sp) {
    if (!e->spLQ) return 1;
    if (int r = sparse_chol_assemble(e->sp, e->stream, e->spLQ, true, e->Q_csr.p, e->Q_csr.i, e->Q_csr.x, e->A_csc.p, e->A_csc.i,
                                     e->A_csc.x, e->A_csr.p, e->A_csr.i, e->A_csr.x, nullptr, e->sigma, 0.0)) return r;
    return sparse_chol_factor(e->sp, e->stream, e->spLQ, e->info_dev);
  }
  if (!e->LQ) return 1;
  if (int r = init_lower_from_Q(e, e->LQ)) return r;
  QB_LAUNCH(k_add_diag_pad, cdiv(e->npad, 256), 256, 0, e->stream, e->n, e->npad, e->LQ, e->ld, 0.0);
  return potrf_lower(e->stream, e->npad, e->LQ, e->ld, e->invdiagQ, e->info_dev);
}
int step_dual_objective(Engine *e, double *val_host) {
  QB_LAUNCH(k_add_to_pad, cdiv(e->npad, 256), 256, 0, e->stream, e->n, e->npad, e->Aty, e->q, e->vpad, e->tmp_n);
  if (e->sp) { if (int r = sparse_chol_solve(e->sp, e->stream, e->spLQ, e->tmp_n, e->vpad, false)) return r; }
  else if (int r = chol_solve(e->stream, e->npad, e->LQ, e->ld, e->invdiagQ, e->vpad)) return r;
  const int len = e->n > e->m ? e->n : e->m;
  const int g = red_grid(len);
  QB_LAUNCH(k_dual_obj, g, kRedThreads, 0, e->stream, e->n, e->m, e->tmp_n, e->vpad, e->y, e->bmin, e->bmax, e->partials);
  finalize(e, {S_TMP0, S_TMP1}, g);
  if (int r = sync_scalars(e)) return r;
  *val_host = -0.5 * e->scal_host[S_TMP0] - e->scal_host[S_TMP1];
  return 0;
}

// ================================================================================================
// Ruiz equilibration on the device (scaling.c:34-113).  max/sqrt/reciprocal/multiply are exact or
// correctly rounded, and the multiplication order of cholmod_scale is kept ((a*E_i)*D_j, q*(D_j*D_i)*c),
// so the scaled data are bit-identical to the reference's.
// ================================================================================================
__global__ void __launch_bounds__(256) k_csr_absmax(int rows, const int *__restrict__ p, const double *__restrict__ v, double *out) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  double mx = 0.0;
  for (int k = p[row] + lane; k < p[row + 1]; k += 32) mx = fmax(mx, fabs(v[k]));
  mx = warp_max(mx);
  if (lane == 0) out[row] = mx;
}
__global__ void __launch_bounds__(256) k_dense_absmax_cols(int len, int ncols, int ld, const double *__restrict__ M, double *out) {
  const int lane = threadIdx.x & 31;
  const int col = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (col >= ncols) return;
  const double *c = M + (size_t)col * ld;
  double mx = 0.0;
  for (int i = lane; i < len; i += 32) mx = fmax(mx, fabs(c[i]));
  mx = warp_max(mx);
  if (lane == 0) out[col] = mx;
}
__global__ void __launch_bounds__(128) k_dense_absmax_rows(int nrows, int ncols, int ld, const double *__restrict__ M,
                                                           double *partial, int cols_per_split) {
  const int i = blockIdx.x * 128 + threadIdx.x;
  if (i >= nrows) return;
  const int k0 = blockIdx.y * cols_per_split, k1 = min(ncols, k0 + cols_per_split);
  double mx = 0.0;
  for (int k = k0; k < k1; k++) mx = fmax(mx, fabs(M[(size_t)i + (size_t)k * ld]));
  partial[(size_t)blockIdx.y * nrows + i] = mx;
}
__global__ void k_max_splits(int nrows, int splits, const double *__restrict__ partial, double *y) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nrows) return;
  double mx = 0.0;
  for (int s = 0; s < splits; s++) mx = fmax(mx, partial[(size_t)s * nrows + i]);
  y[i] = mx;
}
__global__ void k_ruiz_post(int len, double *t, double *acc) {   // t <- 1/sqrt(limit(t)); acc <- acc * t
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= len) return;
  double v = t[i];
  v = v < 1e-12 ? 1.0 : v;
  v = sqrt(v);
  v = 1.0 / v;
  t[i] = v;
  acc[i] = acc[i] * v;
}
// outer_is_row: CSR (outer = row i, inner = column j); else CSC (outer = column j, inner = row i)
__global__ void __launch_bounds__(256) k_scale_sparse(int outer, const int *__restrict__ p, const int *__restrict__ ci, double *v,
                                                      const double *__restrict__ Et, const double *__restrict__ Dt, int outer_is_row) {
  const int lane = threadIdx.x & 31;
  const int o = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (o >= outer) return;
  for (int k = p[o] + lane; k < p[o + 1]; k += 32) {
    const int in = ci[k];
    const double e = outer_is_row ? Et[o] : Et[in], dd = outer_is_row ? Dt[in] : Dt[o];
    double x = v[k];
    x *= e; x *= dd;
    v[k] = x;
  }
}
__global__ void k_scale_dense_At(int n, int m, double *At, const double *__restrict__ Et, const double *__restrict__ Dt) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
  if (j >= n) return;
  double x = At[(size_t)j + (size_t)n * i];
  x *= Et[i]; x *= Dt[j];
  At[(size_t)j + (size_t)n * i] = x;
}
__global__ void __launch_bounds__(256) k_scale_Q_sparse(int n, const int *__restrict__ p, const int *__restrict__ ci, double *v,
                                                        const double *__restrict__ D, double cc, int use_D) {
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= n) return;
  for (int k = p[r] + lane; k < p[r + 1]; k += 32) {
    double x = v[k];
    if (use_D) x *= D[r] * D[ci[k]];
    x *= cc;
    v[k] = x;
  }
}
__global__ void k_scale_Q_dense(int n, double *Q, const double *__restrict__ D, double cc, int use_D) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
  if (i >= n) return;
  double x = Q[(size_t)i + (size_t)n * j];
  if (use_D) x *= D[j] * D[i];
  x *= cc;
  Q[(size_t)i + (size_t)n * j] = x;
}
__global__ void k_recip(int len, const double *__restrict__ a, double *b) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < len) b[i] = 1.0 / a[i];
}
__global__ void __launch_bounds__(kRedThreads) k_absmax_sum2(int n, const double *__restrict__ a, const double *__restrict__ b,
                                                             double *partials, int slot) {   // max |a + b| (b may be null)
  __shared__ double scratch[32];
  double mx = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) mx = fmax(mx, fabs(b ? a[i] + 1.0 * b[i] : a[i]));
  block_partial<RED_MAX>(mx, scratch, partials, slot);
}

// column / row infinity norms of A (mat_inf_norm_cols / mat_inf_norm_rows, solver_interface.c:276-314)
int ruiz_norms_public(Engine *e, double *Dt, double *Et) {
  const int n = e->n, m = e->m;
  if (m == 0) return vec_set(e, Dt, 0.0, n);
  if (e->A_dense) {
    const int ml = e->m_loc;   // this rank's rows (all of them on a single GPU)
    if (ml > 0) {
      int splits = e->gemv_splits; if (splits > ml) splits = ml;
      const int cps = cdiv(ml, splits); splits = cdiv(ml, cps);
      dim3 grid(cdiv(n, 128), splits);
      QB_LAUNCH(k_dense_absmax_rows, grid, 128, 0, e->stream, n, ml, n, e->At, e->gemv_partials, cps);
      QB_LAUNCH(k_max_splits, cdiv(n, 256), 256, 0, e->stream, n, splits, e->gemv_partials, Dt);
      QB_LAUNCH(k_dense_absmax_cols, cdiv(ml, 8), 256, 0, e->stream, n, ml, n, e->At, Et + e->m_lo);
    } else if (int r = vec_set(e, Dt, 0.0, n)) return r;
    if (e->sh_world > 1) {   // column norms: max over the ranks' row blocks; row norms: gather the blocks
      if (int r = shard_allreduce(Dt, Dt, (size_t)n, true, e->stream)) return r;
      if (int r = shard_allgather(Et, (size_t)e->m_cap, e->stream)) return r;
    }
  } else {
    QB_LAUNCH(k_csr_absmax, cdiv(n, 8), 256, 0, e->stream, n, e->A_csc.p, e->A_csc.x, Dt);
    QB_LAUNCH(k_csr_absmax, cdiv(m, 8), 256, 0, e->stream, m, e->A_csr.p, e->A_csr.x, Et);
  }
  return 0;
}

int scale_Q_values(Engine *e, double cc, bool use_D) {
  if (e->Q_dense) {
    dim3 grid(cdiv(e->n, 256), e->n);
    QB_LAUNCH(k_scale_Q_dense, grid, 256, 0, e->stream, e->n, e->Qd, e->D, cc, use_D ? 1 : 0);
  } else {
    QB_LAUNCH(k_scale_Q_sparse, cdiv(e->n, 8), 256, 0, e->stream, e->n, e->Q_csr.p, e->Q_csr.i, e->Q_csr.x, e->D, cc, use_D ? 1 : 0);
  }
  e->H_valid = false;
  return 0;
}

static int ruiz_impl(Engine *e, int iters, bool use_Qx, double *c_out) {
  const int n = e->n, m = e->m;
  vec_set(e, e->D, 1.0, n); vec_set(e, e->E, 1.0, m);
  for (int it = 0; it < iters && m > 0; it++) {
    double *Dt = e->tmp_n, *Et = e->tmp_m;
    if (int r = ruiz_norms_public(e, Dt, Et)) return r;
    QB_LAUNCH(k_ruiz_post, cdiv(n, 256), 256, 0, e->stream, n, Dt, e->D);
    QB_LAUNCH(k_ruiz_post, cdiv(m, 256), 256, 0, e->stream, m, Et, e->E);
    if (e->A_dense) {
      if (e->m_loc > 0) {
        dim3 grid(cdiv(n, 256), e->m_loc);
        QB_LAUNCH(k_scale_dense_At, grid, 256, 0, e->stream, n, e->m_loc, e->At, Et + e->m_lo, Dt);
      }
    } else {
      QB_LAUNCH(k_scale_sparse, cdiv(n, 8), 256, 0, e->stream, n, e->A_csc.p, e->A_csc.i, e->A_csc.x, Et, Dt, 0);
      QB_LAUNCH(k_scale_sparse, cdiv(m, 8), 256, 0, e->stream, m, e->A_csr.p, e->A_csr.i, e->A_csr.x, Et, Dt, 1);
    }
  }
  vec_ewprod(e, e->D, e->q, e->q, n);
  const int g = red_grid(n);
  if (use_Qx) {
    vec_ewprod(e, e->D, e->Qx, e->Qx, n);
    QB_LAUNCH(k_absmax_sum2, g, kRedThreads, 0, e->stream, n, e->Qx, e->q, e->partials, S_TMP4);
  } else {
    QB_LAUNCH(k_absmax_sum2, g, kRedThreads, 0, e->stream, n, e->q, (const double *)nullptr, e->partials, S_TMP4);
  }
  finalize(e, {S_TMP4}, g);
  if (int r = sync_scalars(e)) return r;
  const double nrm = e->scal_host[S_TMP4];
  const double cc = 1 / (nrm > 1.0 ? nrm : 1.0);
  vec_scale(e, cc, e->q, n);
  scale_Q_values(e, cc, true);
  QB_LAUNCH(k_recip, cdiv(n, 256), 256, 0, e->stream, n, e->D, e->Dinv);
  if (m > 0) QB_LAUNCH(k_recip, cdiv(m, 256), 256, 0, e->stream, m, e->E, e->Einv);
  vec_ewprod(e, e->E, e->bmin, e->bmin, m);
  vec_ewprod(e, e->E, e->bmax, e->bmax, m);
  *c_out = cc;
  QB_CUDA_TRY(cudaGetLastError());
  return 0;
}
int engine_ruiz_scale(Engine *e, int iters, double *c_out) { return ruiz_impl(e, iters, false, c_out); }
int engine_ruiz_rescale(Engine *e, int iters, double *c_out) { return ruiz_impl(e, iters, true, c_out); }

// ================================================================================================
// LOBPCG (nonconvex.c:29-168): lambda_min of the (scaled) Q.  Vectors stay on the device; the 2x2 / 3x3
// (generalised) eigenproblems are solved on the host from one scalar block per iteration.
// ================================================================================================
struct DotList { int n; const double *a[10]; const double *b[10]; int slot[10]; };
__global__ void __launch_bounds__(kRedThreads) k_multi_dot(int len, DotList dl, double *partials) {
  __shared__ double scratch[32];
  for (int t = 0; t < dl.n; t++) {
    double acc = 0.0;
    const double *a = dl.a[t], *b = dl.b[t];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < len; i += gridDim.x * blockDim.x) acc += a[i] * b[i];
    block_partial<RED_SUM>(acc, scratch, partials, dl.slot[t]);
  }
}
static int multi_dot(Engine *e, int len, std::initializer_list<std::pair<const double *, const double *>> pairs, int first_slot) {
  DotList dl; dl.n = 0;
  SlotList sl; sl.n = 0;
  for (auto &pr : pairs) { dl.a[dl.n] = pr.first; dl.b[dl.n] = pr.second; dl.slot[dl.n] = first_slot + dl.n; sl.slot[sl.n++] = first_slot + dl.n; dl.n++; }
  const int g = red_grid(len);
  QB_LAUNCH(k_multi_dot, g, kRedThreads, 0, e->stream, len, dl, e->partials);
  QB_LAUNCH(k_finalize, sl.n, 256, 0, e->stream, sl, e->partials, g, e->scal_dev);
  return 0;
}
__global__ void k_axpby(int len, double a, const double *x, double b, const double *y, double *out) {   // out = a*x + b*y
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < len) out[i] = a * x[i] + b * y[i];
}
static int axpby(Engine *e, int len, double a, const double *x, double b, const double *y, double *out) {
  QB_LAUNCH(k_axpby, cdiv(len, 256), 256, 0, e->stream, len, a, x, b, y, out);
  return 0;
}
__global__ void __launch_bounds__(kRedThreads) k_absmax1(int n, const double *__restrict__ a, double *partials, int slot) {
  __shared__ double scratch[32];
  double mx = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) mx = fmax(mx, fabs(a[i]));
  block_partial<RED_MAX>(mx, scratch, partials, slot);
}

static void jacobi_eig3(int n, double A[3][3], double V[3][3], double w[3]) {
  for (int i = 0; i < n; i++) for (int j = 0; j < n; j++) V[i][j] = (i == j);
  for (int sweep = 0; sweep < 100; sweep++) {
    double off = 0; for (int i = 0; i < n; i++) for (int j = i + 1; j < n; j++) off += A[i][j] * A[i][j];
    if (off < 1e-300) break;
    for (int p = 0; p < n; p++) for (int q = p + 1; q < n; q++) {
      if (A[p][q] == 0.0) continue;
      const double th = (A[q][q] - A[p][p]) / (2 * A[p][q]);
      const double t = (th >= 0 ? 1.0 : -1.0) / (fabs(th) + sqrt(th * th + 1)), c = 1 / sqrt(t * t + 1), s = t * c;
      for (int k = 0; k < n; k++) { const double akp = A[k][p], akq = A[k][q]; A[k][p] = c * akp - s * akq; A[k][q] = s * akp + c * akq; }
      for (int k = 0; k < n; k++) { const double apk = A[p][k], aqk = A[q][k]; A[p][k] = c * apk - s * aqk; A[q][k] = s * apk + c * aqk; }
      for (int k = 0; k < n; k++) { const double vkp = V[k][p], vkq = V[k][q]; V[k][p] = c * vkp - s * vkq; V[k][q] = s * vkp + c * vkq; }
    }
  }
  for (int i = 0; i < n; i++) w[i] = A[i][i];
  for (int i = 0; i < n; i++) for (int j = i + 1; j < n; j++) if (w[j] < w[i]) {
    double t = w[i]; w[i] = w[j]; w[j] = t;
    for (int k = 0; k < n; k++) { t = V[k][i]; V[k][i] = V[k][j]; V[k][j] = t; }
  }
}
// smallest eigenpair of B y = lambda C y, y'Cy = 1 (what LAPACKE_dsygv itype 1 returns in column 0)
static double gen_eig_min3(int n, double B[3][3], double Cm[3][3], double y[3]) {
  double R[3][3] = {{0}}, Ri[3][3] = {{0}}, T[3][3], M[3][3], V[3][3], w[3];
  for (int j = 0; j < n; j++) {
    double s = Cm[j][j]; for (int k = 0; k < j; k++) s -= R[j][k] * R[j][k];
    R[j][j] = sqrt(s);
    for (int i = j + 1; i < n; i++) { s = Cm[i][j]; for (int k = 0; k < j; k++) s -= R[i][k] * R[j][k]; R[i][j] = s / R[j][j]; }
  }
  for (int j = 0; j < n; j++) {
    Ri[j][j] = 1 / R[j][j];
    for (int i = j + 1; i < n; i++) { double s = 0; for (int k = j; k < i; k++) s -= R[i][k] * Ri[k][j]; Ri[i][j] = s / R[i][i]; }
  }
  for (int i = 0; i < n; i++) for (int j = 0; j < n; j++) { double s = 0; for (int k = 0; k < n; k++) s += Ri[i][k] * B[k][j]; T[i][j] = s; }
  for (int i = 0; i < n; i++) for (int j = 0; j < n; j++) { double s = 0; for (int k = 0; k < n; k++) s += T[i][k] * Ri[j][k]; M[i][j] = s; }
  for (int i = 0; i < n; i++) for (int j = i + 1; j < n; j++) M[i][j] = M[j][i] = 0.5 * (M[i][j] + M[j][i]);
  jacobi_eig3(n, M, V, w);
  for (int i = 0; i < n; i++) { double s = 0; for (int k = 0; k < n; k++) s += Ri[k][i] * V[k][0]; y[i] = s; }
  return w[0];
}

int lobpcg_device(Engine *e, const double *x0_host, double *lambda_out, long long *iters_out) {
  const int n = e->n;
  // vector aliases follow the reference: x=d, Ax=Qd, w=vpad(neg_dphi), Aw=Atyh, p=tmp_n, Ap=tmp_n2
  double *x = e->d, *Ax = e->Qdv, *w = e->vpad, *Aw = e->Atyh, *p = e->tmp_n, *Ap = e->tmp_n2;
  double *h = e->scal_host;
  if (int r = upload(e, x, x0_host, n)) return r;
  multi_dot(e, n, {{x, x}}, S_L0);
  if (int r = sync_scalars(e)) return r;
  vec_scale(e, 1.0 / sqrt(h[S_L0]), x, n);
  spmv_Q(e, x, Ax);
  multi_dot(e, n, {{x, Ax}}, S_L0);
  if (int r = sync_scalars(e)) return r;
  double lambda = h[S_L0];
  axpby(e, n, 1.0, Ax, -lambda, x, w);
  multi_dot(e, n, {{x, w}}, S_L0);
  if (int r = sync_scalars(e)) return r;
  axpby(e, n, 1.0, w, -h[S_L0], x, w);
  multi_dot(e, n, {{w, w}}, S_L0);
  if (int r = sync_scalars(e)) return r;
  vec_scale(e, 1.0 / sqrt(h[S_L0]), w, n);
  spmv_Q(e, w, Aw);
  multi_dot(e, n, {{Aw, x}, {Aw, w}}, S_L0);
  if (int r = sync_scalars(e)) return r;
  double xAw = h[S_L0], wAw = h[S_L1];
  double B[3][3] = {{lambda, xAw, 0}, {xAw, wAw, 0}, {0, 0, 0}}, I2[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}}, y[3];
  lambda = gen_eig_min3(2, B, I2, y);
  axpby(e, n, y[1], w, 0.0, w, p);
  axpby(e, n, y[1], Aw, 0.0, Aw, Ap);
  axpby(e, n, 1.0, p, y[0], x, x);
  axpby(e, n, 1.0, Ap, y[0], Ax, Ax);
  long long it; const long long max_iter = 1000;
  const int g = red_grid(n);
  for (it = 0; it < max_iter; it++) {
    axpby(e, n, 1.0, Ax, -lambda, x, w);
    QB_LAUNCH(k_absmax1, g, kRedThreads, 0, e->stream, n, w, e->partials, S_LMAX);
    finalize(e, {S_LMAX}, g);
    multi_dot(e, n, {{x, w}, {w, w}, {p, p}}, S_L0);
    if (int r = sync_scalars(e)) return r;
    if (h[S_LMAX] < 1e-5) {
      const double norm_w = sqrt(h[S_L1]);
      lambda -= sqrt(2.0) * norm_w + 1e-6;
      if (n <= 3) lambda -= 1e-6;
      break;
    }
    axpby(e, n, 1.0, w, -h[S_L0], x, w);
    const double p_norm_inv = 1.0 / sqrt(h[S_L2]);
    vec_scale(e, p_norm_inv, p, n);
    vec_scale(e, p_norm_inv, Ap, n);
    multi_dot(e, n, {{w, w}}, S_L0);
    if (int r = sync_scalars(e)) return r;
    vec_scale(e, 1.0 / sqrt(h[S_L0]), w, n);
    spmv_Q(e, w, Aw);
    multi_dot(e, n, {{Ax, w}, {w, Aw}, {Ax, p}, {Aw, p}, {Ap, p}, {x, p}, {w, p}}, S_L0);
    if (int r = sync_scalars(e)) return r;
    xAw = h[S_L0]; wAw = h[S_L1];
    const double xAp = h[S_L2], wAp = h[S_L3], pAp = h[S_L4], xp = h[S_L5], wp = h[S_L6];
    double B3[3][3] = {{lambda, xAw, xAp}, {xAw, wAw, wAp}, {xAp, wAp, pAp}};
    double C3[3][3] = {{1, 0, xp}, {0, 1, wp}, {xp, wp, 1}};
    lambda = gen_eig_min3(3, B3, C3, y);
    axpby(e, n, y[2], p, y[1], w, p);
    axpby(e, n, y[2], Ap, y[1], Aw, Ap);
    axpby(e, n, y[0], x, 1.0, p, x);
    axpby(e, n, y[0], Ax, 1.0, Ap, Ax);
  }
  *lambda_out = lambda;
  if (iters_out) *iters_out = it;
  QB_CUDA_TRY(cudaGetLastError());
  return 0;
}

// ================================================================================================
// engine construction: host CSC (int64, the CHOLMOD layout of the drop-in API) -> device layouts
// ================================================================================================
int init_slot_ops();

__global__ void k_transpose_to_At(int m, int n, const double *__restrict__ A /* m x n col-major */, double *At /* n x m */) {
  __shared__ double tile[32][33];
  const int i0 = blockIdx.x * 32, j0 = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int i = i0 + threadIdx.x, j = j0 + r;
    if (i < m && j < n) tile[r][threadIdx.x] = A[(size_t)i + (size_t)m * j];
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int j = j0 + threadIdx.x, i = i0 + r;
    if (i < m && j < n) At[(size_t)j + (size_t)n * i] = tile[threadIdx.x][r];
  }
}
// packed lower CSC of a fully dense symmetric matrix (column j holds rows j..n-1) -> full n x n
__global__ void k_expand_packed_lower(int n, const double *__restrict__ packed, double *Q) {
  const int j = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || i < j) return;
  const size_t off = (size_t)j * n - (size_t)j * (j - 1) / 2;   // start of column j in the packed array
  const double v = packed[off + (i - j)];
  Q[(size_t)i + (size_t)n * j] = v;
  Q[(size_t)j + (size_t)n * i] = v;
}

// Host -> device copy of a large PAGEABLE buffer (the caller's CSC values: 1.28 GB at n = 8000, m = 16000).  cudaMemcpy stages
// pageable memory through one internal pinned buffer with a single host thread (~9 GB/s measured on the box: 117 ms for A).  Here T
// host threads each copy their own interleaved 16 MB chunks into their own pinned slots and queue the DMA on their own stream, so the
// host-side memcpy runs T-wide and overlaps the transfers.  Falls back to cudaMemcpy for small buffers or if the staging memory
// cannot be allocated.  Blocking: everything has landed when it returns.
static int staged_upload(void *dst, const void *src, size_t bytes) {
  constexpr size_t CH = 16u << 20;
  constexpr int T = 4, NS = 2;
  static void *stage[T][NS] = {};
  static int stage_ok = -1;
  static std::mutex mu;
  if (bytes < (size_t)(64u << 20)) { QB_CUDA_TRY(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice)); return 0; }
  std::lock_guard<std::mutex> lk(mu);
  if (stage_ok < 0) {
    stage_ok = 1;
    for (int t = 0; t < T && stage_ok; t++)
      for (int k = 0; k < NS && stage_ok; k++)
        if (cudaHostAlloc(&stage[t][k], CH, cudaHostAllocDefault) != cudaSuccess) { stage_ok = 0; cudaGetLastError(); }
  }
  if (!stage_ok) { QB_CUDA_TRY(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice)); return 0; }
  int dev = 0;
  QB_CUDA_TRY(cudaGetDevice(&dev));
  const size_t nchunks = (bytes + CH - 1) / CH;
  int rc[T] = {};
  auto work = [&](int t) {
    if (cudaSetDevice(dev) != cudaSuccess) { rc[t] = 1; return; }
    cudaStream_t st; cudaEvent_t ev[NS];
    if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) { rc[t] = 1; return; }
    for (int k = 0; k < NS; k++) cudaEventCreateWithFlags(&ev[k], cudaEventDisableTiming);
    int used = 0;
    for (size_t c = (size_t)t; c < nchunks; c += T, used++) {
      const int k = used % NS;
      const size_t off = c * CH, len = (bytes - off < CH) ? bytes - off : CH;
      if (used >= NS && cudaEventSynchronize(ev[k]) != cudaSuccess) { rc[t] = 1; break; }
      memcpy(stage[t][k], (const char *)src + off, len);
      if (cudaMemcpyAsync((char *)dst + off, stage[t][k], len, cudaMemcpyHostToDevice, st) != cudaSuccess) { rc[t] = 1; break; }
      cudaEventRecord(ev[k], st);
    }
    if (cudaStreamSynchronize(st) != cudaSuccess) rc[t] = 1;
    for (int k = 0; k < NS; k++) cudaEventDestroy(ev[k]);
    cudaStreamDestroy(st);
  };
  std::vector<std::thread> th;
  for (int t = 0; t < T; t++) th.emplace_back(work, t);
  for (auto &x : th) x.join();
  for (int t = 0; t < T; t++) if (rc[t]) { fprintf(stderr, "[qpalm_b200] staged upload failed\n"); return 1; }
  return 0;
}

template <typename T>
static int up(T **dst, const T *src, size_t count) {
  if (int r = dev_alloc((void **)dst, sizeof(T) * (count ? count : 1))) return r;
  if (count) { if (int r = staged_upload(*dst, src, sizeof(T) * count)) return r; }
  return 0;
}
static int upload_sparse(SparseDev *S, int rows, int cols, const int *p, const int *i, const double *x) {
  S->rows = rows; S->cols = cols; S->nnz = p[rows];
  if (int r = up(&S->p, p, (size_t)rows + 1)) return r;
  // two elements of zero padding: the SpMV kernel reads aligned pairs (masked lanes may touch the element after the last)
  {
    const size_t cnt = (size_t)S->nnz;
    if (int r = dev_alloc((void **)&S->i, sizeof(int) * (cnt + 2))) return r;
    if (int r = dev_alloc((void **)&S->x, sizeof(double) * (cnt + 2))) return r;
    QB_CUDA_TRY(cudaMemset(S->i + cnt, 0, sizeof(int) * 2));
    QB_CUDA_TRY(cudaMemset(S->x + cnt, 0, sizeof(double) * 2));
    if (cnt) {
      QB_CUDA_TRY(cudaMemcpy(S->i, i, sizeof(int) * cnt, cudaMemcpyHostToDevice));
      QB_CUDA_TRY(cudaMemcpy(S->x, x, sizeof(double) * cnt, cudaMemcpyHostToDevice));
    }
    return 0;
  }
}

// The dense fast paths upload the value array verbatim, which is only right when the column listings are complete AND in
// ascending row order (callers may pass sorted = 0, and a duplicate entry can make the count match by accident): check the
// row indices before trusting them.  Memory-bound scan, a few host threads.
static bool csc_is_full_dense(int n, int m, const long long *Ap, const long long *Ai) {
  for (int j = 0; j <= n; j++) if (Ap[j] != (long long)j * m) return false;
  const int nt = (n >= 64 && (long long)n * m > (1 << 22)) ? 8 : 1;
  std::vector<int> ok(nt, 1);
  auto scan = [&](int t) {
    for (int j = t; j < n && ok[t]; j += nt) {
      const long long *col = Ai + (size_t)j * m;
      long long bad = 0;
      for (int i = 0; i < m; i++) bad |= col[i] ^ (long long)i;
      if (bad) ok[t] = 0;
    }
  };
  if (nt == 1) scan(0);
  else { std::vector<std::thread> th; for (int t = 0; t < nt; t++) th.emplace_back(scan, t); for (auto &x : th) x.join(); }
  for (int v : ok) if (!v) return false;
  return true;
}
static bool csc_is_packed_lower(int n, const long long *Qp, const long long *Qi) {
  long long pos = 0;
  for (int j = 0; j < n; j++) { if (Qp[j] != pos) return false; pos += n - j; }
  if (Qp[n] != pos) return false;
  const int nt = (n >= 512) ? 8 : 1;
  std::vector<int> ok(nt, 1);
  auto scan = [&](int t) {
    for (int j = t; j < n && ok[t]; j += nt) {
      const long long *col = Qi + Qp[j];
      long long bad = 0;
      for (int i = j; i < n; i++) bad |= col[i - j] ^ (long long)i;
      if (bad) ok[t] = 0;
    }
  };
  if (nt == 1) scan(0);
  else { std::vector<std::thread> th; for (int t = 0; t < nt; t++) th.emplace_back(scan, t); for (auto &x : th) x.join(); }
  for (int v : ok) if (!v) return false;
  return true;
}

static int engine_create_impl(Engine *e, Engine **out, int n, int m, const long long *Ap, const long long *Ai, const double *Ax,
                              const long long *Qp, const long long *Qi, const double *Qx,
                              const double *q, const double *bmin, const double *bmax, bool need_LQ, int newton_override);

// Every failure exit releases what was allocated so far (the stream, the arena, matrices, factors): a caller that handles
// the NULL workspace and retries with another configuration finds the HBM free again.
int engine_create(Engine **out, int n, int m, const long long *Ap, const long long *Ai, const double *Ax,
                  const long long *Qp, const long long *Qi, const double *Qx,
                  const double *q, const double *bmin, const double *bmax, bool need_LQ, int newton_override) {
  *out = nullptr;
  int ndev = 0;
  QB_CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (ndev <= 0) { fprintf(stderr, "[qpalm_b200] no CUDA device: this library has no CPU fallback\n"); return 1; }
  Engine *e = new Engine();
  const int rc = engine_create_impl(e, out, n, m, Ap, Ai, Ax, Qp, Qi, Qx, q, bmin, bmax, need_LQ, newton_override);
  if (rc) { *out = nullptr; engine_destroy(e); }
  return rc;
}

static int engine_create_impl(Engine *e, Engine **out, int n, int m, const long long *Ap, const long long *Ai, const double *Ax,
                              const long long *Qp, const long long *Qi, const double *Qx,
                              const double *q, const double *bmin, const double *bmax, bool need_LQ, int newton_override) {
  {   // the device forms use int32 indices: refuse what does not fit instead of overflowing
    const long long nnzA_ = m > 0 ? Ap[n] : 0, nnzQ_ = Qp[n];
    if (nnzA_ > 2147483647LL || 2 * nnzQ_ > 2147483647LL) {
      fprintf(stderr, "[qpalm_b200] nnz(A) = %lld / nnz(Q) = %lld exceed the int32 index range of the device storage\n", nnzA_, nnzQ_);
      return 3;
    }
  }
  const bool timing = getenv("QPALM_B200_SETUP_TIMING") != nullptr;   // phase timers of the setup path (stderr)
  auto t_last = std::chrono::steady_clock::now();
  auto lap = [&](const char *what) {
    if (!timing) return;
    cudaDeviceSynchronize();
    const auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[qpalm_b200] setup: %-32s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(now - t_last).count());
    t_last = now;
  };
  QB_CUDA_TRY(cudaGetDevice(&e->device));
  // a BLOCKING stream: setup uses cudaMemset/cudaMemcpy on the legacy default stream, which must stay ordered
  // with the kernels of this engine (a non-blocking stream raced with the allocation memsets)
  QB_CUDA_TRY(cudaStreamCreate(&e->stream));
  if (int r = init_slot_ops()) return r;
  e->n = n; e->m = m; e->npad = round_up(n > 0 ? n : 1, kPanel); e->ld = e->npad;
  const long long nnzA = m > 0 ? Ap[n] : 0;
  std::vector<int> hA_cp, hA_ci, hA_rp, hA_rj;   // host int32 copies of sparse A for the symbolic analysis
  // ---- A ----
  const char *newton_mode = getenv("QPALM_B200_NEWTON");   // dense | sparse: overrides the density heuristics (tests)
  if (newton_override == 5) newton_override = -1;   // FACTORIZE_SCHUR asked for: density heuristics as usual, never the KKT path
  const bool force_sparse = newton_override == 2 || (!newton_override && newton_mode && !strcmp(newton_mode, "sparse"));
  const bool force_dense = newton_override == 1 || (!newton_override && newton_mode && !strcmp(newton_mode, "dense"));
  e->A_dense = !force_sparse && (m > 0) && ((double)nnzA >= 0.25 * (double)m * (double)n);
  e->m_lo = 0; e->m_loc = m; e->m_cap = m;
  if (e->A_dense && shard_world() > 1 && m >= shard_world()) {   // row-sharded dense QP (shard.cu): keep only this rank's rows of A
    e->sh_world = shard_world(); e->sh_rank = shard_rank();
    e->m_cap = cdiv(m, e->sh_world);
    e->m_lo = e->sh_rank * e->m_cap;
    e->m_loc = m - e->m_lo < e->m_cap ? m - e->m_lo : e->m_cap;
    if (e->m_loc < 0) e->m_loc = 0;
  }
  if (m > 0 && e->A_dense) {
    const int ml = e->m_loc, lo = e->m_lo;
    double *tmp = nullptr;
    if (int r = dev_alloc((void **)&tmp, sizeof(double) * (size_t)(ml ? ml : 1) * n)) return r;
    if (ml > 0 && nnzA == (long long)m * n && csc_is_full_dense(n, m, Ap, Ai)) {   // complete dense CSC in row order: rows lo..lo+ml-1 of every column
      if (ml == m) { if (int r = staged_upload(tmp, Ax, sizeof(double) * (size_t)m * n)) return r; }
      else QB_CUDA_TRY(cudaMemcpy2D(tmp, sizeof(double) * (size_t)ml, Ax + lo, sizeof(double) * (size_t)m, sizeof(double) * (size_t)ml,
                                    (size_t)n, cudaMemcpyHostToDevice));
    } else if (ml > 0) {
      double *hd = (double *)calloc((size_t)ml * n, sizeof(double));
      for (int j = 0; j < n; j++)
        for (long long k = Ap[j]; k < Ap[j + 1]; k++) { const long long r = Ai[k] - lo; if (r >= 0 && r < ml) hd[(size_t)r + (size_t)ml * j] += Ax[k]; }   // duplicates sum, as in the CSR path
      QB_CUDA_TRY(cudaMemcpy(tmp, hd, sizeof(double) * (size_t)ml * n, cudaMemcpyHostToDevice));
      free(hd);
    }
    if (int r = dev_alloc((void **)&e->At, sizeof(double) * (size_t)(ml ? ml : 1) * n)) return r;
    if (ml > 0) {
      dim3 grid(cdiv(ml, 32), cdiv(n, 32)), block(32, 8);
      QB_LAUNCH(k_transpose_to_At, grid, block, 0, e->stream, ml, n, tmp, e->At);
    }
    QB_CUDA_TRY(cudaStreamSynchronize(e->stream));
    cudaFree(tmp);
  } else if (m > 0) {
    int *cp = (int *)malloc(sizeof(int) * ((size_t)n + 1)), *ci = (int *)malloc(sizeof(int) * (size_t)(nnzA + 1));
    for (int j = 0; j <= n; j++) cp[j] = (int)Ap[j];
    for (long long k = 0; k < nnzA; k++) ci[k] = (int)Ai[k];
    if (int r = upload_sparse(&e->A_csc, n, m, cp, ci, Ax)) return r;
    int *rp = (int *)calloc((size_t)m + 2, sizeof(int)), *rj = (int *)malloc(sizeof(int) * (size_t)(nnzA + 1));
    double *rx = (double *)malloc(sizeof(double) * (size_t)(nnzA + 1));
    for (long long k = 0; k < nnzA; k++) rp[Ai[k] + 2]++;
    for (int i = 0; i < m; i++) rp[i + 2] += rp[i + 1];
    for (int j = 0; j < n; j++) for (long long k = Ap[j]; k < Ap[j + 1]; k++) { const int dpos = rp[Ai[k] + 1]++; rj[dpos] = j; rx[dpos] = Ax[k]; }
    if (int r = upload_sparse(&e->A_csr, m, n, rp, rj, rx)) return r;
    hA_cp.assign(cp, cp + n + 1); hA_ci.assign(ci, ci + nnzA); hA_rp.assign(rp + 0, rp + m + 1); hA_rj.assign(rj, rj + nnzA);
    free(cp); free(ci); free(rp); free(rj); free(rx);
  }
  lap("A: convert + upload");
  // ---- Q (only row >= col entries are read: stype -1) ----
  long long nnzL = 0;
  {
    const int nt = (Qp[n] > (1 << 22)) ? 8 : 1;
    std::vector<long long> part(nt, 0);
    auto count = [&](int t) { long long c = 0; for (int j = t; j < n; j += nt) for (long long k = Qp[j]; k < Qp[j + 1]; k++) c += (Qi[k] >= j); part[t] = c; };
    if (nt == 1) count(0);
    else { std::vector<std::thread> th; for (int t = 0; t < nt; t++) th.emplace_back(count, t); for (auto &x : th) x.join(); }
    for (long long c : part) nnzL += c;
  }
  e->Q_dense = !force_sparse && (double)nnzL >= 0.25 * 0.5 * (double)n * ((double)n + 1.0);
  if (e->Q_dense) {
    if (int r = dev_alloc((void **)&e->Qd, sizeof(double) * (size_t)n * n)) return r;
    if (nnzL == (long long)n * (n + 1) / 2 && Qp[n] == nnzL && csc_is_packed_lower(n, Qp, Qi)) {   // packed dense lower triangle in row order: expand on the device
      double *tmp = nullptr;
      if (int r = up(&tmp, Qx, (size_t)nnzL)) return r;
      dim3 grid(cdiv(n, 256), n);
      QB_LAUNCH(k_expand_packed_lower, grid, 256, 0, e->stream, n, tmp, e->Qd);
      QB_CUDA_TRY(cudaStreamSynchronize(e->stream));
      cudaFree(tmp);
    } else {
      double *hd = (double *)calloc((size_t)n * n, sizeof(double));
      for (int j = 0; j < n; j++) for (long long k = Qp[j]; k < Qp[j + 1]; k++) if (Qi[k] >= j) {
        hd[(size_t)Qi[k] + (size_t)n * j] += Qx[k];          // duplicates sum, as in the CSR path
        if (Qi[k] != j) hd[(size_t)j + (size_t)n * Qi[k]] += Qx[k];
      }
      QB_CUDA_TRY(cudaMemcpy(e->Qd, hd, sizeof(double) * (size_t)n * n, cudaMemcpyHostToDevice));
      free(hd);
    }
  } else {
    // full symmetric CSR: row i = entries (i, j <= i) in ascending j, then (i, k > i) in ascending k
    const long long nnzF = 2 * nnzL;   // upper bound (diagonal counted twice)
    int *rj = (int *)malloc(sizeof(int) * (size_t)(nnzF + 1));
    double *rx = (double *)malloc(sizeof(double) * (size_t)(nnzF + 1));
    int *cnt = (int *)calloc((size_t)n + 1, sizeof(int));
    for (int j = 0; j < n; j++) for (long long k = Qp[j]; k < Qp[j + 1]; k++) { const long long i = Qi[k]; if (i < j) continue; cnt[i]++; if (i != j) cnt[j]++; }
    int *start = (int *)malloc(sizeof(int) * ((size_t)n + 1));
    start[0] = 0; for (int i = 0; i < n; i++) start[i + 1] = start[i] + cnt[i];
    int *fill = (int *)malloc(sizeof(int) * ((size_t)n + 1));
    memcpy(fill, start, sizeof(int) * ((size_t)n + 1));
    for (int j = 0; j < n; j++) for (long long k = Qp[j]; k < Qp[j + 1]; k++) { const long long i = Qi[k]; if (i < j) continue; const int dpos = fill[i]++; rj[dpos] = j; rx[dpos] = Qx[k]; }
    for (int j = 0; j < n; j++) for (long long k = Qp[j]; k < Qp[j + 1]; k++) { const long long i = Qi[k]; if (i <= j) continue; const int dpos = fill[j]++; rj[dpos] = (int)i; rx[dpos] = Qx[k]; }
    if (int r = upload_sparse(&e->Q_csr, n, n, start, rj, rx)) return r;
    free(cnt); free(start); free(fill); free(rj); free(rx);
  }
  lap("Q: convert + upload");
  // ---- vectors ----
  const size_t N = (size_t)n, M = (size_t)(e->sh_world > 1 ? e->sh_world * e->m_cap : m);   // m-vectors padded for the in-place allgather
  {   // slab for everything allocated through dv / iv / the sort buffers below (sizes: 40 m-, 24 n-, 8 2m-vectors + slack)
    const size_t cap = 8 * (40 * M + 24 * N + 8 * (2 * M + 1) + (size_t)e->npad) + 4 * 12 * M + 256 * 128 + (1u << 20);
    if (cudaMalloc((void **)&e->arena, cap) == cudaSuccess) {
      e->arena_cap = cap; e->arena_off = 0;
      QB_CUDA_TRY(cudaMemset(e->arena, 0, cap));
    } else { (void)cudaGetLastError(); e->arena = nullptr; }
  }
  auto dv = [&](double **p, size_t len) { return arena_alloc(e, (void **)p, sizeof(double) * (len ? len : 1)); };
  auto iv = [&](int **p, size_t len) { return arena_alloc(e, (void **)p, sizeof(int) * (len ? len : 1)); };
  int rc = 0;
  rc |= up(&e->q, q, N); rc |= dv(&e->bmin, M); rc |= dv(&e->bmax, M);
  if (!rc && m > 0) { rc |= upload(e, e->bmin, bmin, m); rc |= upload(e, e->bmax, bmax, m); }
  rc |= dv(&e->D, N); rc |= dv(&e->Dinv, N); rc |= dv(&e->E, M); rc |= dv(&e->Einv, M);
  rc |= dv(&e->x, N); rc |= dv(&e->y, M); rc |= dv(&e->Ax, M); rc |= dv(&e->Qx, N); rc |= dv(&e->Aty, N);
  rc |= dv(&e->x_prev, N); rc |= dv(&e->x0, N);
  rc |= dv(&e->sigma, M); rc |= dv(&e->sigma_inv, M); rc |= dv(&e->sqrt_sigma, M); rc |= dv(&e->sig_fac, M);
  rc |= dv(&e->Axys, M); rc |= dv(&e->z, M); rc |= dv(&e->pri_res, M); rc |= dv(&e->pri_res_in, M); rc |= dv(&e->yh, M);
  rc |= dv(&e->Atyh, N); rc |= dv(&e->df, N); rc |= dv(&e->dphi, N); rc |= dv(&e->d, N); rc |= dv(&e->Qdv, N); rc |= dv(&e->Ad, M);
  rc |= dv(&e->delta_y, M); rc |= dv(&e->delta_x, N); rc |= dv(&e->tmp_n, N); rc |= dv(&e->tmp_n2, N); rc |= dv(&e->tmp_m, M);
  rc |= dv(&e->vpad, (size_t)e->npad);
  rc |= iv(&e->active, M); rc |= iv(&e->active_old, M); rc |= iv(&e->active_cand, M); rc |= iv(&e->enter, M); rc |= iv(&e->leave, M);
  rc |= iv(&e->changed, M); rc |= iv(&e->list_pos, M); rc |= iv(&e->list_neg, M); rc |= dv(&e->w_pos, M); rc |= dv(&e->w_neg, M);
  rc |= iv(&e->activeH, M); rc |= dv(&e->sigmaH, M);
  rc |= arena_alloc(e, (void **)&e->ls_key[0], sizeof(unsigned long long) * (2 * M + 1));
  rc |= arena_alloc(e, (void **)&e->ls_key[1], sizeof(unsigned long long) * (2 * M + 1));
  rc |= arena_alloc(e, (void **)&e->ls_val[0], sizeof(unsigned int) * (2 * M + 1));
  rc |= arena_alloc(e, (void **)&e->ls_val[1], sizeof(unsigned int) * (2 * M + 1));
  rc |= dv(&e->ls_da, 2 * M); rc |= dv(&e->ls_db, 2 * M);
  e->rs_tiles = cdiv((int)(2 * M) > 0 ? (int)(2 * M) : 1, rsort::TILE);
  rc |= dev_alloc((void **)&e->rs_hist, sizeof(unsigned int) * 256 * (size_t)e->rs_tiles);
  if (rc) return rc;
  lap("vectors");
  // ---- Newton system ----
  // sparse problems whose Schur complement Q + A'A stays sparse: supernodal factor (sparse.cu) instead of dense H / L.
  {
    if (!force_dense && !e->A_dense && !e->Q_dense && e->sh_world == 1 && n > 0) {
      if (hA_cp.empty()) { hA_cp.assign((size_t)n + 1, 0); hA_rp.assign((size_t)m + 1, 0); }
      if (int r = sparse_chol_analyze(&e->sp, n, m, hA_cp.data(), hA_ci.data(), hA_rp.data(), hA_rj.data(), Qp, Qi, force_sparse, e->stream)) return r;
      if (e->sp) {
        const SparseCholInfo *I = sparse_chol_info(e->sp);
        if (getenv("QPALM_B200_VERBOSE"))
          fprintf(stderr, "[qpalm_b200] sparse Newton path: n=%d nnz(S)=%lld nnz(L)=%lld (%.2f%% of dense) supernodes=%d levels=%d "
                          "max front %d x %d, %.3g flop/factorization\n", n, I->nnzS, I->nnzL, 100.0 * I->nnzL / (0.5 * n * (n + 1.0)),
                  I->nsuper, I->nlevels, I->max_nf, I->max_ns, I->flops);
      }
    }
  }
  lap("sparse symbolic analysis + upload");
  // ---- KKT path (kkt.cu).  newton_override 3: asked for (settings->factorization_method == FACTORIZE_KKT, or
  // QPALM_B200_NEWTON=kkt).  Automatic: A and Q sparse, the Schur complement too dense for the supernodal path (so the
  // alternative is a dense n x n factor), n >= 6000 (QPALM_B200_KKT_AUTO_MIN_N), and the reference's own nnz criterion prefers the KKT system.
  {
    const bool sparse_data = !e->A_dense && !e->Q_dense && m > 0 && e->sh_world == 1;
    bool want_kkt = sparse_data && (newton_override == 3 || (!newton_override && newton_mode && !strcmp(newton_mode, "kkt")));
    // (measured: below n ~ 6000 the dense DMMA factor of the filled-in Schur complement is still faster than the level-scheduled KKT factor)
    const char *kkt_min_s = getenv("QPALM_B200_KKT_AUTO_MIN_N");
    const int kkt_auto_min_n = kkt_min_s ? atoi(kkt_min_s) : 6000;
    if (!want_kkt && sparse_data && !newton_override && !newton_mode && !e->sp && n >= kkt_auto_min_n)
      want_kkt = kkt_heuristic_prefers_kkt(n, m, Ap, Ai, Qp, Qi);
    if (want_kkt) {
      if (need_LQ && !e->sp) { fprintf(stderr, "[qpalm_b200] enable_dual_termination is not available on the KKT path without the supernodal Schur structure\n"); return 5; }
      if (int r = kkt_create(&e->kkt, e, n, m, Ap, Ai, Qp, Qi)) { if (r != 1) return r; }
    }
  }
  lap("KKT symbolic analysis + upload");
  const bool no_dense_factor = e->sp || e->kkt;
  const size_t LL = no_dense_factor ? 1 : (size_t)e->ld * e->npad;
  size_t free_b = 0, total_b = 0;
  QB_CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
  e->wcols = e->sp ? 16 : round_up(m < 64 ? 64 : (m > 2048 ? 2048 : m), 16);   // >= one 64-column update sweep
  if (e->sp) {
    rc |= dv(&e->spL, sparse_chol_factor_doubles(e->sp));
    if (need_LQ) rc |= dv(&e->spLQ, sparse_chol_factor_doubles(e->sp));
    if (rc) return rc;
  }
  const size_t need = no_dense_factor ? 0 : sizeof(double) * (LL * (need_LQ ? 3 : 2) + (size_t)e->ld * e->wcols + (size_t)e->npad * kPanel * 2);
  if (need + (256u << 20) > free_b) {
    fprintf(stderr, "[qpalm_b200] dense Newton path needs %.1f GB for n=%d but only %.1f GB of HBM is free "
                    "(and the union pattern Q + A'A is too dense for the supernodal sparse path)\n", need / 1e9, n, free_b / 1e9);
    return 2;
  }
  if (!no_dense_factor) {
    rc |= dv(&e->H, LL); rc |= dv(&e->L, LL); rc |= dv(&e->invdiag, (size_t)e->npad * kPanel);
    rc |= dv(&e->W, (size_t)e->ld * e->wcols);
    if (need_LQ) { rc |= dv(&e->LQ, LL); rc |= dv(&e->invdiagQ, (size_t)e->npad * kPanel); }
  }
  rc |= dv(&e->ud_coef, 2 * 32 * 18 + 16);
  rc |= dv(&e->partials, (size_t)S_COUNT * kRedBlocks);
  {
    const int rowctas = cdiv(n > 0 ? n : 1, 128);
    int splits = cdiv(2048, rowctas); splits = splits < 1 ? 1 : (splits > 64 ? 64 : splits);
    e->gemv_splits = splits;
    rc |= dv(&e->gemv_partials, (size_t)splits * N);
  }
  rc |= dv(&e->scal_dev, S_COUNT);
  rc |= dev_alloc((void **)&e->info_dev, sizeof(int) * 4);
  if (rc) return rc;
  QB_CUDA_TRY(cudaMallocHost((void **)&e->scal_host, sizeof(double) * S_COUNT));
  memset(e->scal_host, 0, sizeof(double) * S_COUNT);
  QB_CUDA_TRY(cudaMallocHost((void **)&e->info_host, sizeof(int) * 4));
  memset(e->info_host, 0, sizeof(int) * 4);
  QB_CUDA_TRY(cudaEventCreate(&e->ev0)); QB_CUDA_TRY(cudaEventCreate(&e->ev1));
  QB_CUDA_TRY(cudaEventCreate(&e->evs0)); QB_CUDA_TRY(cudaEventCreate(&e->evs1));
  e->launches0 = g_kernel_launches;
  if (const char *s = getenv("QPALM_B200_UPDOWN_MAX_RANK")) e->updown_max_rank = atoi(s);
  if (const char *s = getenv("QPALM_B200_UPDOWN_FORCE")) e->updown_force = atoi(s);
  if (const char *s = getenv("QPALM_B200_UPDOWN_GEN_SCALE")) e->updown_gen_scale = atof(s);
  QB_CUDA_TRY(cudaDeviceSynchronize());
  lap("factor storage + scratch");
  *out = e;
  return 0;
}

void engine_destroy(Engine *e) {
  if (!e) return;
  cudaStreamSynchronize(e->stream);
  void *ptrs[] = {e->A_csr.p, e->A_csr.i, e->A_csr.x, e->A_csc.p, e->A_csc.i, e->A_csc.x, e->Q_csr.p, e->Q_csr.i, e->Q_csr.x,
                  e->At, e->Qd, e->q, e->bmin, e->bmax, e->D, e->Dinv, e->E, e->Einv, e->x, e->y, e->Ax, e->Qx, e->Aty,
                  e->x_prev, e->x0, e->sigma, e->sigma_inv, e->sqrt_sigma, e->sig_fac, e->Axys, e->z, e->pri_res,
                  e->pri_res_in, e->yh, e->Atyh, e->df, e->dphi, e->d, e->Qdv, e->Ad, e->delta_y, e->delta_x, e->tmp_n,
                  e->tmp_n2, e->tmp_m, e->vpad, e->active, e->active_old, e->active_cand, e->enter, e->leave, e->changed,
                  e->list_pos, e->list_neg, e->w_pos, e->w_neg, e->activeH, e->sigmaH, e->ls_key[0], e->ls_key[1],
                  e->ls_val[0], e->ls_val[1], e->ls_da, e->ls_db, e->rs_hist, e->H, e->L, e->invdiag, e->W, e->LQ,
                  e->invdiagQ, e->ud_coef, e->partials, e->gemv_partials, e->scal_dev, e->info_dev, e->spL, e->spLQ};
  for (void *p : ptrs) if (p && !in_arena(e, p)) cudaFree(p);
  if (e->arena) cudaFree(e->arena);
  sparse_chol_destroy(e->sp);
  kkt_destroy(e->kkt);
  if (e->scal_host) cudaFreeHost(e->scal_host);
  if (e->info_host) cudaFreeHost(e->info_host);
  if (e->ev0) cudaEventDestroy(e->ev0);
  if (e->ev1) cudaEventDestroy(e->ev1);
  if (e->evs0) cudaEventDestroy(e->evs0);
  if (e->evs1) cudaEventDestroy(e->evs1);
  if (e->stream) { chol_solve_release(e->stream); chol_updown_gen_release(e->stream); cudaStreamDestroy(e->stream); }
  delete e;
}

}  // namespace qb
