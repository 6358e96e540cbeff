// updown_gen.cu -- rank-k update / downdate of the dense Cholesky factor in GENERATOR form: a triangular solve with k
// right-hand sides followed by fully parallel passes, instead of a sweep whose serial chain visits every 32-column panel.
//
// Replaces cholmod_updown (Modify/cholmod_updown.c, kernel Modify/t_cholmod_updown_numkr.c:289-376) as called by
// ldlupdate_entering_constraints / ldldowndate_leaving_constraints / ldlupdate_sigma_changed
// (src/solver_interface.c:407-503):   L L'  <-  L L' + W S W',   S = diag(+1 x kpos, -1 x (k - kpos)),  k <= 32 per pass.
//
// With  What = inv(L) W  the new matrix is  L (I + What S What') L',  so  L_new = L K  with  K = chol(I + What S What').
// K is the identity plus a rank-k semiseparable part with closed-form generators: for column j, with the k x k matrix
//     M_j = S + sum_{p < j} what_p what_p'              (what_p = row p of What; S = inv(S)),
// the Schur complement of the leading j x j block of I + What S What' is  I + What_{>=j} inv(M_j) What_{>=j}',  hence
//     d_j = sqrt(1 + what_j' inv(M_j) what_j),     K_jj = d_j,     K_ij = what_i' z_j  (i > j),     z_j = inv(M_j) what_j / d_j,
// and  L_new(r, j) = d_j L(r, j) + t_r^(j+1)' z_j  with the running remainder  t_r^(j+1) = W_r - sum_{i <= j} L(r, i) what_i
// (the row recurrence w_r -= w_j l_rj of CHOLMOD's kernel, for all k ranks at once).  inv(M_{j+1}) = inv(M_j) - z_j z_j'
// (Sherman-Morrison), so no k x k factorization is needed per row.
//
// What is serial, and what is not:
//   1. k_fwd_multi  -- What = inv(L) W: ONE cooperative dataflow launch, CTA c owns the 128-row blocks c, c + G, ...;
//      solution blocks travel as epoch-tagged 16-byte packets (as flow::k_solve_flow).  This is the only chain: npad / 128
//      steps.  On its way the owner of block
//      row I stores its running sums  sum_{J' < J} L(I, J') What(J')  for every tile (I, J): the start value of t in step 3.
//   2. k_gen_gram / k_gen_scan / k_gen_rows -- Gram matrices of 32-row blocks of What, their exclusive prefix (+ S) = M at
//      the start of each block, then per block (one warp each, all blocks in parallel) inv(M) by Gauss-Jordan in
//      registers and 32 Sherman-Morrison steps giving d_j and z_j.
//   3. k_gen_apply  -- every 128 x 128 tile of L independently: one thread per row walks the tile's columns.
// Every sum has a fixed order (no atomics): re-solves are bit-reproducible (tests/src/test_basic_qp.c:298-305).
// The caller refreshes the inverses of the diagonal blocks afterwards (trtri_diag_blocks).
#include "dense.cuh"
#include "chol32.cuh"
#include <map>
#include <mutex>

namespace qb {
namespace udgen {
constexpr int NB = 128, NT = 256, GB = 32;

__device__ __forceinline__ void pk_store(uint4 *pk, double v, int epoch) {
  const long long b = __double_as_longlong(v);
  asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %2};" ::"l"(pk), "r"((unsigned)(b & 0xffffffffll)), "r"((unsigned)epoch),
               "r"((unsigned)((unsigned long long)b >> 32)) : "memory");
}
__device__ __forceinline__ uint4 pk_load(const uint4 *pk) {
  uint4 v;
  asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(pk) : "memory");
  return v;
}

template <int KW> struct FwdSmem {
  static constexpr int WS = KW + 4;                      // row stride of the What / rs blocks: WS = 4 mod 16 -> conflict-free B fragments
  static constexpr int XLD = NB + 4;                     // column stride of the inverted diagonal block: conflict-free A fragments
  static constexpr size_t bytes = sizeof(double) * ((size_t)XLD * NB + 2 * (size_t)NB * WS);
};

// tile index of (I, J), J <= I
__device__ __host__ __forceinline__ long long tile_id(int I, int J) { return (long long)I * (I + 1) / 2 + J; }

// FP64 tensor-core tile: d (8 x 8) += a (8 x 4, row) * b (4 x 8, col), mma.sync m8n8k4.  Lane l holds a[l >> 2][l & 3],
// b[l & 3][l >> 2] and d[l >> 2][2 (l & 3) + {0, 1}].
__device__ __forceinline__ void dmma884(double &d0, double &d1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// What = inv(L) W.  Warp w of the CTA that owns block row i keeps the 16 x KW block of running sums of rows 16 w .. 16 w + 15
// in DMMA accumulators; the A fragments of tile (i, j) come straight from global memory (requested before the CTA waits
// for What_j), the B fragments from the What_j block in shared memory.  (A first version with one row per thread and scalar
// FMAs against shared-memory operands was bound by the shared-memory pipe: 30 us per block step at k = 32; this one: see
// DESIGN.md.)
template <int KW>
__global__ void __launch_bounds__(NT, 1)
k_fwd_multi(const double *__restrict__ L, int ld, const double *__restrict__ X, const double *__restrict__ W, int ldw, int k,
            double *What, int npad, double *Tdump, int nblk, uint4 *packets, int epoch, int kt) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // the k right-hand sides are independent: blockIdx.y selects a group of KW of the pass's kt columns (its own CTAs, packets
  // and chain), so a 32-column pass runs as two 16-column solves side by side on twice the SMs
  {
    const int c0 = (int)blockIdx.y * KW;
    W += (size_t)c0 * ldw; What += (size_t)c0 * npad; Tdump += (size_t)c0 * NB; packets += (size_t)blockIdx.y * npad * KW;
    k = max(0, min(KW, k - c0));
  }
  constexpr int WS = FwdSmem<KW>::WS, XLD = FwdSmem<KW>::XLD, NN = KW / 8, NP = NB * KW / NT;
  double *Xs = reinterpret_cast<double *>(smem_raw);   // inverse of the current diagonal block, column-major, ld XLD
  double *ws = Xs + XLD * NB;                          // incoming What block  [128][WS]
  double *rs = ws + NB * WS;                           // right-hand side of the diagonal solve  [128][WS]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, tq = lane & 3;
  const int G = gridDim.x;
  for (int i = blockIdx.x; i < nblk; i += G) {
    {
      const double2 *src = reinterpret_cast<const double2 *>(X + (size_t)i * NB * NB);
#pragma unroll 8
      for (int idx = tid; idx < NB * NB / 2; idx += NT) {
        const int rr = (2 * idx) & (NB - 1), c = (2 * idx) >> 7;
        *reinterpret_cast<double2 *>(Xs + rr + XLD * c) = __ldcg(src + idx);
      }
    }
    double acc[2][NN][2];
#pragma unroll
    for (int mb = 0; mb < 2; mb++)
#pragma unroll
      for (int nb = 0; nb < NN; nb++) acc[mb][nb][0] = acc[mb][nb][1] = 0.0;
    const int r0 = 16 * warp + g;                        // this lane's fragment rows: r0 and r0 + 8
    for (int j = 0; j < i; j++) {
      const double *Lp = L + (size_t)(i * NB + r0) + (size_t)(j * NB + tq) * ld;
      double t[2][32];
#pragma unroll
      for (int ks = 0; ks < 32; ks++) {                  // in flight while waiting for What_j
        t[0][ks] = Lp[(size_t)(4 * ks) * ld];
        t[1][ks] = Lp[(size_t)(4 * ks) * ld + 8];
      }
      __syncthreads();   // the previous step's readers of ws are done
      {
        const uint4 *pk = packets + (size_t)j * NB * KW;
        uint4 v[NP];
        bool ok;
        do {
          ok = true;
#pragma unroll
          for (int e = 0; e < NP; e++) v[e] = pk_load(pk + tid + NT * e);
#pragma unroll
          for (int e = 0; e < NP; e++) ok = ok && v[e].y == (unsigned)epoch && v[e].w == (unsigned)epoch;
        } while (!ok);
#pragma unroll
        for (int e = 0; e < NP; e++) {
          const int idx = tid + NT * e, q = idx >> 7, rr = idx & (NB - 1);     // packets are [q][row]
          ws[rr * WS + q] = __longlong_as_double((long long)(((unsigned long long)v[e].z << 32) | v[e].x));
        }
      }
      __syncthreads();
      if (j >= 1) {      // running sums before tile (i, j): the start of the row recurrence in k_gen_apply
        double *dp = Tdump + (size_t)tile_id(i, j) * kt * NB;
#pragma unroll
        for (int mb = 0; mb < 2; mb++)
#pragma unroll
          for (int nb = 0; nb < NN; nb++) {
            dp[(size_t)(8 * nb + 2 * tq) * NB + r0 + 8 * mb] = acc[mb][nb][0];
            dp[(size_t)(8 * nb + 2 * tq + 1) * NB + r0 + 8 * mb] = acc[mb][nb][1];
          }
      }
#pragma unroll
      for (int ks = 0; ks < 32; ks++) {
        const double *bp = ws + (size_t)(4 * ks + tq) * WS + g;
#pragma unroll
        for (int nb = 0; nb < NN; nb++) {
          const double bv = bp[8 * nb];
          dmma884(acc[0][nb][0], acc[0][nb][1], t[0][ks], bv);
          dmma884(acc[1][nb][0], acc[1][nb][1], t[1][ks], bv);
        }
      }
    }
    if (i >= 1) {
      double *dp = Tdump + (size_t)tile_id(i, i) * kt * NB;
#pragma unroll
      for (int mb = 0; mb < 2; mb++)
#pragma unroll
        for (int nb = 0; nb < NN; nb++) {
          dp[(size_t)(8 * nb + 2 * tq) * NB + r0 + 8 * mb] = acc[mb][nb][0];
          dp[(size_t)(8 * nb + 2 * tq + 1) * NB + r0 + 8 * mb] = acc[mb][nb][1];
        }
    }
    __syncthreads();     // rs of this CTA's previous block row is no longer read
#pragma unroll
    for (int mb = 0; mb < 2; mb++)
#pragma unroll
      for (int nb = 0; nb < NN; nb++)
#pragma unroll
        for (int e = 0; e < 2; e++) {
          const int q = 8 * nb + 2 * tq + e, rr = r0 + 8 * mb;
          const double wv = (q < k) ? W[(size_t)(i * NB + rr) + (size_t)q * ldw] : 0.0;
          rs[rr * WS + q] = wv - acc[mb][nb][e];
        }
    __syncthreads();
    {   // What_i = inv(L_ii) rs   (Xs lower triangular: columns beyond the warp's last row contribute nothing)
      double y[2][NN][2];
#pragma unroll
      for (int mb = 0; mb < 2; mb++)
#pragma unroll
        for (int nb = 0; nb < NN; nb++) y[mb][nb][0] = y[mb][nb][1] = 0.0;
      const int ksmax = 4 * warp + 4;
#pragma unroll 4
      for (int ks = 0; ks < ksmax; ks++) {
        const double a0 = Xs[r0 + XLD * (4 * ks + tq)], a1 = Xs[r0 + 8 + XLD * (4 * ks + tq)];
        const double *bp = rs + (size_t)(4 * ks + tq) * WS + g;
#pragma unroll
        for (int nb = 0; nb < NN; nb++) {
          const double bv = bp[8 * nb];
          dmma884(y[0][nb][0], y[0][nb][1], a0, bv);
          dmma884(y[1][nb][0], y[1][nb][1], a1, bv);
        }
      }
      uint4 *pk = packets + (size_t)i * NB * KW;
#pragma unroll
      for (int mb = 0; mb < 2; mb++)
#pragma unroll
        for (int nb = 0; nb < NN; nb++)
#pragma unroll
          for (int e = 0; e < 2; e++) {
            const int q = 8 * nb + 2 * tq + e, rr = r0 + 8 * mb;
            pk_store(pk + (size_t)q * NB + rr, y[mb][nb][e], epoch);                 // for the CTAs below
            What[(size_t)q * npad + (size_t)i * NB + rr] = y[mb][nb][e];
          }
    }
    __syncthreads();   // Xs / rs are reused by the next block row of this CTA
  }
}

// G[B] = What_B' What_B for the 32-row block B (KW x KW, row-major)
template <int KW>
__global__ void __launch_bounds__(256) k_gen_gram(const double *__restrict__ What, int npad, double *G) {
  __shared__ double wb[GB][KW + 1];
  const int B = blockIdx.x, tid = threadIdx.x;
  for (int idx = tid; idx < GB * KW; idx += 256) { const int p = idx & (GB - 1), q = idx >> 5; wb[p][q] = What[(size_t)q * npad + (size_t)B * GB + p]; }
  __syncthreads();
  for (int idx = tid; idx < KW * KW; idx += 256) {
    const int a = idx / KW, b = idx - a * KW;
    double s = 0.0;
#pragma unroll 8
    for (int p = 0; p < GB; p++) s = fma(wb[p][a], wb[p][b], s);
    G[(size_t)B * KW * KW + idx] = s;
  }
}

// in place: G[B] <- S + sum_{B' < B} G[B']   (S = diag(+1 x kpos, -1 x (k - kpos), +1 pad)).  Two-level scan inside one CTA per 64
// matrix entries: 16 threads per entry, each scans a contiguous chunk of blocks (its loads are independent and all in flight),
// the chunk totals meet in shared memory.  (One thread per entry walking all npad / 32 blocks: 41 us at n = 8000.)  The
// summation order is fixed by the chunking (chunk sums, then their prefix), so results are reproducible.
constexpr int SCAN_E = 64, SCAN_C = 16;
template <int KW>
__global__ void __launch_bounds__(SCAN_E * SCAN_C) k_gen_scan(double *G, int nblocks, int k, int kpos) {
  __shared__ double tot[SCAN_C][SCAN_E + 1];
  const int el = threadIdx.x % SCAN_E, ch = threadIdx.x / SCAN_E;
  const int idx = (int)blockIdx.x * SCAN_E + el, a = idx / KW, b = idx - a * KW;
  const int per = (nblocks + SCAN_C - 1) / SCAN_C, B0 = ch * per, B1 = min(nblocks, B0 + per);
  double sum = 0.0;
  for (int B = B0; B < B1; B += 8) {
    double v[8];
#pragma unroll
    for (int u = 0; u < 8; u++) v[u] = (B + u < B1) ? G[(size_t)(B + u) * KW * KW + idx] : 0.0;
#pragma unroll
    for (int u = 0; u < 8; u++) sum += v[u];
  }
  tot[ch][el] = sum;
  __syncthreads();
  double run = (a == b) ? ((a < kpos || a >= k) ? 1.0 : -1.0) : 0.0;
  for (int c = 0; c < ch; c++) run += tot[c][el];
  for (int B = B0; B < B1; B += 8) {
    double v[8];
#pragma unroll
    for (int u = 0; u < 8; u++) v[u] = (B + u < B1) ? G[(size_t)(B + u) * KW * KW + idx] : 0.0;
#pragma unroll
    for (int u = 0; u < 8; u++) if (B + u < B1) { G[(size_t)(B + u) * KW * KW + idx] = run; run += v[u]; }
  }
}

// one warp per 32-row block: P = inv(M_B) by Gauss-Jordan (lane = row, no pivoting: M_B is positive definite for an
// update, quasi-definite with the positive block first for a mixed pass), then per row j of the block
//   g = P what_j,  d_j = sqrt(1 + what_j' g),  z_j = g / d_j,  P <- P - z_j z_j'.
template <int KW>
__global__ void __launch_bounds__(32) k_gen_rows(const double *__restrict__ What, int npad, const double *__restrict__ Mpre,
                                                 double *D, double *Z, int *info) {
  __shared__ double wb[GB][KW + 1];
  const int B = blockIdx.x, lane = threadIdx.x, a = lane % KW;
  for (int idx = lane; idx < GB * KW; idx += 32) { const int p = idx & (GB - 1), q = idx >> 5; wb[p][q] = What[(size_t)q * npad + (size_t)B * GB + p]; }
  double m[KW], p[KW];
#pragma unroll
  for (int c = 0; c < KW; c++) { m[c] = Mpre[(size_t)B * KW * KW + a * KW + c]; p[c] = (c == a) ? 1.0 : 0.0; }
  __syncwarp();
  bool bad = false;
#pragma unroll
  for (int pv = 0; pv < KW; pv++) {
    const double mpp = __shfl_sync(0xffffffffu, m[pv], pv);
    if (!(fabs(mpp) > 0.0)) bad = true;
    const double inv = 1.0 / mpp;
    const double f = (a == pv) ? 0.0 : m[pv] * inv;
#pragma unroll
    for (int c = 0; c < KW; c++) {
      const double mr = __shfl_sync(0xffffffffu, m[c], pv), pr = __shfl_sync(0xffffffffu, p[c], pv);
      m[c] = fma(-f, mr, m[c]);
      p[c] = fma(-f, pr, p[c]);
      if (a == pv) { m[c] *= inv; p[c] *= inv; }
    }
  }
#pragma unroll 1
  for (int jj = 0; jj < GB; jj++) {
    double g0 = 0.0, g1 = 0.0, g2 = 0.0, g3 = 0.0;
#pragma unroll
    for (int c = 0; c < KW; c += 4) {
      g0 = fma(p[c], wb[jj][c], g0); g1 = fma(p[c + 1], wb[jj][c + 1], g1);
      g2 = fma(p[c + 2], wb[jj][c + 2], g2); g3 = fma(p[c + 3], wb[jj][c + 3], g3);
    }
    const double g = (g0 + g1) + (g2 + g3);
    double s = (lane < KW) ? wb[jj][a] * g : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const double d2 = 1.0 + s;
    if (!(d2 > 0.0)) bad = true;
    double d, rd;
    chol32::sqrt_and_rcp(d2, d, rd);       // branch-free correctly rounded sqrt and its reciprocal (no slow-path calls on the chain)
    const double z = g * rd;
#pragma unroll
    for (int c = 0; c < KW; c++) p[c] = fma(-z, __shfl_sync(0xffffffffu, z, c), p[c]);
    const size_t row = (size_t)B * GB + jj;
    if (lane == 0) D[row] = d;
    if (lane < KW) Z[(size_t)a * npad + row] = z;
  }
  if (bad && lane == 0) atomicExch(info, 1 + B * GB);
}

template <int KW> struct ApplySmem {
  static constexpr int WS = KW + 2;
  static constexpr size_t bytes = sizeof(double) * (2 * (size_t)NB * WS + NB);
};

// tile (I, J) of L, one thread per row:  t -= l what_j;  l_new = d_j l + t' z_j  for the tile's columns in order
template <int KW>
__global__ void __launch_bounds__(NB) k_gen_apply(double *L, int ld, const double *__restrict__ W, int ldw, int k,
                                                  const double *__restrict__ What, const double *__restrict__ Z,
                                                  const double *__restrict__ D, int npad, const double *__restrict__ Tdump) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int WS = ApplySmem<KW>::WS;
  double *ws = reinterpret_cast<double *>(smem_raw), *zs = ws + NB * WS, *ds = zs + NB * WS;
  // blockIdx.x -> (I, J), J <= I
  const int bid = blockIdx.x;
  int I = (int)((sqrtf(8.0f * (float)bid + 1.0f) - 1.0f) * 0.5f);
  while ((long long)(I + 1) * (I + 2) / 2 <= bid) I++;
  while ((long long)I * (I + 1) / 2 > bid) I--;
  const int J = bid - I * (I + 1) / 2;
  const int r = threadIdx.x;
  for (int idx = r; idx < NB * KW; idx += NB) {
    const int jj = idx & (NB - 1), q = idx >> 7;
    ws[jj * WS + q] = What[(size_t)q * npad + (size_t)J * NB + jj];
    zs[jj * WS + q] = Z[(size_t)q * npad + (size_t)J * NB + jj];
  }
  ds[r] = D[(size_t)J * NB + r];
  const size_t row = (size_t)I * NB + r;
  double t[KW];
#pragma unroll
  for (int q = 0; q < KW; q++) {
    const double wv = (q < k) ? W[row + (size_t)q * ldw] : 0.0;
    const double sv = (J >= 1) ? Tdump[((size_t)tile_id(I, J) * KW + q) * NB + r] : 0.0;
    t[q] = wv - sv;
  }
  __syncthreads();
  const int jmax = (I == J) ? r : NB - 1;
  double *Lp = L + row + (size_t)(J * NB) * ld;
  for (int j0 = 0; j0 <= jmax; j0 += 8) {
    double lv[8];
#pragma unroll
    for (int u = 0; u < 8; u++) lv[u] = (j0 + u <= jmax) ? Lp[(size_t)(j0 + u) * ld] : 0.0;
#pragma unroll
    for (int u = 0; u < 8; u++) {
      const int j = j0 + u;
      const double2 *w2 = reinterpret_cast<const double2 *>(ws + (size_t)j * WS);
      const double2 *z2 = reinterpret_cast<const double2 *>(zs + (size_t)j * WS);
      double o0 = ds[j] * lv[u], o1 = 0.0;
#pragma unroll
      for (int q = 0; q < KW; q += 2) {
        const double2 wv = w2[q >> 1], zv = z2[q >> 1];
        t[q] = fma(-lv[u], wv.x, t[q]);
        t[q + 1] = fma(-lv[u], wv.y, t[q + 1]);
        o0 = fma(t[q], zv.x, o0);
        o1 = fma(t[q + 1], zv.y, o1);
      }
      lv[u] = o0 + o1;
    }
#pragma unroll
    for (int u = 0; u < 8; u++) if (j0 + u <= jmax) Lp[(size_t)(j0 + u) * ld] = lv[u];
  }
}

struct State {
  uint4 *packets = nullptr;
  double *buf = nullptr;        // What | Z | D | G
  double *tdump = nullptr;
  int cap_npad = 0, epoch = 0, max_grid[3] = {0, 0, 0};
};
static std::mutex g_mu;
static std::map<cudaStream_t, State> g_state;
// test hooks (host only, no kernel reads them): the per-group grid of this thread's last k_fwd_multi launch and the limit it
// was launched under, and a cap on that limit.  The cap applies to gmax, never to max_grid: a max_grid below NS would mark the
// pass unavailable on the stream for good.  0: no cap (the default; only qpalm_b200_dense_probe_updown sets one).
static thread_local int g_last_grid = 0, g_last_gmax = 0, g_grid_cap = 0;

template <int KT, int KW>     // KT columns per pass, solved as KT / KW independent groups
static int run(cudaStream_t s, State &st, int slot, int npad, double *L, int ld, const double *X, const double *W, int ldw, int k, int kpos,
               int *info_dev) {
  constexpr int NS = KT / KW;
  if (st.max_grid[slot] == 0) {
    int dev = 0, coop = 0, sms = 0, per_sm = 0;
    QB_CUDA_TRY(cudaGetDevice(&dev));
    QB_CUDA_TRY(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
    QB_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    QB_CUDA_TRY(cudaFuncSetAttribute(k_fwd_multi<KW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FwdSmem<KW>::bytes));
    QB_CUDA_TRY(cudaFuncSetAttribute(k_gen_apply<KT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ApplySmem<KT>::bytes));
    QB_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_fwd_multi<KW>, NT, FwdSmem<KW>::bytes));
    st.max_grid[slot] = (coop && per_sm > 0) ? sms * per_sm : -1;
  }
  if (st.max_grid[slot] < NS) return 1;
  const int nblk = npad / NB, nblocks = npad / GB;
  double *What = st.buf, *Z = What + (size_t)npad * 32, *D = Z + (size_t)npad * 32, *G = D + npad;
  {
    const int gmax = (g_grid_cap > 0 && g_grid_cap < st.max_grid[slot] / NS) ? g_grid_cap : st.max_grid[slot] / NS;
    const int grid = nblk < gmax ? nblk : gmax;
    int ld_a = ld, ldw_a = ldw, k_a = k, npad_a = npad, nblk_a = nblk, epoch = st.epoch, kt = KT;
    uint4 *pk = st.packets;
    double *td = st.tdump;
    void *args[] = {(void *)&L, (void *)&ld_a, (void *)&X, (void *)&W, (void *)&ldw_a, (void *)&k_a, (void *)&What, (void *)&npad_a,
                    (void *)&td, (void *)&nblk_a, (void *)&pk, (void *)&epoch, (void *)&kt};
    const bool prof = g_prof_on && prof_begin("udgen::k_fwd_multi", s);
    const cudaError_t err = cudaLaunchCooperativeKernel((const void *)k_fwd_multi<KW>, dim3(grid, NS), dim3(NT), args, FwdSmem<KW>::bytes, s);
    if (prof) prof_end(s);
    if (err != cudaSuccess) { (void)cudaGetLastError(); st.max_grid[slot] = -1; return 1; }
    ++g_kernel_launches;
    g_last_grid = grid; g_last_gmax = gmax;
  }
  QB_LAUNCH(k_gen_gram<KT>, nblocks, 256, 0, s, What, npad, G);
  QB_LAUNCH(k_gen_scan<KT>, KT * KT / SCAN_E, SCAN_E * SCAN_C, 0, s, G, nblocks, k, kpos);
  QB_LAUNCH(k_gen_rows<KT>, nblocks, 32, 0, s, What, npad, G, D, Z, info_dev);
  const int ntile = nblk * (nblk + 1) / 2;
  QB_LAUNCH(k_gen_apply<KT>, ntile, NB, ApplySmem<KT>::bytes, s, L, ld, W, ldw, k, What, Z, D, npad, st.tdump);
  QB_CUDA_TRY(cudaGetLastError());
  return 0;
}
}  // namespace udgen

int chol_updown_gen_max_rank() { return 32; }

// returns 0 when the pass ran, 1 when the cooperative kernel is not available on this device / partition or the pass's work
// space cannot be allocated (the caller uses the per-panel launches), < 0 on a CUDA error.  invdiag must hold the inverses of the
// diagonal blocks of the CURRENT L; the caller refreshes it afterwards (trtri_diag_blocks).
int chol_updown_gen(cudaStream_t s, int npad, double *L, int ld, const double *invdiag, const double *W, int ldw, int k, int kpos,
                    int *info_dev) {
  using namespace udgen;
  g_last_grid = g_last_gmax = 0;
  if (k <= 0) return 0;
  if (k > 32 || (npad % NB)) return 1;
  std::lock_guard<std::mutex> lk(g_mu);
  State &st = g_state[s];
  if (st.cap_npad < npad) {
    if (st.packets) QB_CUDA_TRY(cudaFree(st.packets));
    if (st.buf) QB_CUDA_TRY(cudaFree(st.buf));
    if (st.tdump) QB_CUDA_TRY(cudaFree(st.tdump));
    st.packets = nullptr; st.buf = nullptr; st.tdump = nullptr; st.cap_npad = 0;
    const size_t nblk = (size_t)npad / NB, nblocks = (size_t)npad / GB;
    // work space of a pass: 16 B x 32 per row of packets, 65 doubles per row of What | Z | D, the Gram prefixes and the running sums of
    // every tile (n = 8000: 66 MB; n = 30 000: 0.9 GB).  If HBM cannot hold it the caller takes the per-panel kernels, which need none.
    const cudaError_t e1 = cudaMalloc(&st.packets, sizeof(uint4) * (size_t)npad * 32);
    const cudaError_t e2 = e1 == cudaSuccess ? cudaMalloc(&st.buf, sizeof(double) * ((size_t)npad * 65 + nblocks * 32 * 32)) : e1;
    const cudaError_t e3 = e2 == cudaSuccess ? cudaMalloc(&st.tdump, sizeof(double) * (nblk * (nblk + 1) / 2) * NB * 32) : e2;
    if (e3 != cudaSuccess) {
      (void)cudaGetLastError();
      if (st.packets) cudaFree(st.packets);
      if (st.buf) cudaFree(st.buf);
      st.packets = nullptr; st.buf = nullptr; st.tdump = nullptr;
      return 1;
    }
    QB_CUDA_TRY(cudaMemsetAsync(st.packets, 0, sizeof(uint4) * (size_t)npad * 32, s));
    st.cap_npad = npad;
    st.epoch = 0;
  }
  st.epoch++;
  if (k <= 8) return run<8, 8>(s, st, 0, npad, L, ld, invdiag, W, ldw, k, kpos, info_dev);
  if (k <= 16) return run<16, 8>(s, st, 1, npad, L, ld, invdiag, W, ldw, k, kpos, info_dev);
  return run<32, 16>(s, st, 2, npad, L, ld, invdiag, W, ldw, k, kpos, info_dev);
}

int chol_updown_gen_last_grid(int *gmax) {
  if (gmax) *gmax = udgen::g_last_gmax;
  return udgen::g_last_grid;
}
void chol_updown_gen_set_grid_cap(int cap) { udgen::g_grid_cap = cap > 0 ? cap : 0; }

const double *chol_updown_gen_workspace(cudaStream_t s) {
  std::lock_guard<std::mutex> lk(udgen::g_mu);
  auto it = udgen::g_state.find(s);
  return it == udgen::g_state.end() ? nullptr : it->second.buf;
}

void chol_updown_gen_release(cudaStream_t s) {
  std::lock_guard<std::mutex> lk(udgen::g_mu);
  auto it = udgen::g_state.find(s);
  if (it == udgen::g_state.end()) return;
  if (it->second.packets) cudaFree(it->second.packets);
  if (it->second.buf) cudaFree(it->second.buf);
  if (it->second.tdump) cudaFree(it->second.tdump);
  udgen::g_state.erase(it);
}

}  // namespace qb
