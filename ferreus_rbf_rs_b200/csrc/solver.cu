// fr_model: device-resident RBF solve (FGMRES + multilevel Schwarz DDM) and interpolant evaluation.
//   fgmres / schwarz_ddm_solver     ferreus_rbf/src/iterative_solvers.rs:38-281
//   schwarz_preconditioner           ferreus_rbf/src/preconditioning/schwarz.rs:32-155
//   Domain::factorise / solve        ferreus_rbf/src/domain.rs:153-467 (device part: Q^T A Q assembly, Cholesky,
//                                    triangular solves; the packed RFP storage of linalg.rs is replaced by a
//                                    full row-major square per domain, only the lower triangle is streamed)
//   fast_matrix_vector_product       ferreus_rbf/src/rbf.rs:1338-1379
//   RBFInterpolator fit / evaluate   ferreus_rbf/src/rbf.rs:317-582, 676-924, 1180-1270
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <memory>

#include "fmm.h"
#include "isosurface.h"
#include "solver_host.h"

namespace fb {

static inline unsigned nblk(size_t n, int bs) { return (unsigned)((n + bs - 1) / bs); }

// ------------------------------------------------------------------------------------ vector kernels
__global__ void k_dot(const double *a, const double *b, size_t n, double *out) {
  __shared__ double red[32];
  double s = 0;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) s += a[i] * b[i];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    s = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0;
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if (threadIdx.x == 0) atomicAdd(out, s);
  }
}

__global__ void k_absmax(const double *a, size_t n, unsigned long long *out) {
  double s = 0;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) s = fmax(s, fabs(a[i]));
  for (int o = 16; o > 0; o >>= 1) s = fmax(s, __shfl_down_sync(0xffffffffu, s, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out, (unsigned long long)__double_as_longlong(s));  // non-negative doubles order as integers
}

__global__ void k_axpy(double a, const double *x, double *y, size_t n) {  // y += a x
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i < n) y[i] += a * x[i];
}

__global__ void k_scale_to(double a, const double *x, double *y, size_t n) {  // y = a x
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i < n) y[i] = a * x[i];
}

__global__ void k_sub_to(const double *a, const double *b, double *y, size_t n) {  // y = a - b
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i < n) y[i] = a[i] - b[i];
}

// y[row] = fmm[i] + nugget * w[row] + P[row, :] . w[n:]   for row = idx[i] (or i); other rows stay zero
__global__ void k_matvec_finish(const double *fmm, const unsigned long long *idx, size_t cnt, const double *w, size_t n,
                                int m, const double *P, double nugget, double *y) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= cnt) return;
  const size_t row = idx ? (size_t)idx[i] : i;
  double v = fmm[i] + nugget * w[row];
  for (int k = 0; k < m; ++k) v += P[row * m + k] * w[n + k];
  y[row] = v;
}

// s1[:n] -= Q (Q^T s1[:n]):  first the m projections, then the update (schwarz.rs:122-126)
__global__ void k_project_dots(const double *Q, const double *v, size_t n, int m, double *out) {
  __shared__ double red[32];
  for (int k = 0; k < m; ++k) {
    double s = 0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) s += Q[i * m + k] * v[i];
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
      s = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0;
      for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
      if (threadIdx.x == 0) atomicAdd(out + k, s);
    }
    __syncthreads();
  }
}

__global__ void k_project_apply(const double *Q, const double *coef, size_t n, int m, double *v) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  double s = 0;
  for (int k = 0; k < m; ++k) s += Q[i * m + k] * coef[k];
  v[i] -= s;
}

// ------------------------------------------------------------------------------------ domain kernels
struct DomainTable {  // one DDM level on the device
  int n_domains = 0;
  const long long *pt_ptr;   // n_domains+1 into pt_idx / pt_mask
  const int *pt_idx;         // global point index, special points first
  const uint8_t *pt_mask;    // internal flag
  const int *rank;           // special points per domain
  const long long *q_off;    // offset of Q_top (rank x mm, row-major) in the q pool
  const long long *l_off;    // offset of the mm x mm factor in the factor pool
  const long long *s_off;    // offset of the 2 x rank x mm assembly scratch (A12, C)
  const uint8_t *use_inverse;  // per domain: the factor slot holds the explicit inverse (indefinite Q^T A Q), or null
};

__device__ __forceinline__ double kval_rt(double r2, const KParams &kp) {
  switch (kp.fam) {
    case KF_LINEAR: return kernel_value<KF_LINEAR>(r2, kp);
    case KF_TPS: return kernel_value<KF_TPS>(r2, kp);
    case KF_CUBIC: return kernel_value<KF_CUBIC>(r2, kp);
    case KF_SPH: return kernel_value<KF_SPH>(r2, kp);
    case KF_LAPLACE: return kernel_value<KF_LAPLACE>(r2, kp);
    case KF_R2: return kernel_value<KF_R2>(r2, kp);
    default: return kernel_value<KF_R4>(r2, kp);
  }
}

__device__ __forceinline__ double pair_r2(const double *px, const double *py, const double *pz, int a, int b) {
  const double dx = px[a] - px[b], dy = py[a] - py[b], dz = pz[a] - pz[b];
  double r2 = dx * dx;
  r2 += dy * dy;
  r2 += dz * dz;
  return r2;
}

// scratch rows for the Q^T A Q assembly: A12[a][j] = k(s_a, x_j) and C[a][j] = A12[a][j] + sum_b A11[a][b] Q[b][j]
__global__ void k_dom_prep(DomainTable t, const double *px, const double *py, const double *pz, KParams kp,
                           double nugget, const double *qpool, double *scratch) {
  const int d = blockIdx.x;
  const int rk = t.rank[d];
  if (rk == 0) return;
  const long long p0 = t.pt_ptr[d];
  const int n = (int)(t.pt_ptr[d + 1] - p0), mm = n - rk;
  const int *idx = t.pt_idx + p0;
  const double *Q = qpool + t.q_off[d];
  double *A12 = scratch + t.s_off[d], *C = A12 + (size_t)rk * mm;
  __shared__ double A11[16][16];
  for (int e = threadIdx.x; e < rk * rk; e += blockDim.x) {
    const int a = e / rk, b = e % rk;
    A11[a][b] = kval_rt(pair_r2(px, py, pz, idx[a], idx[b]), kp) + (a == b ? nugget : 0.0);
  }
  __syncthreads();
  for (int j = threadIdx.x; j < mm; j += blockDim.x) {
    double a12[16];
    for (int a = 0; a < rk; ++a) {
      a12[a] = kval_rt(pair_r2(px, py, pz, idx[a], idx[rk + j]), kp);
      A12[(size_t)a * mm + j] = a12[a];
    }
    for (int a = 0; a < rk; ++a) {
      double c = a12[a];
      for (int b = 0; b < rk; ++b) c += A11[a][b] * Q[(size_t)b * mm + j];
      C[(size_t)a * mm + j] = c;
    }
  }
}

// lower triangle of  Q^T A Q = A22 + Q^T (A12 + A11 Q) + A21 Q   (domain.rs:322-356), 32 x 32 tiles
__global__ void __launch_bounds__(256) k_dom_assemble(DomainTable t, const double *px, const double *py,
                                                      const double *pz, KParams kp, double nugget,
                                                      const double *qpool, const double *scratch, double *lpool) {
  const int d = blockIdx.z;
  const int rk = t.rank[d];
  const long long p0 = t.pt_ptr[d];
  const int n = (int)(t.pt_ptr[d + 1] - p0), mm = n - rk;
  const int ti = blockIdx.y, tj = blockIdx.x;
  if (tj > ti || ti * 32 >= mm) return;
  const int *idx = t.pt_idx + p0 + rk;
  const double *Q = qpool + t.q_off[d];
  const double *A12 = scratch + t.s_off[d], *C = A12 + (size_t)rk * mm;
  double *L = lpool + t.l_off[d];
  __shared__ double xi[3][32], xj[3][32];
  __shared__ double Qi[16][32], Ai[16][32], Qj[16][32], Cj[16][32];
  const int tid = threadIdx.x;
  if (tid < 32) {
    const int i = ti * 32 + tid;
    const int g = i < mm ? idx[i] : idx[0];
    xi[0][tid] = px[g]; xi[1][tid] = py[g]; xi[2][tid] = pz[g];
  } else if (tid < 64) {
    const int j = tj * 32 + tid - 32;
    const int g = j < mm ? idx[j] : idx[0];
    xj[0][tid - 32] = px[g]; xj[1][tid - 32] = py[g]; xj[2][tid - 32] = pz[g];
  }
  for (int e = tid; e < rk * 32; e += 256) {
    const int a = e / 32, c = e % 32;
    const int i = ti * 32 + c, j = tj * 32 + c;
    Qi[a][c] = i < mm ? Q[(size_t)a * mm + i] : 0.0;
    Ai[a][c] = i < mm ? A12[(size_t)a * mm + i] : 0.0;
    Qj[a][c] = j < mm ? Q[(size_t)a * mm + j] : 0.0;
    Cj[a][c] = j < mm ? C[(size_t)a * mm + j] : 0.0;
  }
  __syncthreads();
  const int c = tid & 31;
  for (int r = tid >> 5; r < 32; r += 8) {
    const int i = ti * 32 + r, j = tj * 32 + c;
    if (i >= mm || j >= mm || j > i) continue;
    const double dx = xi[0][r] - xj[0][c], dy = xi[1][r] - xj[1][c], dz = xi[2][r] - xj[2][c];
    double r2 = dx * dx;
    r2 += dy * dy;
    r2 += dz * dz;
    double v = kval_rt(r2, kp) + (i == j ? nugget : 0.0);
    for (int a = 0; a < rk; ++a) v += Qi[a][r] * Cj[a][c] + Ai[a][r] * Qj[a][c];
    L[(size_t)i * mm + j] = v;
  }
}

constexpr int kNB = 32;
constexpr int kPS = kNB + 4;
__device__ __forceinline__ void chol_dmma884(double &d0, double &d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}
// diagonal block kb (Cholesky by warp 0 in shared memory) and the panel below it (one thread per row):
//   L[i, kb:kb+bs] = A[i, kb:kb+bs] Dk^-T
__device__ __forceinline__ void chol_factor_panel(double *A, int n, int kb, int bs, double (*Dk)[kNB + 1],
                                                  uint8_t *fail, int dom) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int e = tid; e < kNB * kNB; e += 256) {
    const int r = e / kNB, c = e % kNB;
    Dk[r][c] = (r < bs && c <= r) ? A[(size_t)(kb + r) * n + kb + c] : (r == c ? 1.0 : 0.0);
  }
  __syncthreads();
  if (warp == 0) {
    for (int k = 0; k < bs; ++k) {
      double dkk = Dk[k][k];
      if (lane == 0 && !(dkk > 0.0)) fail[dom] = 1;
      dkk = sqrt(fmax(dkk, 1e-300));
      __syncwarp();
      if (lane == k) Dk[k][k] = dkk;
      if (lane > k && lane < bs) Dk[lane][k] /= dkk;
      __syncwarp();
      if (lane > k && lane < bs) {
        const double lk = Dk[lane][k];
        for (int c = k + 1; c <= lane; ++c) Dk[lane][c] -= lk * Dk[c][k];
      }
      __syncwarp();
    }
  }
  __syncthreads();
  for (int e = tid; e < bs * bs; e += 256) {
    const int r = e / bs, c = e % bs;
    if (c <= r) A[(size_t)(kb + r) * n + kb + c] = Dk[r][c];
  }
  for (int i = kb + bs + tid; i < n; i += 256) {
    double x[kNB];
    double *row = A + (size_t)i * n + kb;
#pragma unroll
    for (int c = 0; c < kNB; ++c) x[c] = c < bs ? row[c] : 0.0;
#pragma unroll
    for (int c = 0; c < kNB; ++c) {
      if (c < bs) {
        double v = x[c];
#pragma unroll
        for (int k = 0; k < c; ++k) v -= x[k] * Dk[c][k];
        x[c] = v / Dk[c][c];
      }
    }
#pragma unroll
    for (int c = 0; c < kNB; ++c)
      if (c < bs) row[c] = x[c];
  }
}

// trailing update of the tile column jb: A[ib.., jb..] -= P_i P_j^T for the lower tiles ib = ib_first, + ib_step, ...
// (this warp's tiles); the whole CTA stages the j panel tile, every warp its own i panel tile.  C = P Pj^T runs on the
// FP64 tensor cores: 4 x 4 tiles of m8n8k4, 8 k-steps (1.6x the FMA version on the 2048-domain level).
__device__ __forceinline__ void chol_update_column(double *A, int n, int kb, int bs, int jb, double (*Pj)[kPS],
                                                   double (*Pi)[kPS], int ib_first, int ib_step) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int bj = min(kNB, n - jb);
  __syncthreads();
  for (int e = tid; e < kNB * kNB; e += 256) {
    const int r = e / kNB, c = e % kNB;
    Pj[r][c] = (r < bj && c < bs) ? A[(size_t)(jb + r) * n + kb + c] : 0.0;
  }
  __syncthreads();
  for (int ib = ib_first; ib < n; ib += ib_step) {
    const int bi = min(kNB, n - ib);
    double(*P)[kPS] = Pi + warp * kNB;
    for (int r = 0; r < kNB; ++r) P[r][lane] = (r < bi && lane < bs) ? A[(size_t)(ib + r) * n + kb + lane] : 0.0;
    __syncwarp();
    const int g = lane >> 2, t4 = lane & 3;
    double c[4][4][2];
#pragma unroll
    for (int a4 = 0; a4 < 4; ++a4)
#pragma unroll
      for (int b4 = 0; b4 < 4; ++b4) c[a4][b4][0] = c[a4][b4][1] = 0.0;
#pragma unroll 2
    for (int ks = 0; ks < kNB / 4; ++ks) {
      double fa[4], fb4[4];
#pragma unroll
      for (int a4 = 0; a4 < 4; ++a4) fa[a4] = P[8 * a4 + g][4 * ks + t4];
#pragma unroll
      for (int b4 = 0; b4 < 4; ++b4) fb4[b4] = Pj[8 * b4 + g][4 * ks + t4];
#pragma unroll
      for (int a4 = 0; a4 < 4; ++a4)
#pragma unroll
        for (int b4 = 0; b4 < 4; ++b4) chol_dmma884(c[a4][b4][0], c[a4][b4][1], fa[a4], fb4[b4]);
    }
#pragma unroll
    for (int a4 = 0; a4 < 4; ++a4) {
      const int r = 8 * a4 + g;
      if (r >= bi) continue;
      double *row = A + (size_t)(ib + r) * n + jb;
#pragma unroll
      for (int b4 = 0; b4 < 4; ++b4)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int cc = 8 * b4 + 2 * t4 + h;
          if (cc < bj && ib + r >= jb + cc) row[cc] -= c[a4][b4][h];  // lower triangle only
        }
    }
    __syncwarp();
  }
}

#define FB_CHOL_SMEM_VIEWS                                                                                          \
  extern __shared__ double sm[];                                                                                    \
  double(*Dk)[kNB + 1] = reinterpret_cast<double(*)[kNB + 1]>(sm);                       /* diagonal block */       \
  /* panel tiles feed DMMA fragments: row stride kPS == 4 (mod 16): conflict-free fragment loads per half-warp */   \
  double(*Pj)[kPS] = reinterpret_cast<double(*)[kPS]>(sm + kNB * (kNB + 1));              /* j panel tile */         \
  double(*Pi)[kPS] = reinterpret_cast<double(*)[kPS]>(sm + kNB * (kNB + 1) + kNB * kPS);  /* 8 warps x i panel tile */

// blocked right-looking Cholesky, one CTA per domain, lower triangle of a row-major mm x mm matrix in place
__global__ void __launch_bounds__(256) k_cholesky(DomainTable t, double *lpool, uint8_t *fail) {
  const int d = blockIdx.x;
  const int n = (int)(t.pt_ptr[d + 1] - t.pt_ptr[d]) - t.rank[d];
  double *A = lpool + t.l_off[d];
  FB_CHOL_SMEM_VIEWS
  const int warp = threadIdx.x >> 5;
  for (int kb = 0; kb < n; kb += kNB) {
    const int bs = min(kNB, n - kb);
    chol_factor_panel(A, n, kb, bs, Dk, fail, d);
    __syncthreads();
    for (int jb = kb + bs; jb < n; jb += kNB) chol_update_column(A, n, kb, bs, jb, Pj, Pi, jb + warp * kNB, 8 * kNB);
    __syncthreads();
  }
}

// the same factorisation of ONE large matrix (the coarse domain) spread over the GPU: per block column one small
// launch for the diagonal block + panel and one grid for the trailing update
__global__ void __launch_bounds__(256) k_chol_big_panel(double *A, int n, int kb, uint8_t *fail) {
  extern __shared__ double sm[];
  chol_factor_panel(A, n, kb, min(kNB, n - kb), reinterpret_cast<double(*)[kNB + 1]>(sm), fail, 0);
}
__global__ void __launch_bounds__(256) k_chol_big_update(double *A, int n, int kb) {
  extern __shared__ double sm[];
  double(*Pj)[kPS] = reinterpret_cast<double(*)[kPS]>(sm + kNB * (kNB + 1));
  double(*Pi)[kPS] = reinterpret_cast<double(*)[kPS]>(sm + kNB * (kNB + 1) + kNB * kPS);
  const int bs = min(kNB, n - kb);
  const int jb = kb + bs + blockIdx.x * kNB;
  const int ib = jb + (blockIdx.y * 8 + (threadIdx.x >> 5)) * kNB;
  chol_update_column(A, n, kb, bs, jb, Pj, Pi, ib, n);  // at most one i tile per warp
}

// ---- Domain::solve (domain.rs:393-467) + scatter of schwarz.rs:94-155, one CTA of kSolveThreads threads per domain
//   mode 0: fine level — write internal points only;  mode 1: coarse — write all points (+ polynomial tail)
// The two substitutions are chains of 2 x mm / 32 dependent block steps over the lower triangle of L, streamed from HBM
// row block by row block.  What sits between the loads is kept off the critical path:
//   * the 32 x 32 diagonal blocks of L are inverted in place once, at setup (k_inv_diag_inplace), so a block step is a
//     32-lane dot product per row, all 32 warps at once, no division, no dependency chain;
//   * the forward substitution is left-looking: every row of the block has its own warp and four independent partial
//     sums per lane;
//   * the backward substitution is right-looking: as soon as the 32 values of a block are known, every thread subtracts
//     their contribution from ITS column of the right-hand side — 32 independent, row-contiguous loads per thread —
//     instead of walking a column block (256 B out of every 7.8 KB row).
constexpr int kSolveThreads = 1024;
constexpr int kSolveWarps = kSolveThreads / 32;

// A^-1 of the lower-triangular bs x bs block A (row stride ld, bs <= kNB) into the lower triangle of Ainv, which may be
// A itself; one warp, lane c forms column c by forward substitution.  The strict upper triangle of Ainv is not written.
__device__ __forceinline__ void tri_inv_block(const double *A, size_t ld, int bs, double *Ainv) {
  const int lane = threadIdx.x;
  __shared__ double D[kNB][kNB + 1];
  for (int r = 0; r < bs; ++r) D[r][lane] = (lane < bs && lane <= r) ? A[(size_t)r * ld + lane] : 0.0;
  __syncwarp();
  double x[kNB];
#pragma unroll
  for (int r = 0; r < kNB; ++r) x[r] = 0.0;
  if (lane < bs) {
#pragma unroll
    for (int r = 0; r < kNB; ++r) {
      if (r < bs && r >= lane) {
        double v = r == lane ? 1.0 : 0.0;
#pragma unroll
        for (int k = 0; k < kNB; ++k)
          if (k < r && k >= lane) v -= D[r][k] * x[k];
        x[r] = v / D[r][r];
      }
    }
  }
  // a lane reads and writes only its own column; this fence keeps ptxas from scheduling the stores into the
  // substitution, which takes the in-place kernel from 90 to 117 registers
  __syncwarp();
  if (lane < bs)
#pragma unroll
    for (int r = 0; r < kNB; ++r)
      if (r < bs && r >= lane) Ainv[(size_t)r * ld + lane] = x[r];
}

__global__ void k_inv_diag_inplace(DomainTable t, double *lpool) {
  const int d = blockIdx.x;
  const int mm = (int)(t.pt_ptr[d + 1] - t.pt_ptr[d]) - t.rank[d];
  const int kb = blockIdx.y * kNB;
  if (kb >= mm) return;
  double *blk = lpool + t.l_off[d] + (size_t)kb * mm + kb;
  tri_inv_block(blk, mm, min(kNB, mm - kb), blk);
}

// The end of Domain::solve (domain.rs:434-463) and its scatter, for one domain on one CTA of kSolveThreads threads:
// lambda = [Q gamma; gamma] goes to out[idx] (mode 1: every point; mode 0: the internal ones), and in mode 1 the
// polynomial tail follows: r = d_special - A_special lambda, poly = sp_mono^-1 r.  Every dot product is one warp per
// row, lane-strided, reduced with __shfl_down to lane 0.  d_special: the rk residuals at the special points; top and
// red: shared scratch of rk doubles each (red may be d_special itself: an entry is read before it is overwritten).
__device__ __forceinline__ void dom_solve_finish(const double *Q, const double *gamma, const double *d_special,
                                                 const int *idx, const uint8_t *mask, int n, int rk, int mode,
                                                 int add_poly, const double *a_special, const double *sp_inv,
                                                 size_t n_total, double *top, double *red, double *out) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int mm = n - rk;
  // lambda_top = Q gamma
  for (int a = warp; a < rk; a += kSolveWarps) {
    double sacc = 0.0;
    for (int j = lane; j < mm; j += 32) sacc += Q[(size_t)a * mm + j] * gamma[j];
    for (int o = 16; o > 0; o >>= 1) sacc += __shfl_down_sync(0xffffffffu, sacc, o);
    if (lane == 0) top[a] = sacc;
  }
  __syncthreads();
  for (int i = tid; i < n; i += kSolveThreads) {
    const double lam = i < rk ? top[i] : gamma[i - rk];
    if (mode == 1 || mask[i]) out[idx[i]] = lam;
  }
  if (mode == 1 && add_poly && rk > 0 && a_special) {
    __syncthreads();
    for (int a = warp; a < rk; a += kSolveWarps) {
      const double *row = a_special + (size_t)a * n;
      double sacc = 0.0;
      for (int i = lane; i < n; i += 32) sacc += row[i] * (i < rk ? top[i] : gamma[i - rk]);
      for (int o = 16; o > 0; o >>= 1) sacc += __shfl_down_sync(0xffffffffu, sacc, o);
      if (lane == 0) red[a] = d_special[a] - sacc;
    }
    __syncthreads();
    if (tid < rk) {
      double sacc = 0.0;
      for (int b = 0; b < rk; ++b) sacc += sp_inv[tid * rk + b] * red[b];
      out[n_total - rk + tid] = sacc;  // schwarz.rs:147-152: tail rows
    }
  }
}

__global__ void __launch_bounds__(kSolveThreads) k_dom_solve(DomainTable t, const double *qpool, const double *lpool,
                                                             const double *res, double *out, int mode, int add_poly,
                                                             const double *a_special, const double *sp_inv,
                                                             size_t n_total) {
  const int d = blockIdx.x;
  const int rk = t.rank[d];
  const long long p0 = t.pt_ptr[d];
  const int n = (int)(t.pt_ptr[d + 1] - p0), mm = n - rk;
  const int *idx = t.pt_idx + p0;
  const uint8_t *mask = t.pt_mask + p0;
  const double *Q = qpool + t.q_off[d];
  const double *L = lpool + t.l_off[d];
  extern __shared__ double sm[];
  double *dv = sm;        // n gathered residuals
  double *x = dv + n;     // mm rhs / solution
  double *red = x + mm;   // 32 partial sums
  double *top = red + kSolveWarps * 32;  // rk
  __shared__ double Dg[32][33];          // inverse of the diagonal block of the current step (lower triangle)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < n; i += kSolveThreads) dv[i] = res[idx[i]];
  __syncthreads();
  for (int j = tid; j < mm; j += kSolveThreads) {  // rhs = Q^T d_special + d_rest
    double v = dv[rk + j];
    for (int a = 0; a < rk; ++a) v += Q[(size_t)a * mm + j] * dv[a];
    x[j] = v;
  }
  __syncthreads();
  const bool inverse = t.use_inverse != nullptr && t.use_inverse[d] != 0;
  if (inverse) {
    // Cholesky failed for this domain (Q^T A Q indefinite; domain.rs:63-68 falls back to a pivoted factorisation): the
    // slot holds the explicit inverse, gamma = Inv rhs.  d_rest (dv[rk..n)) is dead once rhs is formed: it takes gamma
    for (int r = warp; r < mm; r += kSolveWarps) {
      const double *row = L + (size_t)r * mm;
      double sacc = 0.0;
      for (int c = lane; c < mm; c += 32) sacc += row[c] * x[c];
      for (int o = 16; o > 0; o >>= 1) sacc += __shfl_down_sync(0xffffffffu, sacc, o);
      if (lane == 0) dv[rk + r] = sacc;
    }
    __syncthreads();
    for (int j = tid; j < mm; j += kSolveThreads) x[j] = dv[rk + j];
    __syncthreads();
  }
  // forward substitution L y = rhs, left-looking: row r of the block belongs to warp r
  for (int kb = 0; !inverse && kb < mm; kb += 32) {
    const int bs = min(32, mm - kb);
    if (warp < bs) {
      const double *row = L + (size_t)(kb + warp) * mm;
      double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
      int c = lane;
      for (; c + 96 < kb; c += 128) {
        s0 += row[c] * x[c];
        s1 += row[c + 32] * x[c + 32];
        s2 += row[c + 64] * x[c + 64];
        s3 += row[c + 96] * x[c + 96];
      }
      for (; c < kb; c += 32) s0 += row[c] * x[c];
      Dg[warp][lane] = lane <= warp ? row[kb + lane] : 0.0;  // row `warp` of the inverted diagonal block
      double sacc = (s0 + s1) + (s2 + s3);
      for (int o = 16; o > 0; o >>= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, o);
      if (lane == 0) red[warp] = x[kb + warp] - sacc;
    }
    __syncthreads();
    if (warp < bs) {  // y_r = sum_k Dinv[r][k] (rhs_k - partial_k)
      double v = (lane <= warp) ? Dg[warp][lane] * red[lane] : 0.0;
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) x[kb + warp] = v;
    }
    __syncthreads();
  }
  // backward substitution L^T gamma = y, right-looking
  for (int kb = ((mm - 1) / 32) * 32; !inverse && kb >= 0; kb -= 32) {
    const int bs = min(32, mm - kb);
    if (warp < bs) Dg[warp][lane] = lane <= warp ? L[(size_t)(kb + warp) * mm + kb + lane] : 0.0;
    if (tid < 32) red[tid] = tid < bs ? x[kb + tid] : 0.0;
    __syncthreads();
    if (warp < bs) {  // gamma_r = sum_{k >= r} Dinv[k][r] y_k
      double v = (lane >= warp && lane < bs) ? Dg[lane][warp] * red[lane] : 0.0;
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) x[kb + warp] = v;
    }
    __syncthreads();
    for (int c = tid; c < kb; c += kSolveThreads) {  // y[c] -= sum_r L[kb + r][c] gamma[kb + r]
      const double *col = L + (size_t)kb * mm + c;
      double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
      int r = 0;
      for (; r + 3 < bs; r += 4) {
        a0 += col[(size_t)r * mm] * x[kb + r];
        a1 += col[(size_t)(r + 1) * mm] * x[kb + r + 1];
        a2 += col[(size_t)(r + 2) * mm] * x[kb + r + 2];
        a3 += col[(size_t)(r + 3) * mm] * x[kb + r + 3];
      }
      for (; r < bs; ++r) a0 += col[(size_t)r * mm] * x[kb + r];
      x[c] -= (a0 + a1) + (a2 + a3);
    }
    __syncthreads();
  }
  dom_solve_finish(Q, x, dv, idx, mask, n, rk, mode, add_poly, a_special, sp_inv, n_total, top, red, out);
}

// ---- the single coarse domain (n ~ 2000) -----------------------------------------------------------------------------
// One CTA per domain leaves the two substitutions of the coarse domain as chains of 2 x mm / 32 dependent steps on one SM:
// 3.5 ms for the coarse domain of the 1M-point fit with the first form of k_dom_solve (since removed), three times per
// preconditioner cycle.  For a one-domain level the triangular factor is inverted once at setup (X = L^-1, kept with its
// transpose), and Domain::solve becomes two triangular matrix-vector products spread over the whole GPU:
// gamma = X^T (X rhs)  — the same L^-T L^-1 rhs, a few rounding errors apart.
__global__ void k_tri_inv_diag(const double *L, int n, double *X) {  // X[kb.., kb..] = L[kb.., kb..]^-1, one warp per block
  const int kb = blockIdx.x * kNB;
  const size_t off = (size_t)kb * n + kb;
  tri_inv_block(L + off, n, min(kNB, n - kb), X + off);  // the strict upper triangle of X is zeroed beforehand
}

// block column j of X = L^-1 below the diagonal, one CTA per block column:  X_ij = -X_ii sum_{k=j}^{i-1} L_ik X_kj
__global__ void __launch_bounds__(256) k_tri_inv_column(const double *L, int n, double *X) {
  const int jb = blockIdx.x * kNB, bj = min(kNB, n - jb);
  __shared__ double A[kNB][kNB + 1], B[kNB][kNB + 1], S[kNB][kNB + 1];
  const int tid = threadIdx.x, r = tid >> 3, c0 = (tid & 7) * 4;
  for (int ib = jb + kNB; ib < n; ib += kNB) {
    const int bi = min(kNB, n - ib);
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    for (int kb = jb; kb < ib; kb += kNB) {
      __syncthreads();
      for (int e = tid; e < kNB * kNB; e += 256) {
        const int rr = e / kNB, cc = e % kNB;
        A[rr][cc] = rr < bi ? L[(size_t)(ib + rr) * n + kb + cc] : 0.0;            // kb + cc < ib <= n
        B[rr][cc] = cc < bj ? X[(size_t)(kb + rr) * n + jb + cc] : 0.0;            // rows kb.. < ib: written earlier
      }
      __syncthreads();
#pragma unroll 8
      for (int q = 0; q < kNB; ++q) {
        const double a = A[r][q];
#pragma unroll
        for (int u = 0; u < 4; ++u) acc[u] += a * B[q][c0 + u];
      }
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < 4; ++u) S[r][c0 + u] = acc[u];
    for (int e = tid; e < kNB * kNB; e += 256) {  // A <- X_ii (lower triangular, from k_tri_inv_diag)
      const int rr = e / kNB, cc = e % kNB;
      A[rr][cc] = (rr < bi && cc <= rr) ? X[(size_t)(ib + rr) * n + ib + cc] : 0.0;
    }
    __syncthreads();
    double o[4] = {0.0, 0.0, 0.0, 0.0};
    for (int q = 0; q <= r; ++q) {
      const double a = A[r][q];
#pragma unroll
      for (int u = 0; u < 4; ++u) o[u] -= a * S[q][c0 + u];
    }
    if (r < bi)
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (c0 + u < bj) X[(size_t)(ib + r) * n + jb + c0 + u] = o[u];
    __threadfence_block();
  }
}

__global__ void k_transpose(const double *A, int n, double *At) {
  __shared__ double T[32][33];
  const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y)
    T[r][threadIdx.x] = (by + r < n && bx + threadIdx.x < n) ? A[(size_t)(by + r) * n + bx + threadIdx.x] : 0.0;
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y)
    if (bx + r < n && by + threadIdx.x < n) At[(size_t)(bx + r) * n + by + threadIdx.x] = T[threadIdx.x][r];
}

// rhs = Q^T d_special + d_rest of the coarse domain (domain.rs:405-416)
__global__ void k_big_rhs(DomainTable t, const double *qpool, const double *res, double *rhs) {
  const int rk = t.rank[0];
  const int n = (int)(t.pt_ptr[1] - t.pt_ptr[0]), mm = n - rk;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= mm) return;
  const int *idx = t.pt_idx + t.pt_ptr[0];
  const double *Q = qpool + t.q_off[0];
  double v = res[idx[rk + j]];
  for (int a = 0; a < rk; ++a) v += Q[(size_t)a * mm + j] * res[idx[a]];
  rhs[j] = v;
}

// y[r] = sum over the stored triangle of row r of M[r][c] v[c]: one warp per row, fixed summation order
template <bool LOWER>
__global__ void __launch_bounds__(256) k_tri_gemv(const double *M, int n, const double *v, double *y) {
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (r >= n) return;
  const double *row = M + (size_t)r * n;
  const int lo = LOWER ? 0 : (r & ~31), hi = LOWER ? r + 1 : n;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  int c = lo + lane;
  for (; c + 96 < hi; c += 128) {
    s0 += row[c] * v[c];
    s1 += row[c + 32] * v[c + 32];
    s2 += row[c + 64] * v[c + 64];
    s3 += row[c + 96] * v[c + 96];
  }
  for (; c < hi; c += 32) s0 += row[c] * v[c];  // the upper case starts inside the zero part of the diagonal block
  double sacc = (s0 + s1) + (s2 + s3);
  for (int o = 16; o > 0; o >>= 1) sacc += __shfl_down_sync(0xffffffffu, sacc, o);
  if (lane == 0) y[r] = sacc;
}

// lambda_top = Q gamma, scatter, polynomial tail of the coarse domain, one CTA (the end of k_dom_solve)
__global__ void __launch_bounds__(kSolveThreads) k_big_finish(DomainTable t, const double *qpool, const double *gamma,
                                                              const double *res, double *out, int mode, int add_poly,
                                                              const double *a_special, const double *sp_inv,
                                                              size_t n_total) {
  const long long p0 = t.pt_ptr[0];
  const int rk = t.rank[0];
  const int *idx = t.pt_idx + p0;
  __shared__ double top[16], red[16];
  if ((int)threadIdx.x < rk) red[threadIdx.x] = res[idx[threadIdx.x]];  // d_special
  dom_solve_finish(qpool + t.q_off[0], gamma, red, idx, t.pt_mask + p0, (int)(t.pt_ptr[1] - p0), rk, mode, add_poly,
                   a_special, sp_inv, n_total, top, red, out);
}

// A[special, :] rows of the coarse domain (domain.rs:366)
__global__ void k_special_rows(const int *idx, int n, int rk, const double *px, const double *py, const double *pz,
                               KParams kp, double nugget, double *out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  for (int a = 0; a < rk; ++a)
    out[(size_t)a * n + i] = kval_rt(pair_r2(px, py, pz, idx[a], idx[i]), kp) + (a == i ? nugget : 0.0);
}

// ------------------------------------------------------------------------------------------ level
struct LevelDev {
  DomainTable tab{};
  int n_domains = 0;
  size_t max_n = 0, max_mm = 0;
  DBuf<long long> pt_ptr, q_off, l_off, s_off;
  DBuf<int> pt_idx, rank;
  DBuf<uint8_t> pt_mask;
  DBuf<double> qpool, lpool;
  DBuf<uint8_t> use_inverse;  // all zero unless a domain needed the indefinite fallback
  int n_fallback = 0;
  // one-domain level: X = L^-1 and its transpose (row-major mm x mm), vectors of the spread solve
  bool big_inverse = false;
  DBuf<double> linv, linv_t, big_v;
  DBuf<uint8_t> fail;         // per domain: Cholesky met a non-positive pivot
  std::vector<int> h_mms;     // order of every domain's Q^T A Q (host copy, for the fallback)
  std::vector<long long> h_l_off;
  unsigned tiles = 0;
  DBuf<unsigned long long> level_idx;  // point_indices of the level (matvec_partial target set)
  size_t n_level_pts = 0;
  TargetBuffers tb;
  TargetSet ts{};
  bool all_points = false;
  // coarse extras
  DBuf<double> a_special, sp_inv;
  bool solve_for_poly = false;
};

}  // namespace fb

using namespace fb;

struct fr_model {
  int dim = 0;
  size_t n = 0, n_cols = 0, n_in = 0;
  Settings st;
  fr_params params{};
  KParams kp{};
  std::vector<double> points, values;  // after duplicate removal, row-major (original coordinates)
  // global trend (global_trend.rs:128-287): kernel-space coordinates x' = [x 1] * aff; `kpts` holds the kernel-space
  // copy of `points` the trees / DDM / domain matrices are built from (empty without a trend: `points` is used)
  bool has_trend = false;
  fr_global_trend trend{};
  double aff[16] = {0}, aff_inv[16] = {0};  // (dim+1) x (dim+1), row-major, applied to homogeneous ROW vectors
  std::vector<double> kpts;
  const double *kernel_points() const { return has_trend ? kpts.data() : points.data(); }
  void build_trend_transform();
  void apply_affine(const double *a, const double *in, size_t cnt, ptrdiff_t rs, ptrdiff_t cs, double *out) const;
  void transform_extents(double *ext) const;  // [mins..., maxs...] -> extents of the transformed box corners
  std::vector<double> translation, scale;
  std::vector<double> point_coeff, poly_coeff;
  std::vector<LevelHost> ddm;
  fr_model_info info{};
  std::unique_ptr<fb_tree, void (*)(fb_tree *)> evaluator{nullptr, fb_tree_free};
  fr_progress_cb cb = nullptr;
  void *cb_user = nullptr;

  void fit();
  fb_tree *make_tree(bool sparse, const double *extents);
  // make_tree with the point coefficients uploaded and their multipoles computed
  std::unique_ptr<fb_tree, void (*)(fb_tree *)> transient_tree(bool sparse, const double *extents);
  // [mins..., maxs...] of the source points and target_ext together, mapped to kernel space (ext may be target_ext)
  void evaluation_extents(const double *target_ext, double *ext) const;
  // the interpolant at targets in device memory, on t->stream; every evaluation entry point ends here
  void eval_tree(fb_tree *t, const double *d_targets, size_t m, ptrdiff_t rs, ptrdiff_t cs, bool leaves, bool add_nugget,
                 double *d_out, double *d_grads);
  // host targets for eval_staged: their rows, row-major, in d_targets, queued on s
  void stage_targets(const double *targets, size_t m, ptrdiff_t rs, ptrdiff_t cs, cudaStream_t s);
  // eval_tree of the staged targets into the tree's output buffers, then downloaded to row-major host arrays
  void eval_staged(fb_tree *t, size_t m, bool leaves, bool add_nugget, double *out_vals, double *out_grads);
  DBuf<double> d_poly;     // poly_coeff on the device, uploaded on first use
  DBuf<double> d_ext;      // partial results of the device extents reduction (fr_evaluate, fr_evaluate_device)
  DBuf<double> d_targets;  // host targets staged by stage_targets
  void emit(int kind, uint64_t iter, double residual, double progress, const char *msg) {
    if (!cb) return;
    fr_event ev{kind, iter, residual, progress, msg};
    cb(&ev, cb_user);
  }
};

namespace {

double progress_from_rel(double current_res, double start_res, double target_res) {  // progress.rs:124-130
  if (current_res <= target_res) return 1.0;
  return (std::log10(start_res) - std::log10(current_res)) / (std::log10(start_res) - std::log10(target_res));
}

// inverse of a dense n x n matrix (row-major) by Gauss-Jordan elimination with partial pivoting; false when singular
static bool invert_pivoted(const std::vector<double> &a_in, int n, std::vector<double> &inv) {
  std::vector<double> a(a_in);
  inv.assign((size_t)n * n, 0.0);
  for (int i = 0; i < n; ++i) inv[(size_t)i * n + i] = 1.0;
  double amax = 0.0;
  for (double v : a) amax = std::max(amax, std::fabs(v));
  for (int k = 0; k < n; ++k) {
    int piv = k;
    for (int i = k + 1; i < n; ++i)
      if (std::fabs(a[(size_t)i * n + k]) > std::fabs(a[(size_t)piv * n + k])) piv = i;
    if (!(std::fabs(a[(size_t)piv * n + k]) > 1e-14 * amax)) return false;
    if (piv != k)
      for (int c = 0; c < n; ++c) {
        std::swap(a[(size_t)k * n + c], a[(size_t)piv * n + c]);
        std::swap(inv[(size_t)k * n + c], inv[(size_t)piv * n + c]);
      }
    const double d = 1.0 / a[(size_t)k * n + k];
    for (int c = 0; c < n; ++c) {
      a[(size_t)k * n + c] *= d;
      inv[(size_t)k * n + c] *= d;
    }
#pragma omp parallel for schedule(static)
    for (int i = 0; i < n; ++i) {
      if (i == k) continue;
      const double f = a[(size_t)i * n + k];
      if (f == 0.0) continue;
      double *ai = &a[(size_t)i * n], *ii = &inv[(size_t)i * n];
      const double *ak = &a[(size_t)k * n], *ik = &inv[(size_t)k * n];
      for (int c = 0; c < n; ++c) {
        ai[c] -= f * ak[c];
        ii[c] -= f * ik[c];
      }
    }
  }
  return true;
}

struct DeviceSolver {
  fr_model &M;
  fb_tree *tree;
  cudaStream_t s;
  size_t n, m, nt;  // points, basis, n + m
  DBuf<double> px, py, pz, P, Qp, proj, scalar;
  DBuf<unsigned long long> umax;
  std::vector<std::unique_ptr<LevelDev>> levels;
  DBuf<double> scratch;
  uint64_t matvecs = 0;

  cudaStream_t upload_stream = nullptr;
  cudaEvent_t upload_done = nullptr;

  DeviceSolver(fr_model &model, fb_tree *t) : M(model), tree(t), s(t ? t->stream : nullptr) {}
  ~DeviceSolver() {
    if (upload_done) cudaEventDestroy(upload_done);
    if (upload_stream) cudaStreamDestroy(upload_stream);
  }

  void upload_points(cudaStream_t stream) {
    n = M.n;
    m = (size_t)M.st.basis_size;
    nt = n + m;
    std::vector<double> x(n), y(n, 0.0), z(n, 0.0);
    for (size_t i = 0; i < n; ++i) {
      const double *kp = M.kernel_points();
      x[i] = kp[i * M.dim];
      if (M.dim > 1) y[i] = kp[i * M.dim + 1];
      if (M.dim > 2) z[i] = kp[i * M.dim + 2];
    }
    px.upload(x, stream);
    py.upload(y, stream);
    pz.upload(z, stream);
    scalar.reserve(16);
    umax.reserve(1);
  }

  // ---- Cholesky of every slot of a level's factor pool; domains whose Q^T A Q is not positive definite take the
  //      reference's fallback (domain.rs:63-68: faer's Bunch-Kaufman LBL^T, linalg.rs:514-616): the matrix is assembled
  //      again, inverted on the host with a pivoted elimination and the explicit inverse stored in the slot
  //      (DomainTable::use_inverse); both solve the same symmetric indefinite system.
  void factorise_launch(LevelDev &lv, cudaStream_t stream) {  // asynchronous: nothing here waits for the device
    const size_t nd = lv.h_mms.size();
    lv.fail.reserve(nd);
    lv.use_inverse.reserve(nd);
    FB_CUDA(cudaMemsetAsync(lv.fail.p, 0, nd, stream));
    FB_CUDA(cudaMemsetAsync(lv.use_inverse.p, 0, nd, stream));
    lv.tab.use_inverse = lv.use_inverse.p;
    const size_t smem = sizeof(double) * ((size_t)(kNB + 1) * kNB + (size_t)kPS * kNB * (1 + 8));
    FB_CUDA(cudaFuncSetAttribute(k_cholesky, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (nd == 1 && lv.max_mm >= 512) {  // one big matrix: spread every block column over the GPU
      const int nn = (int)lv.max_mm;
      FB_CUDA(cudaFuncSetAttribute(k_chol_big_panel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      FB_CUDA(cudaFuncSetAttribute(k_chol_big_update, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      for (int kb = 0; kb < nn; kb += kNB) {
        FB_LAUNCH(k_chol_big_panel, 1, 256, smem, stream, lv.lpool.p, nn, kb, lv.fail.p);
        const int ntile = (nn - (kb + kNB) + kNB - 1) / kNB;
        if (ntile > 0) {
          dim3 grid((unsigned)ntile, (unsigned)((ntile + 7) / 8));
          FB_LAUNCH(k_chol_big_update, grid, 256, smem, stream, lv.lpool.p, nn, kb);
        }
      }
      // X = L^-1 and X^T for the spread solve (unused if the factorisation failed: factorise_finish then stores the
      // explicit inverse and k_dom_solve serves the level)
      lv.linv.reserve((size_t)nn * nn);
      lv.linv_t.reserve((size_t)nn * nn);
      lv.big_v.reserve(3 * (size_t)nn);
      FB_CUDA(cudaMemsetAsync(lv.linv.p, 0, sizeof(double) * (size_t)nn * nn, stream));
      const unsigned nblock = (unsigned)((nn + kNB - 1) / kNB);
      FB_LAUNCH(k_tri_inv_diag, nblock, 32, 0, stream, lv.lpool.p, nn, lv.linv.p);
      FB_LAUNCH(k_tri_inv_column, nblock, 256, 0, stream, lv.lpool.p, nn, lv.linv.p);
      FB_LAUNCH(k_transpose, dim3(nblock, nblock), dim3(32, 8), 0, stream, lv.linv.p, nn, lv.linv_t.p);
      lv.big_inverse = true;
    } else {
      FB_LAUNCH(k_cholesky, (unsigned)nd, 256, smem, stream, lv.tab, lv.lpool.p, lv.fail.p);
      if (lv.max_mm > 0)
        FB_LAUNCH(k_inv_diag_inplace, dim3((unsigned)nd, (unsigned)((lv.max_mm + kNB - 1) / kNB)), 32, 0, stream, lv.tab,
                  lv.lpool.p);
    }
  }

  template <class Reassemble>
  void factorise_finish(LevelDev &lv, Reassemble &&reassemble, cudaStream_t stream) {
    const size_t nd = lv.h_mms.size();
    std::vector<uint8_t> h_fail(nd, 0);
    FB_CUDA(cudaMemcpyAsync(h_fail.data(), lv.fail.p, nd, cudaMemcpyDeviceToHost, stream));
    FB_CUDA(cudaStreamSynchronize(stream));
    std::vector<double> a, inv;
    for (size_t d = 0; d < nd; ++d) {
      if (!h_fail[d]) continue;
      const int mm = lv.h_mms[d];
      reassemble(d);
      a.resize((size_t)mm * mm);
      FB_CUDA(cudaMemcpyAsync(a.data(), lv.lpool.p + lv.h_l_off[d], a.size() * sizeof(double), cudaMemcpyDeviceToHost,
                              stream));
      FB_CUDA(cudaStreamSynchronize(stream));
      for (int i = 0; i < mm; ++i)  // the slot holds the lower triangle
        for (int j = i + 1; j < mm; ++j) a[(size_t)i * mm + j] = a[(size_t)j * mm + i];
      if (!invert_pivoted(a, mm, inv))
        throw Error(FB_ERR_INVALID_ARGUMENT, "subdomain matrix Q^T A Q is singular (domain " + std::to_string(d) + ")");
      FB_CUDA(cudaMemcpyAsync(lv.lpool.p + lv.h_l_off[d], inv.data(), inv.size() * sizeof(double), cudaMemcpyHostToDevice,
                              stream));
      const uint8_t one = 1;
      FB_CUDA(cudaMemcpyAsync(lv.use_inverse.p + d, &one, 1, cudaMemcpyHostToDevice, stream));
      FB_CUDA(cudaStreamSynchronize(stream));
      ++lv.n_fallback;
    }
  }

  // ---- Cholesky of every slot of a level's factor pool; domains whose Q^T A Q is not positive definite take the
  //      reference's fallback (domain.rs:63-68: faer's Bunch-Kaufman LBL^T, linalg.rs:514-616): the matrix is assembled
  //      again, inverted on the host with a pivoted elimination and the explicit inverse stored in the slot
  //      (DomainTable::use_inverse); both solve the same symmetric indefinite system.
  template <class Reassemble>
  void factorise_pool(LevelDev &lv, const std::vector<int> &mms, const std::vector<long long> &l_off,
                      Reassemble &&reassemble, cudaStream_t stream) {
    lv.h_mms = mms;
    lv.h_l_off = l_off;
    factorise_launch(lv, stream);
    factorise_finish(lv, reassemble, stream);
  }

  // ---- factorise one level on the device (domain.rs:322-382)
  // queue the whole factorisation of a level (tables, assembly, Cholesky) without waiting for the device: the host goes on
  // building the next DDM level / the FMM tree meanwhile (fit())
  void build_level_launch(const LevelHost &lh, bool coarse, cudaStream_t stream) {
    static const bool verbose = std::getenv("FB_TIMING") != nullptr;
    auto t_sub = std::chrono::steady_clock::now();
    auto sublap = [&](const char *what) {
      if (!verbose) return;
      fprintf(stderr, "[fr_fit]     %-26s %8.3f s (host, queued)\n", what,
              std::chrono::duration<double>(std::chrono::steady_clock::now() - t_sub).count());
      t_sub = std::chrono::steady_clock::now();
    };
    auto lv = std::make_unique<LevelDev>();
    const size_t nd = lh.domains.size();
    std::vector<long long> pt_ptr(nd + 1, 0), q_off(nd, 0), l_off(nd, 0), s_off(nd, 0);
    std::vector<int> rank(nd, 0), pt_idx;
    std::vector<uint8_t> pt_mask;
    std::vector<double> qpool;
    long long lsize = 0, ssize = 0;
    for (size_t d = 0; d < nd; ++d) {
      const DomainHost &dh = lh.domains[d];
      const size_t nn = dh.idx.size(), mm = nn - dh.rank;
      FB_REQUIRE(dh.rank <= 16, "more than 16 special points per domain");
      rank[d] = dh.rank;
      for (size_t i = 0; i < nn; ++i) {
        pt_idx.push_back((int)dh.idx[i]);
        pt_mask.push_back(i < dh.mask.size() ? dh.mask[i] : 0);
      }
      pt_ptr[d + 1] = (long long)pt_idx.size();
      q_off[d] = (long long)qpool.size();
      qpool.insert(qpool.end(), dh.qtop.begin(), dh.qtop.end());
      l_off[d] = lsize;
      lsize += (long long)(mm * mm);
      s_off[d] = ssize;
      ssize += (long long)(2 * dh.rank * mm);
      lv->max_n = std::max(lv->max_n, nn);
      lv->max_mm = std::max(lv->max_mm, mm);
    }
    lv->n_domains = (int)nd;
    // the tables are pageable host memory: such a copy holds the host until the stream reaches it, i.e. until the previous
    // level's factorisation is done.  They go through an otherwise idle stream; the factorisation stream waits for them.
    if (!upload_stream) {
      FB_CUDA(cudaStreamCreateWithFlags(&upload_stream, cudaStreamNonBlocking));
      FB_CUDA(cudaEventCreateWithFlags(&upload_done, cudaEventDisableTiming));
    }
    lv->pt_ptr.upload(pt_ptr, upload_stream);
    lv->q_off.upload(q_off, upload_stream);
    lv->l_off.upload(l_off, upload_stream);
    lv->s_off.upload(s_off, upload_stream);
    lv->rank.upload(rank, upload_stream);
    lv->pt_idx.upload(pt_idx, upload_stream);
    lv->pt_mask.upload(pt_mask, upload_stream);
    lv->qpool.upload(qpool, upload_stream);
    FB_CUDA(cudaEventRecord(upload_done, upload_stream));
    FB_CUDA(cudaStreamWaitEvent(stream, upload_done, 0));
    sublap("host tables + uploads");
    lv->lpool.reserve((size_t)lsize);
    scratch.reserve((size_t)std::max<long long>(ssize, 1));
    sublap("factor pool allocation");
    DomainTable &t = lv->tab;
    t.n_domains = (int)nd;
    t.pt_ptr = lv->pt_ptr.p;
    t.pt_idx = lv->pt_idx.p;
    t.pt_mask = lv->pt_mask.p;
    t.rank = lv->rank.p;
    t.q_off = lv->q_off.p;
    t.l_off = lv->l_off.p;
    t.s_off = lv->s_off.p;
    const KParams kp = M.kp;
    FB_LAUNCH(k_dom_prep, (unsigned)nd, 128, 0, stream, t, px.p, py.p, pz.p, kp, M.st.nugget, lv->qpool.p, scratch.p);
    const unsigned tiles = (unsigned)((lv->max_mm + 31) / 32);
    // tiles == 0: every domain has as many points as special points (mm = 0), Q^T A Q is empty
    for (size_t d0 = 0; tiles > 0 && d0 < nd; d0 += 32768) {  // grid.z limit
      DomainTable tt = t;
      const unsigned cnt = (unsigned)std::min<size_t>(32768, nd - d0);
      tt.pt_ptr += d0;
      tt.rank += d0;
      tt.q_off += d0;
      tt.l_off += d0;
      tt.s_off += d0;
      FB_LAUNCH(k_dom_assemble, dim3(tiles, tiles, cnt), 256, 0, stream, tt, px.p, py.p, pz.p, kp, M.st.nugget,
                lv->qpool.p, scratch.p, lv->lpool.p);
    }
    sublap("prep + assemble");
    lv->tiles = tiles;
    lv->h_mms.resize(nd);
    for (size_t d = 0; d < nd; ++d) lv->h_mms[d] = (int)(lh.domains[d].idx.size() - lh.domains[d].rank);
    lv->h_l_off = l_off;
    factorise_launch(*lv, stream);
    if (coarse && !lh.domains.empty() && lh.domains[0].solve_for_poly) {
      const DomainHost &dh = lh.domains[0];
      const int nn = (int)dh.idx.size();
      lv->solve_for_poly = true;
      lv->a_special.reserve((size_t)dh.rank * nn);
      lv->sp_inv.upload(dh.sp_inv, upload_stream);
      FB_CUDA(cudaEventRecord(upload_done, upload_stream));
      FB_CUDA(cudaStreamWaitEvent(stream, upload_done, 0));
      FB_LAUNCH(k_special_rows, nblk(nn, 128), 128, 0, stream, lv->pt_idx.p, nn, dh.rank, px.p, py.p, pz.p, kp,
                M.st.nugget, lv->a_special.p);
    }
    lv->n_level_pts = lh.point_indices.size();
    lv->all_points = lv->n_level_pts == n;
    levels.push_back(std::move(lv));
  }

  // wait for the queued factorisations, run the indefinite fallback where Cholesky failed, bin the level's points as
  // the target set of its partial matvecs (needs the FMM tree)
  void finish_level(size_t l, const LevelHost &lh, cudaStream_t stream) {
    LevelDev &lv = *levels[l];
    const KParams kp = M.kp;
    auto reassemble = [&](size_t d) {  // one domain's Q^T A Q again (its slot was overwritten by the failed attempt)
      DomainTable tt = lv.tab;
      tt.pt_ptr += d;
      tt.rank += d;
      tt.q_off += d;
      tt.l_off += d;
      tt.s_off += d;
      tt.n_domains = 1;
      FB_LAUNCH(k_dom_prep, 1, 128, 0, stream, tt, px.p, py.p, pz.p, kp, M.st.nugget, lv.qpool.p, scratch.p);
      FB_LAUNCH(k_dom_assemble, dim3(lv.tiles, lv.tiles, 1), 256, 0, stream, tt, px.p, py.p, pz.p, kp, M.st.nugget,
                lv.qpool.p, scratch.p, lv.lpool.p);
    };
    factorise_finish(lv, reassemble, stream);
    if (std::getenv("FB_TIMING") && lv.n_fallback)
      fprintf(stderr, "[fr_fit]   level %zu: indefinite fallback used for %d domain(s)\n", l, lv.n_fallback);
    if (tree && !lv.all_points) {
      std::vector<unsigned long long> li(lh.point_indices.begin(), lh.point_indices.end());
      lv.level_idx.upload(li, stream);
      lv.ts = tree->subset_target_set_dev(lv.level_idx.p, li.size(), lv.tb);
    }
  }

  void solve_level(const LevelDev &lv, const double *res, double *out, int mode, int add_poly, cudaStream_t stream) {
    // the coarse domain, spread over the GPU.  Fine levels come from bisection in pairs of domains, so a one-domain
    // level is the coarse level or a naive / dense solve: always solved in mode 1
    if (lv.big_inverse && lv.n_fallback == 0) {
      const int mm = (int)lv.max_mm;
      double *rhs = lv.big_v.p, *y = rhs + mm, *gamma = y + mm;
      FB_LAUNCH(k_big_rhs, nblk(mm, 256), 256, 0, stream, lv.tab, lv.qpool.p, res, rhs);
      FB_LAUNCH((k_tri_gemv<true>), (unsigned)((mm + 7) / 8), 256, 0, stream, lv.linv.p, mm, rhs, y);
      FB_LAUNCH((k_tri_gemv<false>), (unsigned)((mm + 7) / 8), 256, 0, stream, lv.linv_t.p, mm, y, gamma);
      FB_LAUNCH(k_big_finish, 1, kSolveThreads, 0, stream, lv.tab, lv.qpool.p, gamma, res, out, mode, add_poly,
                lv.solve_for_poly ? lv.a_special.p : nullptr, lv.solve_for_poly ? lv.sp_inv.p : nullptr, nt);
      return;
    }
    const size_t smem = sizeof(double) * (lv.max_n + lv.max_mm + kSolveWarps * 32 + 32);
    // the gathered residual and the solution of a domain live in shared memory (227 KB per CTA on sm_100a)
    if (smem > 227 * 1024)
      throw Error(FB_ERR_INVALID_ARGUMENT,
                  "a subdomain of " + std::to_string(lv.max_n) + " points exceeds the shared-memory budget of the batched "
                  "subdomain solve (about 14300 points per domain): lower naive_solve_threshold / "
                  "DDMParams.coarse_threshold / DDMParams.leaf_threshold below that");
    FB_CUDA(cudaFuncSetAttribute(k_dom_solve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 1024)));
    FB_LAUNCH(k_dom_solve, (unsigned)lv.n_domains, kSolveThreads, smem, stream, lv.tab, lv.qpool.p, lv.lpool.p, res, out, mode,
              add_poly, lv.solve_for_poly ? lv.a_special.p : nullptr, lv.solve_for_poly ? lv.sp_inv.p : nullptr, nt);
  }

  // ---- vector helpers (device scalars are read back: Givens rotations stay on the host)
  double dot(const double *a, const double *b, size_t len) {
    FB_CUDA(cudaMemsetAsync(scalar.p, 0, sizeof(double), s));
    FB_LAUNCH(k_dot, std::min<unsigned>(nblk(len, 256), 592), 256, 0, s, a, b, len, scalar.p);
    double h = 0;
    FB_CUDA(cudaMemcpyAsync(&h, scalar.p, sizeof(double), cudaMemcpyDeviceToHost, s));
    FB_CUDA(cudaStreamSynchronize(s));
    return h;
  }
  double norm2(const double *a, size_t len) { return std::sqrt(dot(a, a, len)); }
  double norm_max(const double *a, size_t len) {
    FB_CUDA(cudaMemsetAsync(umax.p, 0, sizeof(unsigned long long), s));
    FB_LAUNCH(k_absmax, std::min<unsigned>(nblk(len, 256), 592), 256, 0, s, a, len, umax.p);
    unsigned long long h = 0;
    FB_CUDA(cudaMemcpyAsync(&h, umax.p, sizeof(h), cudaMemcpyDeviceToHost, s));
    FB_CUDA(cudaStreamSynchronize(s));
    double d;
    std::memcpy(&d, &h, sizeof(d));
    return d;
  }
  void axpy(double a, const double *x, double *y, size_t len) { FB_LAUNCH(k_axpy, nblk(len, 256), 256, 0, s, a, x, y, len); }
  void scale_to(double a, const double *x, double *y, size_t len) {
    FB_LAUNCH(k_scale_to, nblk(len, 256), 256, 0, s, a, x, y, len);
  }
  void sub_to(const double *a, const double *b, double *y, size_t len) {
    FB_LAUNCH(k_sub_to, nblk(len, 256), 256, 0, s, a, b, y, len);
  }

  // ---- fast_matrix_vector_product (rbf.rs:1338-1379); lv == nullptr or all_points => all rows
  void matvec(const double *w, const LevelDev *lv, double *y) {
    FB_CUDA(cudaMemsetAsync(y, 0, nt * sizeof(double), s));
    tree->nrhs = 1;
    tree->d_w_user.reserve(n);
    FB_CUDA(cudaMemcpyAsync(tree->d_w_user.p, w, n * sizeof(double), cudaMemcpyDeviceToDevice, s));
    tree->w_cache_valid = false;  // the host copy of the last upload no longer describes d_w_user
    const bool all = lv == nullptr || lv->all_points;
    TargetSet ts = all ? tree->source_target_set() : lv->ts;
    static const bool verbose = std::getenv("FB_TIMING") != nullptr;
    std::chrono::steady_clock::time_point t0;
    if (verbose) {
      FB_CUDA(cudaStreamSynchronize(s));
      t0 = std::chrono::steady_clock::now();
    }
    tree->matvec_dev(ts);
    if (verbose) {
      FB_CUDA(cudaStreamSynchronize(s));
      fprintf(stderr, "[fr_fit]   matvec on %9zu targets %8.3f ms\n", ts.m,
              1e3 * std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
    }
    ++matvecs;
    const size_t cnt = all ? n : lv->n_level_pts;
    FB_LAUNCH(k_matvec_finish, nblk(cnt, 256), 256, 0, s, tree->d_out.p, all ? nullptr : lv->level_idx.p, cnt, w, n,
              (int)m, m ? P.p : nullptr, M.st.nugget, y);
  }

  // ---- schwarz_preconditioner (schwarz.rs:32-79)
  DBuf<double> sl, res, tmp, s1;
  void precon(const double *rg, double *out) {
    sl.reserve(nt);
    res.reserve(nt);
    tmp.reserve(nt);
    s1.reserve(nt);
    FB_CUDA(cudaMemsetAsync(sl.p, 0, nt * sizeof(double), s));
    const int coarse = (int)levels.size() - 1;
    auto coarse_step = [&](bool add_poly) {
      matvec(sl.p, levels[coarse].get(), tmp.p);
      sub_to(rg, tmp.p, res.p, nt);
      FB_CUDA(cudaMemsetAsync(s1.p, 0, nt * sizeof(double), s));
      solve_level(*levels[coarse], res.p, s1.p, 1, add_poly ? 1 : 0, s);
      axpy(1.0, s1.p, sl.p, nt);
    };
    if (coarse > 0) {
      for (int i = 0; i < coarse; ++i) {
        if (i == 0) {
          // sl is still exactly zero: A * 0 = 0 and rg - 0 = rg bit for bit, so the reference's first
          // matvec_partial of the cycle (schwarz.rs:88-92) is skipped — it is the full-size one
          FB_CUDA(cudaMemcpyAsync(res.p, rg, nt * sizeof(double), cudaMemcpyDeviceToDevice, s));
        } else {
          matvec(sl.p, levels[i].get(), tmp.p);
          sub_to(rg, tmp.p, res.p, nt);
        }
        FB_CUDA(cudaMemsetAsync(s1.p, 0, nt * sizeof(double), s));
        solve_level(*levels[i], res.p, s1.p, 0, 0, s);
        if (m) {  // orthogonalise against the global polynomial space (schwarz.rs:111-117)
          FB_CUDA(cudaMemsetAsync(proj.p, 0, m * sizeof(double), s));
          FB_LAUNCH(k_project_dots, std::min<unsigned>(nblk(n, 256), 592), 256, 0, s, Qp.p, s1.p, n, (int)m, proj.p);
          FB_LAUNCH(k_project_apply, nblk(n, 256), 256, 0, s, Qp.p, proj.p, n, (int)m, s1.p);
        }
        axpy(1.0, s1.p, sl.p, nt);
        coarse_step(i == coarse - 1);
      }
    } else {
      coarse_step(true);
    }
    FB_CUDA(cudaMemcpyAsync(out, sl.p, nt * sizeof(double), cudaMemcpyDeviceToDevice, s));
  }
};

void givens_rotation(double f, double g, double &c, double &s, double &r) {  // iterative_solvers.rs:192-232
  const double safmin = 2.2250738585072014e-308, safmax = 1.7976931348623157e308;
  const double rtmin = std::sqrt(safmin), rtmax = std::sqrt(safmax / 2.0);
  if (g == 0.0) { c = 1.0; s = 0.0; r = f; return; }
  if (f == 0.0) { c = 0.0; s = g > 0 ? 1.0 : -1.0; r = std::fabs(g); return; }
  const double f1 = std::fabs(f), g1 = std::fabs(g);
  if (f1 >= rtmin && f1 < rtmax && g1 >= rtmin && g1 < rtmax) {
    r = std::copysign(std::sqrt(f * f + g * g), f);
    c = f1 / std::fabs(r);
    s = g / r;
  } else {
    const double u = std::min(std::max(std::max(f1, g1), safmin), safmax);
    const double fs = f / u, gs = g / u;
    const double mag = std::sqrt(fs * fs + gs * gs);
    r = std::copysign(mag, f) * u;
    c = std::fabs(fs) / mag;
    s = gs / mag;
  }
}

}  // namespace

// ------------------------------------------------------------------------------------------- fit
fb_tree *fr_model::make_tree(bool sparse, const double *extents) {
  fb_fmm_params fp;
  fp.max_points_per_cell = params.max_points_per_cell;
  fp.compression_type = params.compression_type;
  fp.epsilon = params.epsilon;
  fp.eval_chunk_size = params.eval_chunk_size;
  fb_tree *t = new fb_tree();
  try {
    t->build(kernel_points(), n, dim, dim, 1, (int)params.interpolation_order, &st.kparams, 1, sparse ? 1 : 0, extents,
             &fp);
  } catch (...) {
    delete t;
    throw;
  }
  return t;
}

std::unique_ptr<fb_tree, void (*)(fb_tree *)> fr_model::transient_tree(bool sparse, const double *extents) {
  std::unique_ptr<fb_tree, void (*)(fb_tree *)> t(make_tree(sparse, extents), fb_tree_free);
  t->upload_weights(point_coeff.data(), n, n_cols, (ptrdiff_t)n_cols, 1);
  t->upward();
  return t;
}

namespace {

using TreePtr = std::unique_ptr<fb_tree, void (*)(fb_tree *)>;

// The set-up of the solve, shared by fr_model::fit and fr_ddm_level_solve: kernel-space points and monomial scaling, the
// DDM hierarchy (or the single dense domain below naive_solve_threshold) with every level factorised on the device and,
// with_tree, the FMM tree and the levels' target sets.  mono_pts receives the inverse-transformed points of a trend
// fit.  On return S.s is the stream the solve runs on.
void setup_solve(fr_model &M, DeviceSolver &S, cudaStream_t setup_stream, bool with_tree, std::vector<double> &mono_pts,
                 TreePtr &tree) {
  using clk = std::chrono::steady_clock;
  const size_t n = M.n, m = (size_t)M.st.basis_size;
  const int dim = M.dim;
  M.translation.assign(dim, 0.0);
  M.scale.assign(dim, 1.0);
  // global trend (rbf.rs:361-371): kernel space = transformed points; monomials are evaluated at the inverse
  // transform of those (rbf.rs:477-484, domain.rs:169-175), which also become the public points (rbf.rs:579-581)
  if (M.has_trend) {
    M.build_trend_transform();
    M.kpts.resize(n * dim);
    M.apply_affine(M.aff, M.points.data(), n, dim, 1, M.kpts.data());
    mono_pts.resize(n * dim);
    M.apply_affine(M.aff_inv, M.kpts.data(), n, dim, 1, mono_pts.data());
  }
  const double *kp_ptr = M.kernel_points();
  const double *mono_ptr = M.has_trend ? mono_pts.data() : nullptr;
  if (m) cheb_cube_scaling(kp_ptr, nullptr, n, dim, M.translation.data(), M.scale.data());  // rbf.rs:418-421

  const bool naive = n < M.params.naive_solve_threshold;
  const bool verbose = std::getenv("FB_TIMING") != nullptr;
  auto lap = [&](const char *what, clk::time_point &t0) {
    if (verbose) fprintf(stderr, "[fr_fit] %-28s %8.3f s\n", what, std::chrono::duration<double>(clk::now() - t0).count());
    t0 = clk::now();
  };
  auto t_lap = clk::now();
  // Setup order: the device factorises a DDM level (assembly + batched Cholesky, ~0.15 s for the finest level of a
  // 1M-point fit) while the host builds the next level and then the FMM tree (~0.15 s of host work): the hierarchy comes
  // first, every finished level is queued on a setup stream at once, the tree is built under it.
  S.s = setup_stream;
  S.upload_points(setup_stream);
  if (m && !naive) {
    std::vector<double> Pm(n * m), Qm(n * m);
    evaluate_monomials(mono_ptr ? mono_ptr : M.points.data(), nullptr, n, dim, M.st.polynomial_degree, (int)m,
                       M.translation.data(), M.scale.data(), Pm.data());
    thin_q_rowmajor(Pm.data(), n, (int)m, Qm.data());
    S.P.upload(Pm, setup_stream);
    S.Qp.upload(Qm, setup_stream);
    S.proj.reserve(m);
  }
  lap("points / monomials / thin Q", t_lap);
  std::vector<LevelHost> &ddm = M.ddm;
  if (naive) {  // single dense domain (rbf.rs:423-454)
    LevelHost lh;
    lh.point_indices.resize(n);
    for (size_t i = 0; i < n; ++i) lh.point_indices[i] = (int64_t)i;
    DomainHost d;
    d.idx = lh.point_indices;
    d.mask.assign(n, 1);
    d.prepare(kp_ptr, dim, M.st, true, mono_ptr);
    lh.domains.push_back(std::move(d));
    ddm.clear();
    ddm.push_back(std::move(lh));
    S.build_level_launch(ddm[0], true, setup_stream);
  } else {
    const LevelCallback queue_level = [&](size_t, const LevelHost &level, bool is_coarse) {
      S.build_level_launch(level, is_coarse, setup_stream);
    };
    ddm = build_ddm(kp_ptr, n, dim, M.st, M.params, mono_ptr, &queue_level);
    lap("ddm hierarchy (host) + queued factorisations", t_lap);
    if (with_tree) {
      tree.reset(M.make_tree(true, nullptr));  // adaptive, sparse, own extents (rbf.rs:456-467)
      lap("fmm tree + operators", t_lap);
      S.tree = tree.get();
    }
  }
  FB_CUDA(cudaStreamSynchronize(setup_stream));
  if (tree) S.s = tree->stream;  // from here on everything runs on the tree's stream
  for (size_t l = 0; l < ddm.size(); ++l) S.finish_level(l, ddm[l], S.s);
  lap("factorisations finished + level target sets", t_lap);
}

}  // namespace

void fr_model::fit() {
  using clk = std::chrono::steady_clock;
  const auto t_start = clk::now();
  info = fr_model_info{};
  info.dim = (uint64_t)dim;
  info.n_cols = n_cols;
  info.basis_size = (uint64_t)st.basis_size;
  const size_t m = (size_t)st.basis_size;
  const size_t nt = n + m;
  const bool naive = n < params.naive_solve_threshold;
  std::vector<double> mono_pts;
  TreePtr tree(nullptr, fb_tree_free);
  cudaStream_t setup_stream = nullptr;
  FB_CUDA(cudaStreamCreateWithFlags(&setup_stream, cudaStreamNonBlocking));
  std::unique_ptr<DeviceSolver> solver(new DeviceSolver(*this, nullptr));
  try {
    DeviceSolver &S = *solver;
    setup_solve(*this, S, setup_stream, true, mono_pts, tree);
    const cudaStream_t stream = S.s;
    point_coeff.assign(n * n_cols, 0.0);
    poly_coeff.assign(m * n_cols, 0.0);
    info.ddm_levels = ddm.size();
    for (size_t l = 0; l < ddm.size() && l < 8; ++l) info.ddm_domains[l] = ddm[l].domains.size();
    const auto t_setup = clk::now();
    info.setup_seconds = std::chrono::duration<double>(t_setup - t_start).count();

    DBuf<double> b, x, r, w, wj, V, Z, tmp;
    b.reserve(nt);
    x.reserve(nt);
    std::vector<double> hb(nt), hx(nt);
    for (size_t col = 0; col < n_cols; ++col) {
      for (size_t i = 0; i < n; ++i) hb[i] = values[i * n_cols + col];
      for (size_t k = 0; k < m; ++k) hb[n + k] = 0.0;
      FB_CUDA(cudaMemcpyAsync(b.p, hb.data(), nt * sizeof(double), cudaMemcpyHostToDevice, stream));
      if (naive) {
        FB_CUDA(cudaMemsetAsync(x.p, 0, nt * sizeof(double), stream));
        S.solve_level(*S.levels[0], b.p, x.p, 1, 1, stream);
      } else if (params.solver_type == FR_SOLVER_FGMRES) {
        // ---- fgmres(matvec, rhs, precon, x0 = None, 20 outer, 5 inner)  (rbf.rs:536-547)
        const int max_outer = 20, mi = 5;
        r.reserve(nt);
        w.reserve(nt);
        wj.reserve(nt);
        tmp.reserve(nt);
        V.reserve(nt * (mi + 1));
        Z.reserve(nt * mi);
        FB_CUDA(cudaMemsetAsync(x.p, 0, nt * sizeof(double), stream));
        // r = b - A x0 with x0 = 0: the reference runs a zero matvec here (iterative_solvers.rs:56); A 0 = 0
        FB_CUDA(cudaMemcpyAsync(r.p, b.p, nt * sizeof(double), cudaMemcpyDeviceToDevice, stream));
        const bool absolute = st.tolerance_type == FR_TOL_ABSOLUTE;
        const double beta = absolute ? S.norm_max(r.p, nt) : S.norm2(r.p, nt);
        uint64_t iteration = 1;
        bool done = beta == 0.0;
        double H[6][5], g[6], cs[5], sn[5];
        for (int outer = 0; outer < max_outer && !done; ++outer) {
          std::memset(H, 0, sizeof(H));
          std::memset(g, 0, sizeof(g));
          std::memset(cs, 0, sizeof(cs));
          std::memset(sn, 0, sizeof(sn));
          const double r_norm = S.norm2(r.p, nt);
          S.scale_to(1.0 / r_norm, r.p, V.p, nt);
          g[0] = r_norm;
          int used = mi;
          for (int j = 0; j < mi; ++j) {
            double *zj = Z.p + (size_t)j * nt;
            S.precon(V.p + (size_t)j * nt, zj);
            S.matvec(zj, nullptr, wj.p);
            for (int i = 0; i <= j; ++i) {  // modified Gram-Schmidt
              const double hij = S.dot(V.p + (size_t)i * nt, wj.p, nt);
              H[i][j] = hij;
              S.axpy(-hij, V.p + (size_t)i * nt, wj.p, nt);
            }
            const double norm = S.norm2(wj.p, nt);
            H[j + 1][j] = norm;
            for (int i = 0; i < j; ++i) {
              const double temp = cs[i] * H[i][j] + sn[i] * H[i + 1][j];
              H[i + 1][j] = -sn[i] * H[i][j] + cs[i] * H[i + 1][j];
              H[i][j] = temp;
            }
            double c, sv, rr;
            givens_rotation(H[j][j], H[j + 1][j], c, sv, rr);
            H[j][j] = c * H[j][j] + sv * H[j + 1][j];
            H[j + 1][j] = 0.0;
            const double temp = c * g[j] + sv * g[j + 1];
            g[j + 1] = -sv * g[j] + c * g[j + 1];
            g[j] = temp;
            cs[j] = c;
            sn[j] = sv;
            if (norm != 0.0) S.scale_to(1.0 / norm, wj.p, V.p + (size_t)(j + 1) * nt, nt);
            const double res_norm = absolute ? std::fabs(g[j + 1]) : std::fabs(g[j + 1]) / beta;
            info.iterations += 1;
            info.last_residual = res_norm;
            emit(FR_EVENT_SOLVER_ITERATION, iteration, res_norm, progress_from_rel(res_norm, beta, st.tolerance),
                 nullptr);
            if (res_norm < st.tolerance) {
              used = j + 1;
              done = true;
              break;
            }
            ++iteration;
          }
          // x += Z[:, :used] (H[:used,:used]^-1 g[:used])   (iterative_solvers.rs:175-183)
          double y[5];
          for (int i = used - 1; i >= 0; --i) {
            double v = g[i];
            for (int k = i + 1; k < used; ++k) v -= H[i][k] * y[k];
            y[i] = v / H[i][i];
          }
          for (int i = 0; i < used; ++i) S.axpy(y[i], Z.p + (size_t)i * nt, x.p, nt);
          if (done) break;
          S.matvec(x.p, nullptr, tmp.p);
          S.sub_to(b.p, tmp.p, r.p, nt);
          const double res_norm = absolute ? S.norm_max(r.p, nt) : S.norm2(r.p, nt) / beta;
          if (res_norm < st.tolerance) break;
        }
      } else {
        // ---- schwarz_ddm_solver, 100 iterations (iterative_solvers.rs:234-281)
        r.reserve(nt);
        tmp.reserve(nt);
        w.reserve(nt);
        FB_CUDA(cudaMemsetAsync(x.p, 0, nt * sizeof(double), stream));
        FB_CUDA(cudaMemcpyAsync(r.p, b.p, nt * sizeof(double), cudaMemcpyDeviceToDevice, stream));
        const bool absolute = st.tolerance_type == FR_TOL_ABSOLUTE;
        const double beta = absolute ? S.norm_max(r.p, nt) : S.norm2(r.p, nt);
        double res_norm = beta;
        uint64_t it = 0;
        while (res_norm > st.tolerance && it < 100) {
          S.precon(r.p, w.p);
          S.axpy(1.0, w.p, x.p, nt);
          S.matvec(x.p, nullptr, tmp.p);
          S.sub_to(b.p, tmp.p, r.p, nt);
          res_norm = absolute ? S.norm_max(r.p, nt) : S.norm2(r.p, nt) / beta;
          ++it;
          info.iterations += 1;
          info.last_residual = res_norm;
          emit(FR_EVENT_SOLVER_ITERATION, it, res_norm, progress_from_rel(res_norm, beta, st.tolerance), nullptr);
        }
      }
      FB_CUDA(cudaMemcpyAsync(hx.data(), x.p, nt * sizeof(double), cudaMemcpyDeviceToHost, stream));
      FB_CUDA(cudaStreamSynchronize(stream));
      for (size_t i = 0; i < n; ++i) point_coeff[i * n_cols + col] = hx[i];
      // coarse / naive solves write the recovered polynomial into the last `rank` rows (schwarz.rs:147-152)
      for (size_t k = 0; k < m; ++k) poly_coeff[k * n_cols + col] = hx[n + k];
    }
    info.matvecs = S.matvecs;
    info.solve_seconds = std::chrono::duration<double>(clk::now() - t_setup).count();
  } catch (...) {
    solver.reset();
    cudaStreamDestroy(setup_stream);
    throw;
  }
  solver.reset();
  cudaStreamDestroy(setup_stream);
  if (has_trend) {  // rbf.rs:579-581 and 599-601: public points = inverse transform; evaluators transform them again
    points.swap(mono_pts);
    apply_affine(aff, points.data(), n, dim, 1, kpts.data());
  }
  info.n_points = n;
  info.fit_seconds = std::chrono::duration<double>(clk::now() - t_start).count();
}

void fr_model::build_trend_transform() {
  const int d = dim, h = d + 1;
  auto eye = [&](double *mtx) {
    for (int i = 0; i < h * h; ++i) mtx[i] = 0.0;
    for (int i = 0; i < h; ++i) mtx[i * h + i] = 1.0;
  };
  auto mul = [&](const double *a, const double *b, double *c) {
    double t[16] = {0};
    for (int i = 0; i < h; ++i)
      for (int j = 0; j < h; ++j) {
        double v = 0.0;
        for (int k = 0; k < h; ++k) v += a[i * h + k] * b[k * h + j];
        t[i * h + j] = v;
      }
    std::copy(t, t + h * h, c);
  };
  double center[3] = {0, 0, 0};  // get_center: column means (rbf.rs:1300-1305)
  for (int k = 0; k < d; ++k) {
    double sum = 0.0;
    for (size_t i = 0; i < n; ++i) sum += points[i * d + k];
    center[k] = sum / (double)n;
  }
  double T[16], TB[16], S[16], R[16];
  eye(T);
  eye(TB);
  eye(S);
  eye(R);
  for (int k = 0; k < d; ++k) {
    T[k * h + d] = -center[k];
    TB[k * h + d] = center[k];
    S[k * h + k] = 1.0 / trend.ratios[k];
  }
  const double rad = 3.14159265358979323846 / 180.0;
  auto rot_z = [&](double a, double *mtx) {
    eye(mtx);
    mtx[0] = std::cos(a);
    mtx[1] = std::sin(a);
    mtx[h] = -std::sin(a);
    mtx[h + 1] = std::cos(a);
  };
  if (d == 2) {
    rot_z(-trend.angles[0] * rad, R);
  } else if (d == 3) {
    const double dipr = -trend.angles[0] * rad, dipdirr = -trend.angles[1] * rad, pitchr = -trend.angles[2] * rad;
    double RZ[16], RX[16], RZ2[16];
    rot_z(dipdirr, RZ);
    eye(RX);
    RX[1 * h + 1] = std::cos(dipr);
    RX[1 * h + 2] = std::sin(dipr);
    RX[2 * h + 1] = -std::sin(dipr);
    RX[2 * h + 2] = std::cos(dipr);
    rot_z(pitchr, RZ2);
    mul(RZ2, RX, R);
    mul(R, RZ, R);
  }
  double A[16];
  mul(TB, S, A);
  mul(A, R, A);
  mul(A, T, A);
  for (int i = 0; i < h; ++i)  // stored transposed: homogeneous row vectors multiply from the left
    for (int j = 0; j < h; ++j) aff[i * h + j] = A[j * h + i];
  // inverse by Gauss-Jordan with partial pivoting
  double w[16];
  std::copy(aff, aff + h * h, w);
  eye(aff_inv);
  for (int c = 0; c < h; ++c) {
    int piv = c;
    for (int r = c + 1; r < h; ++r)
      if (std::fabs(w[r * h + c]) > std::fabs(w[piv * h + c])) piv = r;
    FB_REQUIRE(w[piv * h + c] != 0.0, "singular global trend transform");
    if (piv != c)
      for (int k = 0; k < h; ++k) {
        std::swap(w[c * h + k], w[piv * h + k]);
        std::swap(aff_inv[c * h + k], aff_inv[piv * h + k]);
      }
    const double dgn = w[c * h + c];
    for (int k = 0; k < h; ++k) {
      w[c * h + k] /= dgn;
      aff_inv[c * h + k] /= dgn;
    }
    for (int r = 0; r < h; ++r) {
      if (r == c) continue;
      const double f = w[r * h + c];
      if (f == 0.0) continue;
      for (int k = 0; k < h; ++k) {
        w[r * h + k] -= f * w[c * h + k];
        aff_inv[r * h + k] -= f * aff_inv[c * h + k];
      }
    }
  }
}

void fr_model::apply_affine(const double *a, const double *in, size_t cnt, ptrdiff_t rs, ptrdiff_t cs, double *out) const {
  const int d = dim, h = d + 1;
  for (size_t i = 0; i < cnt; ++i) {
    double x[4] = {0, 0, 0, 1.0};
    for (int k = 0; k < d; ++k) x[k] = in[(ptrdiff_t)i * rs + (ptrdiff_t)k * cs];
    x[d] = 1.0;
    for (int j = 0; j < d; ++j) {
      double v = 0.0;
      for (int k = 0; k < h; ++k) v += x[k] * a[k * h + j];
      out[i * d + j] = v;
    }
  }
}

void fr_model::transform_extents(double *ext) const {  // rbf.rs:603-615 (bounding_box_corners :1307-1317)
  if (!has_trend) return;
  const int d = dim;
  double lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0};
  for (int i = 0; i < (1 << d); ++i) {
    double c[3] = {0, 0, 0}, tc[3] = {0, 0, 0};
    for (int j = 0; j < d; ++j) c[j] = ((i >> j) & 1) == 0 ? ext[j] : ext[d + j];
    apply_affine(aff, c, 1, d, 1, tc);
    for (int j = 0; j < d; ++j) {
      lo[j] = i == 0 ? tc[j] : std::min(lo[j], tc[j]);
      hi[j] = i == 0 ? tc[j] : std::max(hi[j], tc[j]);
    }
  }
  for (int j = 0; j < d; ++j) {
    ext[j] = lo[j];
    ext[d + j] = hi[j];
  }
}

// union of source and target extents (rbf.rs:640-668)
void fr_model::evaluation_extents(const double *target_ext, double *ext) const {
  for (int d = 0; d < dim; ++d) {
    double lo = points[d], hi = lo;
    for (size_t i = 0; i < n; ++i) {
      lo = std::min(lo, points[i * dim + d]);
      hi = std::max(hi, points[i * dim + d]);
    }
    ext[d] = std::min(lo, target_ext[d]);
    ext[dim + d] = std::max(hi, target_ext[dim + d]);
  }
  transform_extents(ext);
}

// evaluate the interpolant through a tree whose multipoles hold the point coefficients (rbf.rs:1180-1270): the targets
// are mapped through the trend and binned (bin_targets_dev), the leaf pass (after the downward pass unless `leaves`)
// leaves the kernel part in t->d_out / t->d_gout, and k_rbf_finish adds the rest into d_out / d_grads.  These may be
// t->d_out / t->d_gout themselves: the finish reads and writes only its own elements.  add_nugget: the targets are the
// source points, in their order.
void fr_model::eval_tree(fb_tree *t, const double *d_targets, size_t mt, ptrdiff_t rs, ptrdiff_t cs, bool leaves,
                         bool add_nugget, double *d_out, double *d_grads) {
  const int m = st.basis_size;
  if (m > 0 && d_poly.cap < (size_t)m * n_cols) {  // once per model: the coefficients never change after the fit
    d_poly.reserve((size_t)m * n_cols);
    FB_CUDA(cudaMemcpy(d_poly.p, poly_coeff.data(), (size_t)m * n_cols * sizeof(double), cudaMemcpyHostToDevice));
  }
  uint64_t bad = 0;
  TargetSet ts = t->bin_targets_dev(d_targets, mt, rs, cs, has_trend ? aff : nullptr, &bad);
  // every caller has just uploaded the point coefficients into this tree (set_weights semantics, rbf.rs:684, 836):
  // they stay resident, so repeated small-batch evaluate_targets calls move only the targets and the results
  if (!t->have_weights || t->nrhs != (int)n_cols)
    t->upload_weights(point_coeff.data(), n, n_cols, (ptrdiff_t)n_cols, 1);
  if (!leaves) t->downward(ts.cell_flag);
  t->leaf_pass(ts, d_grads != nullptr);
  RbfFinish f;
  f.m = mt;
  f.dim = dim;
  f.n_cols = (int)n_cols;
  f.basis = m;
  f.degree = st.polynomial_degree;
  f.targets = d_targets;
  f.t_rs = rs;
  f.t_cs = cs;
  f.vals = t->d_out.p;
  f.grads = d_grads ? t->d_gout.p : nullptr;
  if (add_nugget) {
    f.w = t->d_w_user.p;  // the point coefficients as uploaded, in input order
    f.nugget = st.nugget;
  }
  f.poly = m > 0 ? d_poly.p : nullptr;
  for (int d = 0; d < dim && m > 0; ++d) {
    f.translation[d] = translation[d];
    f.scale[d] = scale[d];
  }
  if (has_trend) {
    f.trend.on = 1;
    std::copy(aff, aff + 16, f.trend.a);
  }
  f.out = d_out;
  f.out_grads = d_grads;
  launch_rbf_finish(f, t->stream);
}

void fr_model::stage_targets(const double *targets, size_t mt, ptrdiff_t rs, ptrdiff_t cs, cudaStream_t s) {
  const size_t cnt = mt * dim;
  std::vector<double> rows;
  if (cs != 1 || rs != (ptrdiff_t)dim) {
    rows.resize(cnt);
    for (size_t i = 0; i < mt; ++i)
      for (int d = 0; d < dim; ++d) rows[i * dim + d] = targets[(ptrdiff_t)i * rs + (ptrdiff_t)d * cs];
    targets = rows.data();
  }
  d_targets.reserve(cnt);
  // from pageable memory: returns once the source has been read, so `rows` may go
  FB_CUDA(cudaMemcpyAsync(d_targets.p, targets, cnt * sizeof(double), cudaMemcpyHostToDevice, s));
}

void fr_model::eval_staged(fb_tree *t, size_t mt, bool leaves, bool add_nugget, double *out_vals, double *out_grads) {
  // the leaf pass zeroes these in place: reserved here, their addresses hold from now on
  t->d_out.reserve(mt * n_cols);
  if (out_grads) t->d_gout.reserve(mt * n_cols * dim);
  eval_tree(t, d_targets.p, mt, dim, 1, leaves, add_nugget, t->d_out.p, out_grads ? t->d_gout.p : nullptr);
  t->fetch_output(mt, out_grads != nullptr, out_vals, out_grads, (ptrdiff_t)n_cols, 1);
}

// ------------------------------------------------------------------------------------------ C ABI
template <class F>
static int fr_guarded(F &&f) {
  try {
    f();
    return FB_OK;
  } catch (const fb::Error &e) {
    set_last_error(e.what());
    return e.code;
  } catch (const std::exception &e) {
    set_last_error(e.what());
    return FB_ERR_CUDA;
  }
}

extern "C" {

void fr_settings_default(int32_t kernel_type, fr_settings *out) {
  if (!out) return;
  out->kernel_type = kernel_type;
  out->drift = FR_DRIFT_DEFAULT;
  out->spheroidal_order = 3;
  out->nugget = 0.0;
  out->base_range = 1.0;
  out->total_sill = 1.0;
  out->tolerance = 1e-6;
  out->tolerance_type = FR_TOL_RELATIVE;
}

void fr_params_default(int32_t kernel_type, fr_params *out) {
  if (!out) return;
  out->solver_type = FR_SOLVER_FGMRES;
  out->leaf_threshold = 1024;
  out->overlap_quota = 0.5;
  out->coarse_ratio = 0.125;
  out->coarse_threshold = 4096;
  const int order = kernel_type == FR_KERNEL_THIN_PLATE_SPLINE ? 9 : (kernel_type == FR_KERNEL_CUBIC ? 11 : 7);
  out->interpolation_order = (uint64_t)order;
  out->max_points_per_cell = 256;
  out->compression_type = FB_COMPRESSION_ACA;
  out->epsilon = std::pow(10.0, -order);
  out->eval_chunk_size = 1024;
  out->naive_solve_threshold = 4096;
  out->test_unique = 1;
}

int fr_fit(const double *points, size_t n, int dim, ptrdiff_t p_rs, ptrdiff_t p_cs, const double *values, size_t n_cols,
           ptrdiff_t v_rs, ptrdiff_t v_cs, const fr_settings *settings, const fr_params *params_or_null,
           fr_progress_cb cb_or_null, void *user, fr_model **out) {
  return fr_fit_trend(points, n, dim, p_rs, p_cs, values, n_cols, v_rs, v_cs, settings, params_or_null, nullptr,
                      cb_or_null, user, out);
}

// fr_fit_trend up to the solve, shared with fr_ddm_level_solve: settings, params and trend checked, the points (and the
// values, if any) copied and freed of duplicates (rbf.rs:341-359)
static void init_model(fr_model &M, const double *points, size_t n, int dim, ptrdiff_t p_rs, ptrdiff_t p_cs,
                       const double *values, size_t n_cols, ptrdiff_t v_rs, ptrdiff_t v_cs, const fr_settings *settings,
                       const fr_params *params_or_null, const fr_global_trend *trend_or_null) {
  FB_REQUIRE(dim >= 1 && dim <= 3, "Unsupported number of dimensions: " + std::to_string(dim));  // rbf.rs:329-333
  M.dim = dim;
  if (trend_or_null) {
    FB_REQUIRE(trend_or_null->dim == dim, "GlobalTrend variant does not match the dimensionality of the points");
    for (int d = 0; d < dim; ++d) FB_REQUIRE(trend_or_null->ratios[d] > 0.0, "GlobalTrend ratios must be positive");
    M.has_trend = true;
    M.trend = *trend_or_null;
  }
  std::string err;
  FB_REQUIRE(resolve_settings(*settings, dim, M.st, err), err);
  FB_REQUIRE(make_kparams(M.st.kparams, M.kp), "unknown kernel");
  if (params_or_null)
    M.params = *params_or_null;
  else
    fr_params_default(settings->kernel_type, &M.params);
  std::vector<double> pts(n * dim), vals(n * n_cols);
  for (size_t i = 0; i < n; ++i) {
    for (int d = 0; d < dim; ++d) pts[i * dim + d] = points[(ptrdiff_t)i * p_rs + (ptrdiff_t)d * p_cs];
    for (size_t c = 0; c < n_cols; ++c) vals[i * n_cols + c] = values[(ptrdiff_t)i * v_rs + (ptrdiff_t)c * v_cs];
  }
  M.n_in = n;
  const bool verbose = std::getenv("FB_TIMING") != nullptr;
  const auto t_dedup = std::chrono::steady_clock::now();
  if (M.params.test_unique) {  // rbf.rs:341-359
    std::vector<int64_t> keep = remove_duplicates(pts.data(), n, dim, M.kp);
    if (keep.size() != n) {
      M.emit(FR_EVENT_DUPLICATES_REMOVED, n - keep.size(), 0, 0, nullptr);
      std::vector<double> p2(keep.size() * dim), v2(keep.size() * n_cols);
      for (size_t k = 0; k < keep.size(); ++k) {
        std::copy(&pts[keep[k] * dim], &pts[keep[k] * dim] + dim, &p2[k * dim]);
        std::copy(&vals[keep[k] * n_cols], &vals[keep[k] * n_cols] + n_cols, &v2[k * n_cols]);
      }
      pts.swap(p2);
      vals.swap(v2);
    }
  }
  M.points.swap(pts);
  M.values.swap(vals);
  M.n = M.points.size() / dim;
  M.n_cols = n_cols;
  if (verbose)
    fprintf(stderr, "[fr_fit] %-28s %8.3f s\n", "copy + remove_duplicates",
            std::chrono::duration<double>(std::chrono::steady_clock::now() - t_dedup).count());
}

int fr_fit_trend(const double *points, size_t n, int dim, ptrdiff_t p_rs, ptrdiff_t p_cs, const double *values,
                 size_t n_cols, ptrdiff_t v_rs, ptrdiff_t v_cs, const fr_settings *settings,
                 const fr_params *params_or_null, const fr_global_trend *trend_or_null, fr_progress_cb cb_or_null,
                 void *user, fr_model **out) {
  if (!out) return FB_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  fr_model *M = nullptr;
  const int rc = fr_guarded([&] {
    FB_REQUIRE(points && values && settings && n > 0 && n_cols > 0, "points, values and settings are required");
    M = new fr_model();
    M->cb = cb_or_null;
    M->cb_user = user;
    init_model(*M, points, n, dim, p_rs, p_cs, values, n_cols, v_rs, v_cs, settings, params_or_null, trend_or_null);
    M->fit();
    M->info.n_duplicates = n - M->n;
    char msg[256];
    snprintf(msg, sizeof(msg), "Took %.3fs to solve RBF for %zu points (%llu iterations, %llu FMM matvecs)",
             M->info.fit_seconds, M->n, (unsigned long long)M->info.iterations, (unsigned long long)M->info.matvecs);
    M->emit(FR_EVENT_MESSAGE, 0, 0, 0, msg);
  });
  if (rc != FB_OK) {
    delete M;
    return rc;
  }
  *out = M;
  return FB_OK;
}

void fr_free(fr_model *m) { delete m; }

int fr_get_info(const fr_model *m, fr_model_info *info) {
  if (!m || !info) return FB_ERR_INVALID_ARGUMENT;
  *info = m->info;
  return FB_OK;
}

int fr_source_points(const fr_model *m, double *points_out, double *values_out) {
  if (!m) return FB_ERR_INVALID_ARGUMENT;
  if (points_out) std::copy(m->points.begin(), m->points.end(), points_out);
  if (values_out) std::copy(m->values.begin(), m->values.end(), values_out);
  return FB_OK;
}

int fr_coefficients(const fr_model *m, double *point_out, double *poly_out) {
  if (!m) return FB_ERR_INVALID_ARGUMENT;
  if (point_out) std::copy(m->point_coeff.begin(), m->point_coeff.end(), point_out);
  if (poly_out) std::copy(m->poly_coeff.begin(), m->poly_coeff.end(), poly_out);
  return FB_OK;
}

int fr_get_state(const fr_model *m, fr_model_state *out) {
  if (!m || !out) return FB_ERR_INVALID_ARGUMENT;
  std::memset(out, 0, sizeof(*out));
  out->settings.kernel_type = m->st.kernel_type;
  out->settings.drift = m->st.drift;
  out->settings.spheroidal_order = m->st.spheroidal_order;
  out->settings.nugget = m->st.nugget;
  out->settings.base_range = m->st.base_range;
  out->settings.total_sill = m->st.total_sill;
  out->settings.tolerance = m->st.tolerance;
  out->settings.tolerance_type = m->st.tolerance_type;
  out->params = m->params;
  out->basis_size = m->st.basis_size;
  out->polynomial_degree = m->st.polynomial_degree;
  for (int d = 0; d < m->dim && d < (int)m->translation.size(); ++d) {
    out->translation_factor[d] = m->translation[d];
    out->scale_factor[d] = m->scale[d];
  }
  out->has_trend = m->has_trend ? 1 : 0;
  if (m->has_trend) {
    std::copy(m->aff, m->aff + 16, out->affine_transform);
    std::copy(m->aff_inv, m->aff_inv + 16, out->inverse_transform);
  }
  return FB_OK;
}

int fr_model_restore(const double *points, size_t n, int dim, const double *values, size_t n_cols,
                     const double *point_coefficients, const double *poly_coefficients_or_null,
                     const fr_model_state *state, fr_progress_cb cb_or_null, void *user, fr_model **out) {
  if (!out) return FB_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  fr_model *M = nullptr;
  const int rc = fr_guarded([&] {
    FB_REQUIRE(points && values && point_coefficients && state && n > 0 && n_cols > 0, "incomplete model state");
    FB_REQUIRE(dim >= 1 && dim <= 3, "Unsupported number of dimensions: " + std::to_string(dim));
    M = new fr_model();
    M->dim = dim;
    M->cb = cb_or_null;
    M->cb_user = user;
    std::string err;
    FB_REQUIRE(resolve_settings(state->settings, dim, M->st, err), err);
    FB_REQUIRE(M->st.basis_size == state->basis_size && M->st.polynomial_degree == state->polynomial_degree,
               "basis_size / polynomial_degree do not match the kernel, drift and dimension of the model");
    FB_REQUIRE(M->st.basis_size == 0 || poly_coefficients_or_null, "polynomial coefficients are required");
    FB_REQUIRE(make_kparams(M->st.kparams, M->kp), "unknown kernel");
    M->params = state->params;
    M->n = M->n_in = n;
    M->n_cols = n_cols;
    M->points.assign(points, points + n * dim);
    M->values.assign(values, values + n * n_cols);
    M->point_coeff.assign(point_coefficients, point_coefficients + n * n_cols);
    const size_t m = (size_t)M->st.basis_size;
    if (m) M->poly_coeff.assign(poly_coefficients_or_null, poly_coefficients_or_null + m * n_cols);
    M->translation.assign(state->translation_factor, state->translation_factor + dim);
    M->scale.assign(state->scale_factor, state->scale_factor + dim);
    if (state->has_trend) {  // evaluators transform the stored (original-space) points again (rbf.rs:599-601)
      M->has_trend = true;
      std::copy(state->affine_transform, state->affine_transform + 16, M->aff);
      std::copy(state->inverse_transform, state->inverse_transform + 16, M->aff_inv);
      M->kpts.resize(n * dim);
      M->apply_affine(M->aff, M->points.data(), n, dim, 1, M->kpts.data());
    }
    M->info = fr_model_info{};
    M->info.n_points = n;
    M->info.n_cols = n_cols;
    M->info.basis_size = m;
    M->info.dim = (uint64_t)dim;
  });
  if (rc != FB_OK) {
    delete M;
    return rc;
  }
  *out = M;
  return FB_OK;
}

int fr_evaluate(fr_model *m, const double *targets, size_t n_targets, ptrdiff_t t_rs, ptrdiff_t t_cs, double *out_vals,
                double *out_grads_or_null) {
  return fr_guarded([&] {
    FB_REQUIRE(m && targets && out_vals && n_targets > 0, "model, targets and output are required");
    // as fr_evaluate_device, on the legacy default stream (device_extents waits for it)
    m->stage_targets(targets, n_targets, t_rs, t_cs, nullptr);
    double ext[6];
    device_extents(m->d_targets.p, n_targets, m->dim, m->dim, 1, m->d_ext, nullptr, ext);
    m->evaluation_extents(ext, ext);
    auto tree = m->transient_tree(false, ext);  // non-sparse adaptive tree (rbf.rs:677-681)
    m->eval_staged(tree.get(), n_targets, false, false, out_vals, out_grads_or_null);
  });
}

int fr_evaluate_at_source(fr_model *m, int add_nugget, double *out_vals) {
  return fr_guarded([&] {
    FB_REQUIRE(m && out_vals, "model and output are required");
    auto tree = m->transient_tree(true, nullptr);  // rbf.rs:777-781
    m->stage_targets(m->points.data(), m->n, m->dim, 1, tree->stream);
    m->eval_staged(tree.get(), m->n, false, add_nugget != 0, out_vals, nullptr);
  });
}

int fr_build_evaluator(fr_model *m, const double *extents_or_null) {
  return fr_guarded([&] {
    FB_REQUIRE(m, "model required");
    double ext[6];
    if (extents_or_null) {
      std::copy(extents_or_null, extents_or_null + 2 * m->dim, ext);
      m->transform_extents(ext);
    }
    m->evaluator = m->transient_tree(false, extents_or_null ? ext : nullptr);  // rbf.rs:830-838
    fb_tree *t = m->evaluator.get();
    t->downward(t->d_flag_all.p);
    FB_CUDA(cudaStreamSynchronize(t->stream));
  });
}

int fr_evaluate_targets(fr_model *m, const double *targets, size_t n_targets, ptrdiff_t t_rs, ptrdiff_t t_cs,
                        double *out_vals, double *out_grads_or_null) {
  return fr_guarded([&] {
    FB_REQUIRE(m && targets && out_vals && n_targets > 0, "model, targets and output are required");
    FB_REQUIRE(m->evaluator != nullptr, "build_evaluator must be called before evaluate_targets");
    fb_tree *t = m->evaluator.get();
    m->stage_targets(targets, n_targets, t_rs, t_cs, t->stream);
    m->eval_staged(t, n_targets, true, false, out_vals, out_grads_or_null);
  });
}

// the arguments of fr_evaluate_device / fr_evaluate_targets_device (pointer checks on `device`)
static void require_device_eval_args(const fr_model *m, const double *d_targets, size_t n_targets, ptrdiff_t t_rs,
                                     ptrdiff_t t_cs, double *d_out, double *d_grads, int device) {
  require_device_matrix(d_targets, n_targets, m->dim, t_rs, t_cs, device, "target_points");
  require_device_matrix(d_out, n_targets, m->n_cols, (ptrdiff_t)m->n_cols, 1, device, "output");
  if (d_grads)
    require_device_matrix(d_grads, n_targets, m->n_cols * m->dim, (ptrdiff_t)(m->n_cols * m->dim), 1, device,
                          "gradient output");
}

int fr_evaluate_device(fr_model *m, const double *d_targets, size_t n_targets, ptrdiff_t t_rs, ptrdiff_t t_cs,
                       double *d_out, double *d_grads_or_null, void *stream) {
  return fr_guarded([&] {
    FB_REQUIRE(m && d_targets && d_out && n_targets > 0, "model, targets and output are required");
    int device = 0;
    FB_CUDA(cudaGetDevice(&device));
    require_device_eval_args(m, d_targets, n_targets, t_rs, t_cs, d_out, d_grads_or_null, device);
    // the target part of the tree extents is reduced on the device
    double ext[6];
    device_extents(d_targets, n_targets, m->dim, t_rs, t_cs, m->d_ext, (cudaStream_t)stream, ext);
    m->evaluation_extents(ext, ext);
    auto tree = m->transient_tree(false, ext);
    StreamJoin sj((cudaStream_t)stream, tree->stream);
    m->eval_tree(tree.get(), d_targets, n_targets, t_rs, t_cs, false, false, d_out, d_grads_or_null);
    sj.join();
    FB_CUDA(cudaStreamSynchronize(tree->stream));  // the tree is freed on return
  });
}

int fr_evaluate_targets_device(fr_model *m, const double *d_targets, size_t n_targets, ptrdiff_t t_rs, ptrdiff_t t_cs,
                               double *d_out, double *d_grads_or_null, void *stream) {
  return fr_guarded([&] {
    FB_REQUIRE(m && d_targets && d_out && n_targets > 0, "model, targets and output are required");
    FB_REQUIRE(m->evaluator != nullptr, "build_evaluator must be called before evaluate_targets");
    fb_tree *t = m->evaluator.get();
    FB_CUDA(cudaSetDevice(t->device));
    require_device_eval_args(m, d_targets, n_targets, t_rs, t_cs, d_out, d_grads_or_null, t->device);
    StreamJoin sj((cudaStream_t)stream, t->stream);
    m->eval_tree(t, d_targets, n_targets, t_rs, t_cs, true, false, d_out, d_grads_or_null);
    sj.join();
  });
}

// the meshes of fr_isosurface_extract (side kIsoOpen) or the solids of fr_isosurface_extract_solid
static void extract_meshes(fr_model *m, const double *extents, const uint64_t *resolution, const double *isovalues,
                           int n_iso, int column, int refine, int side, fr_isosurface **out) {
  FB_REQUIRE(out, "output handle required");
  *out = nullptr;
  FB_REQUIRE(m, "model required");
  FB_REQUIRE(m->dim == 3, "isosurfaces need a 3-D model, this one is " + std::to_string(m->dim) + "-D");
  const IsoLattice L = iso_lattice(extents, resolution);
  FB_REQUIRE(isovalues && n_iso >= 1, "at least one isovalue is required");
  for (int i = 0; i < n_iso; ++i) FB_REQUIRE(std::isfinite(isovalues[i]), "isovalues must be finite");
  FB_REQUIRE(column >= 0 && (size_t)column < m->n_cols,
             "column " + std::to_string(column) + " is out of range for " + std::to_string(m->n_cols) +
                 " value column(s)");
  using clk = std::chrono::steady_clock;
  auto ms = [](clk::time_point a, clk::time_point b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
  const auto t0 = clk::now();
  // one transient tree over the union of the lattice and the source points, as fr_evaluate_device; the lattice, every
  // refinement batch and the normals are served from its leaf pass
  double ext[6] = {L.lo[0], L.lo[1], L.lo[2], L.hi[0], L.hi[1], L.hi[2]};
  m->evaluation_extents(ext, ext);
  auto tree = m->transient_tree(false, ext);
  fb_tree *t = tree.get();
  t->downward(t->d_flag_all.p);
  const cudaStream_t s = t->stream;
  const uint64_t nodes = L.nodes();
  const size_t nc = m->n_cols;
  DBuf<double> xyz, vals;
  xyz.reserve(3 * nodes);
  vals.reserve(nodes * nc);
  iso_lattice_points(L, xyz.p, s);
  m->eval_tree(t, xyz.p, nodes, 3, 1, true, false, vals.p, nullptr);
  IsoScratch w;
  const double *v = vals.p + column;  // column `column` of the lattice values, stride n_cols
  const uint64_t bad = iso_first_nonfinite(v, nc, nodes, w, s);
  FB_REQUIRE(bad == nodes, "the interpolant is not finite at lattice node " + std::to_string(bad));
  const auto t1 = clk::now();
  auto h = std::make_unique<fr_isosurface>();
  h->device = t->device;
  for (int i = 0; i < n_iso; ++i) {
    h->surf.push_back(std::make_unique<IsoSurface>());
    h->surf.back()->iso = isovalues[i];
    h->surf.back()->side = side;
    iso_extract(v, nc, L, w, *h->surf.back(), s);
  }
  FB_CUDA(cudaStreamSynchronize(s));
  const auto t2 = clk::now();
  if (refine) {
    const IsoEval eval = [&](const double *pts, size_t cnt, double *out_vals) {
      m->eval_tree(t, pts, cnt, 3, 1, true, false, out_vals, nullptr);
    };
    for (auto &f : h->surf) iso_refine(v, nc, L, (int)nc, column, eval, w, *f, s);
  }
  if (side != kIsoOpen)  // from the final vertex positions
    for (auto &f : h->surf) iso_measure(L, w, *f, s);
  FB_CUDA(cudaStreamSynchronize(s));
  const auto t3 = clk::now();
  DBuf<double> gv, gg;
  for (auto &f : h->surf) {
    if (f->nv) {
      gv.reserve(f->nv * nc);
      gg.reserve(f->nv * nc * 3);
      m->eval_tree(t, f->verts.p, f->nv, 3, 1, true, false, gv.p, gg.p);
    }
    iso_normals(gg.p, (int)nc, column, L, *f, s);
  }
  FB_CUDA(cudaStreamSynchronize(s));
  const auto t4 = clk::now();
  h->ms[0] = ms(t0, t1);
  h->ms[1] = ms(t1, t2);
  h->ms[2] = ms(t2, t3);
  h->ms[3] = ms(t3, t4);
  *out = h.release();
}

int fr_isosurface_extract(fr_model *m, const double *extents, const uint64_t *resolution, const double *isovalues,
                          int n_iso, int column, int refine, fr_isosurface **out) {
  return fr_guarded([&] { extract_meshes(m, extents, resolution, isovalues, n_iso, column, refine, kIsoOpen, out); });
}

int fr_isosurface_extract_solid(fr_model *m, const double *extents, const uint64_t *resolution,
                                const double *isovalues, int n_iso, int column, int refine, int side,
                                fr_isosurface **out) {
  return fr_guarded([&] {
    if (out) *out = nullptr;
    FB_REQUIRE(side == 0 || side == 1, "side must be 0 (below) or 1 (above)");
    extract_meshes(m, extents, resolution, isovalues, n_iso, column, refine, side, out);
  });
}

// x = A^-1 b for a dense symmetric matrix through the subdomain machinery on a one-domain level without special points
// (k_cholesky and k_dom_solve; from n = 512 on k_chol_big_* and the spread solve; indefinite matrices take the fallback
// of factorise_pool and k_dom_solve): the entry point of the reference's reproducible known-answer tests
// linalg.rs:638-764 (make_spd) against the device factorisation.
int fr_dense_spd_solve(const double *a, int n, const double *b, int nrhs, double *x, int *used_fallback) {
  return fr_guarded([&] {
    FB_REQUIRE(a && b && x && n > 0 && nrhs > 0, "fr_dense_spd_solve: bad arguments");
    fr_model dummy;
    DeviceSolver S(dummy, nullptr);
    cudaStream_t stream = nullptr;
    FB_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    S.s = stream;
    S.n = (size_t)n;
    S.m = 0;
    S.nt = (size_t)n;
    try {
      LevelDev lv;
      std::vector<long long> pt_ptr{0, n}, zero{0};
      std::vector<int> idx(n), rank{0};
      std::vector<uint8_t> mask(n, 1);
      for (int i = 0; i < n; ++i) idx[i] = i;
      lv.n_domains = 1;
      lv.max_n = lv.max_mm = (size_t)n;
      lv.pt_ptr.upload(pt_ptr, stream);
      lv.q_off.upload(zero, stream);
      lv.l_off.upload(zero, stream);
      lv.s_off.upload(zero, stream);
      lv.rank.upload(rank, stream);
      lv.pt_idx.upload(idx, stream);
      lv.pt_mask.upload(mask, stream);
      lv.qpool.reserve(1);
      lv.lpool.reserve((size_t)n * n);
      DomainTable &t = lv.tab;
      t.n_domains = 1;
      t.pt_ptr = lv.pt_ptr.p;
      t.pt_idx = lv.pt_idx.p;
      t.pt_mask = lv.pt_mask.p;
      t.rank = lv.rank.p;
      t.q_off = lv.q_off.p;
      t.l_off = lv.l_off.p;
      t.s_off = lv.s_off.p;
      auto upload_a = [&](size_t) {
        FB_CUDA(cudaMemcpyAsync(lv.lpool.p, a, (size_t)n * n * sizeof(double), cudaMemcpyHostToDevice, stream));
      };
      upload_a(0);
      S.factorise_pool(lv, std::vector<int>{n}, std::vector<long long>{0}, upload_a, stream);
      if (used_fallback) *used_fallback = lv.n_fallback;
      DBuf<double> db, dx;
      db.reserve((size_t)n);
      dx.reserve((size_t)n);
      std::vector<double> col(n);
      for (int r = 0; r < nrhs; ++r) {
        for (int i = 0; i < n; ++i) col[i] = b[(size_t)i * nrhs + r];
        FB_CUDA(cudaMemcpyAsync(db.p, col.data(), (size_t)n * sizeof(double), cudaMemcpyHostToDevice, stream));
        S.solve_level(lv, db.p, dx.p, 1, 0, stream);
        FB_CUDA(cudaMemcpyAsync(col.data(), dx.p, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, stream));
        FB_CUDA(cudaStreamSynchronize(stream));
        for (int i = 0; i < n; ++i) x[(size_t)i * nrhs + r] = col[i];
      }
    } catch (...) {
      cudaStreamDestroy(stream);
      throw;
    }
    cudaStreamDestroy(stream);
  });
}

// One DDM level's subdomain solves on nvec residual vectors (n_kept + basis_size each, row after row), set up as fr_fit
// sets up the solve (duplicate removal, scaling, hierarchy or single dense domain, factorisations) but without an FMM
// tree: out[v] = solve_level(level, coarse level ? mode 1 : mode 0, add_poly) of res[v], out zeroed first.
int fr_ddm_level_solve(const double *points, size_t n, int dim, const fr_settings *settings, const fr_params *params_or_null,
                       int level, int add_poly, const double *res, int nvec, double *out, uint64_t *n_fallback_or_null,
                       uint64_t *domain_ranks_or_null) {
  return fr_guarded([&] {
    FB_REQUIRE(points && settings && res && out && n > 0 && nvec > 0, "fr_ddm_level_solve: bad arguments");
    fr_model M;
    init_model(M, points, n, dim, dim, 1, nullptr, 0, 0, 0, settings, params_or_null, nullptr);
    std::vector<double> mono_pts;
    TreePtr tree(nullptr, fb_tree_free);
    cudaStream_t setup_stream = nullptr;
    FB_CUDA(cudaStreamCreateWithFlags(&setup_stream, cudaStreamNonBlocking));
    std::unique_ptr<DeviceSolver> solver(new DeviceSolver(M, nullptr));
    try {
      DeviceSolver &S = *solver;
      setup_solve(M, S, setup_stream, false, mono_pts, tree);
      FB_REQUIRE(level >= 0 && (size_t)level < M.ddm.size(),
                 "level " + std::to_string(level) + " out of range: the hierarchy has " + std::to_string(M.ddm.size()));
      const LevelDev &lv = *S.levels[level];
      const bool coarse = (size_t)level + 1 == M.ddm.size();
      if (n_fallback_or_null) *n_fallback_or_null = (uint64_t)lv.n_fallback;
      if (domain_ranks_or_null)
        for (size_t d = 0; d < M.ddm[level].domains.size(); ++d) domain_ranks_or_null[d] = M.ddm[level].domains[d].rank;
      const size_t nt = S.nt;
      DBuf<double> dr, dx;
      dr.reserve(nt);
      dx.reserve(nt);
      for (int v = 0; v < nvec; ++v) {
        FB_CUDA(cudaMemcpyAsync(dr.p, res + (size_t)v * nt, nt * sizeof(double), cudaMemcpyHostToDevice, S.s));
        FB_CUDA(cudaMemsetAsync(dx.p, 0, nt * sizeof(double), S.s));
        S.solve_level(lv, dr.p, dx.p, coarse ? 1 : 0, add_poly, S.s);
        FB_CUDA(cudaMemcpyAsync(out + (size_t)v * nt, dx.p, nt * sizeof(double), cudaMemcpyDeviceToHost, S.s));
        FB_CUDA(cudaStreamSynchronize(S.s));
      }
    } catch (...) {
      solver.reset();
      cudaStreamDestroy(setup_stream);
      throw;
    }
    solver.reset();
    cudaStreamDestroy(setup_stream);
  });
}

// monomial basis of `n` points (polynomials.rs:15-62), host only: degree -1 .. 2, columns [1, x, y, z, x^2, xy, xz, y^2,
// yz, z^2]; out is n x basis row-major, basis = C(dim + degree, degree) is returned through basis_out
int fr_evaluate_monomials(const double *points, size_t n, int dim, int degree, const double *translation,
                          const double *scale, double *out, int *basis_out) {
  if (!points || dim < 1 || dim > 3 || degree < -1 || degree > 2) return FB_ERR_INVALID_ARGUMENT;
  int basis = 0;
  if (degree == 0) basis = 1;
  if (degree == 1) basis = 1 + dim;
  if (degree == 2) basis = (dim + 1) * (dim + 2) / 2;
  if (basis_out) *basis_out = basis;
  if (!out || basis == 0) return FB_OK;
  std::vector<double> tr(dim, 0.0), sc(dim, 1.0);
  evaluate_monomials(points, nullptr, n, dim, degree, basis, translation ? translation : tr.data(),
                     scale ? scale : sc.data(), out);
  return FB_OK;
}

int fr_ddm_level(const fr_model *m, int level, uint64_t *n_domains, uint64_t *n_level_points, uint64_t *level_points,
                 uint64_t *dom_ptr, uint64_t *dom_idx, uint8_t *dom_internal) {
  if (!m || level < 0 || level >= (int)m->ddm.size()) return FB_ERR_INVALID_ARGUMENT;
  const LevelHost &lh = m->ddm[level];
  if (n_domains) *n_domains = lh.domains.size();
  if (n_level_points) *n_level_points = lh.point_indices.size();
  if (level_points)
    for (size_t i = 0; i < lh.point_indices.size(); ++i) level_points[i] = (uint64_t)lh.point_indices[i];
  uint64_t off = 0;
  for (size_t d = 0; d < lh.domains.size(); ++d) {
    if (dom_ptr) dom_ptr[d] = off;
    const DomainHost &dh = lh.domains[d];
    for (size_t i = 0; i < dh.idx.size(); ++i) {
      if (dom_idx) dom_idx[off + i] = (uint64_t)dh.idx[i];
      if (dom_internal) dom_internal[off + i] = i < dh.mask.size() ? dh.mask[i] : 0;
    }
    off += dh.idx.size();
  }
  if (dom_ptr) dom_ptr[lh.domains.size()] = off;
  return FB_OK;
}

}  // extern "C"
