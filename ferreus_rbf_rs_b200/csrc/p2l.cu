// Downward-pass P2L on the tensor grid of the target cell's Chebyshev nodes, optionally fused with the M2P transpose
// (FP64 FMA-pipe bound).  Reference: particle_to_local bbfmm.rs:1001-1048, multipole_to_particle :1254-1355.
#include "fmm.h"

#include <algorithm>
#include <cstdlib>

namespace fb {

// ======================================================================================================
// P2L on the tensor grid of the target cell's Chebyshev nodes (bbfmm.rs:1001-1048).  The targets are the p^d
// nodes of the cell, so r^2 = (dx2[i0] + dy2[i1]) + dz2[i2] with the squared axis offsets tabulated once per
// source: a thread owns one (i0, i1) column of nodes (p accumulators per right-hand side in registers) and a
// slice of the source tile; per pair that is 1 add + kernel + 1 FMA instead of 6 + kernel + 1.  X-list leaves are
// never adjacent to the cell, so r^2 > 0.  Slices are summed through shared memory in a fixed order, one CTA per
// cell: deterministic, no atomics.
// ======================================================================================================
constexpr int kP2LTileMax = 256;  // sources per staged tile (upper bound; one tile point per thread)
constexpr int kP2LJB = 4;          // sources in flight per thread (independent kernel evaluations)
constexpr size_t kP2LFuseBytes = 48 * 1024;  // shared-memory budget of the fused M2P partial sums (x2 when NR > 1:
                                             // those instantiations run one CTA per SM anyway)

template <int FAM, int NR, int PREG, bool FAST, bool FUSE>
__global__ void __launch_bounds__(256, (NR * PREG <= 8) ? 3 : ((NR * PREG <= (FUSE ? 8 : 16)) ? 2 : 1)) k_p2l_grid(const P2LArgs a, const int nslices, const int cols, const int T) {
  const int ci = blockIdx.x;
  const int c = a.cells[ci];
  // P2L is wanted when the cell has targets below it; the fused M2P half when any X-list point is a target (a
  // subset-of-sources target set carries exclusive target counts over the sorted positions)
  const bool need_p2l = a.cell_flag[c] != 0;
  // partitioned tree: one rank applies the M2P half of a cell (the owner of its first point); the others that hold
  // targets below the cell run the P2L half alone
  const bool do_m2p = FUSE && (a.cell_ptb == nullptr || (a.cell_ptb[c] >= a.own_lo && a.cell_ptb[c] < a.own_hi));
  if (!FUSE) {
    if (!need_p2l) return;
  } else if (!need_p2l) {
    if (a.tgt_prefix == nullptr) return;  // every source is a target only when every cell is flagged
    bool any = false;
    for (long long e = a.x_ptr[ci]; e < a.x_ptr[ci + 1] && !any; ++e)
      any = a.tgt_prefix[a.x_begin[e] + a.x_count[e]] != a.tgt_prefix[a.x_begin[e]];
    if (!any) return;
  }
  const int tid = threadIdx.x, nt = blockDim.x;
  const int p = a.p, P = a.P, dim = a.dim;
  extern __shared__ double sm[];
  double *tab = sm;                                 // [dim][T][PREG]
  double *wts = sm + (size_t)dim * T * PREG;        // [NR][T]
  double *part = wts + (size_t)NR * T;              // FUSE: [NR][cols][T + 1] per-column M2P partial sums of the tile points
  const int q = tid % cols, slice = tid / cols;
  const bool active = slice < nslices;
  // FUSE: the kernel matrix of (cell nodes) x (X-leaf points) is the transpose of the M2P matrix of (W-list targets) x
  // (cell nodes) — X is the transpose of W (linear_tree.rs:330-395) and the kernels are symmetric — so every value
  // computed here also feeds out[point] += K * M_cell[node].  A thread sums its column's nodes into a per-(column,
  // point) slot of shared memory (row stride T + 1: conflict-free for both the column-wise writes and the point-wise
  // reads); at the end of the tile thread j adds up the columns of point j and issues one RED per (point, rhs).
  const int Ts = T + 1;
  double mreg[FUSE ? NR : 1][FUSE ? PREG : 1];
  if (FUSE) {
#pragma unroll
    for (int r = 0; r < NR; ++r)
#pragma unroll
      for (int il = 0; il < PREG; ++il)
        mreg[r][il] = (active && il < p) ? a.mult[((size_t)c * a.nrhs + a.rhs0 + r) * coef_stride(P) + q * p + il] *
                                               kernel_weight_scale<FAM, FAST>()
                                         : 0.0;
  }
  const int i0 = dim == 3 ? q / p : q, i1 = dim == 3 ? q % p : 0;
  __shared__ double ncoord[3 * PREG];  // node coordinates of the cell per axis
  if (tid < dim * p) {
    const int d = tid / p, i = tid - d * p;
    const double cd = d == 0 ? a.ccx[c] : (d == 1 ? a.ccy[c] : a.ccz[c]);
    ncoord[d * PREG + i] = cd + a.chalf[c] * a.nodes[i];
  }
  const double *tabA = tab, *tabB = tab + (size_t)T * PREG, *tabL = tab + (size_t)(dim - 1) * T * PREG;
  double acc[NR][PREG];
#pragma unroll
  for (int r = 0; r < NR; ++r)
#pragma unroll
    for (int i = 0; i < PREG; ++i) acc[r][i] = 0.0;

  // cursor over the tiles of the merged X ranges; the next tile's coordinates and weights are fetched into
  // registers while the current one is consumed
  long long e = a.x_ptr[ci];
  const long long e_end = a.x_ptr[ci + 1];
  int rb = 0, rn = 0, c0 = 0;
  if (e < e_end) {
    rb = a.x_begin[e];
    rn = a.x_count[e];
  }
  // tile item t = tid + k * nt (k = 0, 1) is the table row of axis d = t / T, point j = t % T; items past dim * T
  // do not exist (T <= nt, so two items per thread cover dim * T <= 3 nt... see the launch: dim * T <= 2 nt)
  double pc[2] = {0.0, 0.0}, pw[NR];
  int it_d[2], it_j[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int t = tid + k * nt;
    it_d[k] = (t >= T) + (t >= 2 * T) + (t >= 3 * T);
    it_j[k] = t - it_d[k] * T;
  }
  auto prefetch = [&](int &m, int &base) {
    m = 0;
    if (e >= e_end) return;
    m = min(T, rn - c0);
    base = rb + c0;
#pragma unroll
    for (int k = 0; k < 2; ++k)
      if (it_d[k] < dim && it_j[k] < m)
        pc[k] = it_d[k] == 0 ? a.sx[base + it_j[k]] : (it_d[k] == 1 ? a.sy[base + it_j[k]] : a.sz[base + it_j[k]]);
#pragma unroll
    for (int r = 0; r < NR; ++r)
      pw[r] = tid < m ? a.w[(size_t)(a.rhs0 + r) * a.n + base + tid] * kernel_weight_scale<FAM, FAST>() : 0.0;
    c0 += T;
    if (c0 >= rn) {
      ++e;
      c0 = 0;
      if (e < e_end) {
        rb = a.x_begin[e];
        rn = a.x_count[e];
      }
    }
  };
  // FUSE: the M2P sums of a finished tile are flushed by the threads that do not build the next tile's tables
  // more than one row, concurrently with that build, so the flush costs no barrier of its own
  const int n_flush = nt - max(0, dim * T - nt);  // threads with at most one table row to build
  auto flush_m2p = [&](int first, int step, int m_done, int base_done) {
    for (int j = first; j < m_done; j += step) {
      const uint32_t row32 = a.out_row[base_done + j];
      if (row32 == 0xFFFFFFFFu) continue;
      const size_t row = row32;
#pragma unroll
      for (int r = 0; r < NR; ++r) {
        const double *pp = part + (size_t)r * cols * Ts + j;
        double v0 = 0.0, v1 = 0.0;
        int qq = 0;
        for (; qq + 1 < cols; qq += 2) {
          v0 += pp[(size_t)qq * Ts];
          v1 += pp[(size_t)(qq + 1) * Ts];
        }
        if (qq < cols) v0 += pp[(size_t)qq * Ts];
        atomicAdd(a.out + row * a.nrhs + a.rhs0 + r, v0 + v1);
      }
    }
  };
  int m_done = 0, base_done = 0;  // tile whose partial sums are waiting in `part`
  int m_cur = 0, m_next = 0, tile_base = 0, next_base = 0;
  prefetch(m_cur, tile_base);
  while (m_cur > 0) {
    const int m = m_cur;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 2; ++k) {  // squared offsets node - source per axis (chebyshev.rs:951-968)
      const int d = it_d[k], j = it_j[k];
      if (d < dim) {
        double *row = tab + ((size_t)d * T + j) * PREG;
        if (j < m) {
          const double *nc = ncoord + d * PREG;
          for (int i = 0; i < p; ++i) {
            const double o = nc[i] - pc[k];
            row[i] = o * o;
          }
        } else if (m < T) {  // neutral padding rows (r^2 = 1, weight 0) so every thread runs whole groups of kP2LJB
          const double fill = d == dim - 1 ? 1.0 : 0.0;
          for (int i = 0; i < p; ++i) row[i] = fill;
        }
      }
    }
    if (tid < T) {
#pragma unroll
      for (int r = 0; r < NR; ++r) wts[r * T + tid] = pw[r];
    }
    if (FUSE && do_m2p && m_done > 0) {  // the threads that built one row (or none) flush the previous tile's M2P sums
      if (n_flush >= 32) {
        if (tid >= nt - n_flush) flush_m2p(tid - (nt - n_flush), n_flush, m_done, base_done);
      } else {
        flush_m2p(tid, nt, m_done, base_done);
      }
    }
    __syncthreads();
    const int cur_base = tile_base;
    prefetch(m_next, next_base);
    // a tile without targets contributes nothing when the cell itself has no targets either
    const bool tile_wanted = !FUSE || need_p2l || a.tgt_prefix == nullptr ||
                             a.tgt_prefix[cur_base + m] != a.tgt_prefix[cur_base];
    if (active && tile_wanted) {
      const int kmax = (m + nslices - 1) / nslices;
      for (int k = 0; k < kmax; k += kP2LJB) {
        double axy[kP2LJB], wj[kP2LJB][NR], nx[kP2LJB];
        const double *dl[kP2LJB];
#pragma unroll
        for (int u = 0; u < kP2LJB; ++u) {
          const int j = slice + nslices * (k + u);  // < T: T / nslices is a multiple of kP2LJB
          axy[u] = 0.0;
          if (dim == 3) axy[u] = tabA[j * PREG + i0] + tabB[j * PREG + i1];
          else if (dim == 2) axy[u] = tabA[j * PREG + i0];
          dl[u] = tabL + j * PREG;
          nx[u] = dl[u][0];
#pragma unroll
          for (int r = 0; r < NR; ++r) wj[u][r] = wts[r * T + j];
        }
        double tp[FUSE ? kP2LJB : 1][FUSE ? NR : 1];
        if (FUSE) {
#pragma unroll
          for (int u = 0; u < kP2LJB; ++u)
#pragma unroll
            for (int r = 0; r < NR; ++r) tp[u][r] = 0.0;
        }
#pragma unroll
        for (int il = 0; il < PREG; ++il)
          if (il < p) {
            double v[kP2LJB];
#pragma unroll
            for (int u = 0; u < kP2LJB; ++u) {
              const double r2 = axy[u] + nx[u];
              if (il + 1 < PREG) nx[u] = dl[u][il + 1];  // next step's offsets are in flight during this one
              v[u] = kernel_mag<FAM, FAST, false>(r2, a.kp);
            }
#pragma unroll
            for (int u = 0; u < kP2LJB; ++u)
#pragma unroll
              for (int r = 0; r < NR; ++r) {
                kernel_acc<FAM>(acc[r][il], v[u], wj[u][r]);
                if (FUSE) kernel_acc<FAM>(tp[u][r], v[u], mreg[r][il]);
              }
          }
        if (FUSE && do_m2p) {
#pragma unroll
          for (int u = 0; u < kP2LJB; ++u)
#pragma unroll
            for (int r = 0; r < NR; ++r) part[((size_t)r * cols + q) * Ts + slice + nslices * (k + u)] = tp[u][r];
        }
      }
    }
    m_done = tile_wanted ? m : 0;
    base_done = cur_base;
    m_cur = m_next;
    tile_base = next_base;
  }
  if (FUSE && do_m2p) {
    __syncthreads();
    flush_m2p(tid, nt, m_done, base_done);
  }
  if (FUSE && !need_p2l) return;
  // ---- sum the slices in a fixed order and add to the cell's local expansion
  double *red = sm;  // [nslices][P]
#pragma unroll
  for (int r = 0; r < NR; ++r) {
    __syncthreads();
    if (active) {
#pragma unroll
      for (int il = 0; il < PREG; ++il)
        if (il < p) red[(size_t)slice * P + q * p + il] = acc[r][il];
    }
    __syncthreads();
    for (int nd = tid; nd < P; nd += nt) {
      double s = 0.0;
      for (int sl = 0; sl < nslices; ++sl) s += red[(size_t)sl * P + nd];
      a.loc[((size_t)c * a.nrhs + a.rhs0 + r) * coef_stride(P) + nd] += s;
    }
  }
}

// ======================================================================================================
// The same pass with the order and the dimension as template parameters (k_p2l_grid_t).  Same thread shape, tile,
// tables, association of r^2, accumulation order and slice reduction as k_p2l_grid, so the two agree to the last bit;
// what changes is the instruction count around the kernel evaluations.  The column, slice, tile and table strides
// are constants, so every shared-memory offset of the inner loop is an immediate on one base register per group of
// kP2LJB sources, the node loop unrolls to exactly PO steps (no guard on the padding slot of the row) and the last-axis
// offsets are read two at a time (LDS.128); the 49-column sums of the M2P flush unroll with constant offsets.
// ======================================================================================================
template <int PO, int D>
struct P2LShape {
  static_assert(D == 3, "templated P2L: 3-D only");
  static constexpr int PR = (PO + 1) & ~1;  // table row stride: even, so pairs of offsets are 16-byte aligned
  static constexpr int cols = PO * PO;
  static constexpr int nslices = cols >= 256 ? 1 : (256 / cols < 32 ? 256 / cols : 32);
  static constexpr int nthreads = ((nslices * cols + 31) / 32) * 32 < 128 ? 128
                                  : (((nslices * cols + 31) / 32) * 32 > 256 ? 256 : ((nslices * cols + 31) / 32) * 32);
  static constexpr int group = kP2LJB * nslices;
  // as launch_p2l_grid_impl: T <= nthreads, D * T <= 2 * nthreads, FUSE partial sums within ~48 KB (x2 when NR > 1)
  static constexpr int tile(int nr, bool fuse) {
    const int t0 = (kP2LTileMax < 2 * nthreads / D ? kP2LTileMax : 2 * nthreads / D) / group;
    int t = group * (t0 > 1 ? t0 : 1);
    if (fuse) {
      const int cap = (int)((nr > 1 ? 2 : 1) * kP2LFuseBytes / (sizeof(double) * (size_t)nr * cols)) - 1;
      const int c1 = (t < cap ? t : cap) / group;
      t = group * (c1 > 1 ? c1 : 1);
    }
    return t;
  }
};

template <int FAM, int NR, int PO, int D, bool FAST, bool FUSE>
__global__ void __launch_bounds__(P2LShape<PO, D>::nthreads, (NR * 8 <= 8) ? 3 : ((NR * 8 <= (FUSE ? 8 : 16)) ? 2 : 1))
    k_p2l_grid_t(const P2LArgs a) {
  using S = P2LShape<PO, D>;
  constexpr int PR = S::PR, cols = S::cols, nslices = S::nslices, nt = S::nthreads, T = S::tile(NR, FUSE);
  constexpr int Ts = T + 1;
  const int ci = blockIdx.x;
  const int c = a.cells[ci];
  const bool need_p2l = a.cell_flag[c] != 0;
  const bool do_m2p = FUSE && (a.cell_ptb == nullptr || (a.cell_ptb[c] >= a.own_lo && a.cell_ptb[c] < a.own_hi));
  if (!FUSE) {
    if (!need_p2l) return;
  } else if (!need_p2l) {
    if (a.tgt_prefix == nullptr) return;
    bool any = false;
    for (long long e = a.x_ptr[ci]; e < a.x_ptr[ci + 1] && !any; ++e)
      any = a.tgt_prefix[a.x_begin[e] + a.x_count[e]] != a.tgt_prefix[a.x_begin[e]];
    if (!any) return;
  }
  const int tid = threadIdx.x;
  constexpr int P = cols * PO;
  extern __shared__ __align__(16) double smt[];
  double *tab = smt;                      // [D][T][PR]
  double *wts = smt + (size_t)D * T * PR;  // [NR][T]
  double *part = wts + (size_t)NR * T;     // FUSE: [NR][cols][T + 1]
  const int q = tid % cols, slice = tid / cols;
  const bool active = slice < nslices;
  double mreg[FUSE ? NR : 1][FUSE ? PO : 1];
  if (FUSE) {
#pragma unroll
    for (int r = 0; r < NR; ++r)
#pragma unroll
      for (int il = 0; il < PO; ++il)
        mreg[r][il] = active ? a.mult[((size_t)c * a.nrhs + a.rhs0 + r) * coef_stride(P) + q * PO + il] *
                                   kernel_weight_scale<FAM, FAST>()
                             : 0.0;
  }
  const int i0 = q / PO, i1 = q % PO;
  __shared__ double ncoord[3 * PR];
  if (tid < D * PO) {
    const int d = tid / PO, i = tid - d * PO;
    const double cd = d == 0 ? a.ccx[c] : (d == 1 ? a.ccy[c] : a.ccz[c]);
    ncoord[d * PR + i] = cd + a.chalf[c] * a.nodes[i];
  }
  double acc[NR][PO];
#pragma unroll
  for (int r = 0; r < NR; ++r)
#pragma unroll
    for (int i = 0; i < PO; ++i) acc[r][i] = 0.0;

  long long e = a.x_ptr[ci];
  const long long e_end = a.x_ptr[ci + 1];
  int rb = 0, rn = 0, c0 = 0;
  if (e < e_end) {
    rb = a.x_begin[e];
    rn = a.x_count[e];
  }
  double pc[2] = {0.0, 0.0}, pw[NR];
  int it_d[2], it_j[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int t = tid + k * nt;
    it_d[k] = (t >= T) + (t >= 2 * T) + (t >= 3 * T);
    it_j[k] = t - it_d[k] * T;
  }
  auto prefetch = [&](int &m, int &base) {
    m = 0;
    if (e >= e_end) return;
    m = min(T, rn - c0);
    base = rb + c0;
#pragma unroll
    for (int k = 0; k < 2; ++k)
      if (it_d[k] < D && it_j[k] < m)
        pc[k] = it_d[k] == 0 ? a.sx[base + it_j[k]] : (it_d[k] == 1 ? a.sy[base + it_j[k]] : a.sz[base + it_j[k]]);
#pragma unroll
    for (int r = 0; r < NR; ++r)
      pw[r] = tid < m ? a.w[(size_t)(a.rhs0 + r) * a.n + base + tid] * kernel_weight_scale<FAM, FAST>() : 0.0;
    c0 += T;
    if (c0 >= rn) {
      ++e;
      c0 = 0;
      if (e < e_end) {
        rb = a.x_begin[e];
        rn = a.x_count[e];
      }
    }
  };
  constexpr int n_flush = nt - (D * T - nt > 0 ? D * T - nt : 0);
  auto flush_m2p = [&](int first, int step, int m_done, int base_done) {
    for (int j = first; j < m_done; j += step) {
      const uint32_t row32 = a.out_row[base_done + j];
      if (row32 == 0xFFFFFFFFu) continue;
      const size_t row = row32;
#pragma unroll
      for (int r = 0; r < NR; ++r) {
        const double *pp = part + (size_t)r * cols * Ts + j;
        double v0 = 0.0, v1 = 0.0;
#pragma unroll
        for (int qq = 0; qq + 1 < cols; qq += 2) {
          v0 += pp[qq * Ts];
          v1 += pp[(qq + 1) * Ts];
        }
        if (cols % 2) v0 += pp[(cols - 1) * Ts];
        atomicAdd(a.out + row * a.nrhs + a.rhs0 + r, v0 + v1);
      }
    }
  };
  // per-thread bases: source j of the group sits at + nslices * (k + u) rows
  const double *pA = tab + slice * PR + i0, *pB = tab + (T + slice) * PR + i1, *pL = tab + (2 * T + slice) * PR;
  const double *pW = wts + slice;
  double *pP = part + q * Ts + slice;
  int m_done = 0, base_done = 0;
  int m_cur = 0, m_next = 0, tile_base = 0, next_base = 0;
  prefetch(m_cur, tile_base);
  while (m_cur > 0) {
    const int m = m_cur;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 2; ++k) {  // squared offsets node - source per axis (chebyshev.rs:951-968)
      const int d = it_d[k], j = it_j[k];
      if (d < D) {
        double *row = tab + (d * T + j) * PR;
        if (j < m) {
          const double *nc = ncoord + d * PR;
#pragma unroll
          for (int i = 0; i < PO; ++i) {
            const double o = nc[i] - pc[k];
            row[i] = o * o;
          }
        } else if (m < T) {  // neutral padding rows (r^2 = 1, weight 0)
          const double fill = d == D - 1 ? 1.0 : 0.0;
#pragma unroll
          for (int i = 0; i < PO; ++i) row[i] = fill;
        }
      }
    }
    if (tid < T) {
#pragma unroll
      for (int r = 0; r < NR; ++r) wts[r * T + tid] = pw[r];
    }
    if (FUSE && do_m2p && m_done > 0) {
      if (n_flush >= 32) {
        if (tid >= nt - n_flush) flush_m2p(tid - (nt - n_flush), n_flush, m_done, base_done);
      } else {
        flush_m2p(tid, nt, m_done, base_done);
      }
    }
    __syncthreads();
    const int cur_base = tile_base;
    prefetch(m_next, next_base);
    const bool tile_wanted = !FUSE || need_p2l || a.tgt_prefix == nullptr ||
                             a.tgt_prefix[cur_base + m] != a.tgt_prefix[cur_base];
    if (active && tile_wanted) {
      const int kmax = (m + nslices - 1) / nslices;
      for (int k = 0; k < kmax; k += kP2LJB) {
        const int o = nslices * k;
        double axy[kP2LJB], wj[kP2LJB][NR];
#pragma unroll
        for (int u = 0; u < kP2LJB; ++u) {
          axy[u] = pA[(o + nslices * u) * PR] + pB[(o + nslices * u) * PR];
#pragma unroll
          for (int r = 0; r < NR; ++r) wj[u][r] = pW[r * T + o + nslices * u];
        }
        double tp[FUSE ? kP2LJB : 1][FUSE ? NR : 1];
        if (FUSE) {
#pragma unroll
          for (int u = 0; u < kP2LJB; ++u)
#pragma unroll
            for (int r = 0; r < NR; ++r) tp[u][r] = 0.0;
        }
        auto step = [&](const int il, const double (&dz)[kP2LJB]) {
          double v[kP2LJB];
#pragma unroll
          for (int u = 0; u < kP2LJB; ++u) v[u] = kernel_mag<FAM, FAST, false>(axy[u] + dz[u], a.kp);
#pragma unroll
          for (int u = 0; u < kP2LJB; ++u)
#pragma unroll
            for (int r = 0; r < NR; ++r) {
              kernel_acc<FAM>(acc[r][il], v[u], wj[u][r]);
              if (FUSE) kernel_acc<FAM>(tp[u][r], v[u], mreg[FUSE ? r : 0][FUSE ? il : 0]);
            }
        };
#pragma unroll
        for (int il = 0; il < PO; il += 2) {
          double dz0[kP2LJB], dz1[kP2LJB];
#pragma unroll
          for (int u = 0; u < kP2LJB; ++u) {
            const double *row = pL + (o + nslices * u) * PR + il;
            if (il + 1 < PO) {
              const double2 z = *reinterpret_cast<const double2 *>(row);
              dz0[u] = z.x;
              dz1[u] = z.y;
            } else {
              dz0[u] = row[0];
            }
          }
          step(il, dz0);
          if (il + 1 < PO) step(il + 1, dz1);
        }
        if (FUSE && do_m2p) {
#pragma unroll
          for (int u = 0; u < kP2LJB; ++u)
#pragma unroll
            for (int r = 0; r < NR; ++r) pP[r * cols * Ts + o + nslices * u] = tp[u][r];
        }
      }
    }
    m_done = tile_wanted ? m : 0;
    base_done = cur_base;
    m_cur = m_next;
    tile_base = next_base;
  }
  if (FUSE && do_m2p) {
    __syncthreads();
    flush_m2p(tid, nt, m_done, base_done);
  }
  if (FUSE && !need_p2l) return;
  double *red = smt;  // [nslices][P]
#pragma unroll
  for (int r = 0; r < NR; ++r) {
    __syncthreads();
    if (active) {
#pragma unroll
      for (int il = 0; il < PO; ++il) red[slice * P + q * PO + il] = acc[r][il];
    }
    __syncthreads();
    for (int nd = tid; nd < P; nd += nt) {
      double s = 0.0;
#pragma unroll
      for (int sl = 0; sl < nslices; ++sl) s += red[sl * P + nd];
      a.loc[((size_t)c * a.nrhs + a.rhs0 + r) * coef_stride(P) + nd] += s;
    }
  }
}

template <int FAM, int NR, int PO, int D, bool FAST, bool FUSE>
static void launch_p2l_grid_t_impl(const P2LArgs &a, cudaStream_t s) {
  using S = P2LShape<PO, D>;
  constexpr int T = S::tile(NR, FUSE);
  constexpr size_t tab_d = (size_t)D * T * S::PR + (size_t)NR * T + (FUSE ? (size_t)NR * S::cols * (T + 1) : 0);
  constexpr size_t red_d = (size_t)S::nslices * S::cols * PO;
  constexpr size_t smem = sizeof(double) * (tab_d > red_d ? tab_d : red_d);
  if (smem > 48 * 1024)
    FB_CUDA(cudaFuncSetAttribute(k_p2l_grid_t<FAM, NR, PO, D, FAST, FUSE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)smem));
  FB_LAUNCH((k_p2l_grid_t<FAM, NR, PO, D, FAST, FUSE>), a.n_cells, S::nthreads, smem, s, a);
}

// orders with a templated kernel; FB_GENERIC_P2L=1 forces k_p2l_grid everywhere (A/B baseline)
#define FB_P2L_ORDER_SWITCH(CALL) \
  if (a.dim == 3) {               \
    switch (a.p) {                \
      case 7: CALL(7, 3); return true; \
      default: return false;      \
    }                             \
  }                               \
  return false;

template <int FAM, int NR, bool FAST, bool FUSE>
static bool launch_p2l_grid_t(const P2LArgs &a, cudaStream_t s) {
  static const bool off = [] {
    const char *v = std::getenv("FB_GENERIC_P2L");
    return v && v[0] == '1';
  }();
  if (off) return false;
#define CALL(PO, D) launch_p2l_grid_t_impl<FAM, NR, PO, D, FAST, FUSE>(a, s)
  FB_P2L_ORDER_SWITCH(CALL)
#undef CALL
}

template <int FAM, int NR, int PREG, bool FAST, bool FUSE>
static void launch_p2l_grid_impl(const P2LArgs &a, cudaStream_t s) {
  if constexpr (PREG == 8)
    if (launch_p2l_grid_t<FAM, NR, FAST, FUSE>(a, s)) return;
  const int cols = a.dim == 3 ? a.p * a.p : (a.dim == 2 ? a.p : 1);
  const int nslices = std::min(32, std::max(1, 256 / cols));
  const int nthreads = std::max(128, std::min(256, ((nslices * cols + 31) / 32) * 32));
  const int group = kP2LJB * nslices;
  // T <= nthreads (one weight per thread) and dim * T <= 2 * nthreads (two table rows per thread)
  int T = group * std::max(1, std::min(kP2LTileMax, (2 * nthreads) / std::max(2, a.dim)) / group);
  if (FUSE) {  // per-(column, point) partial sums: keep them within ~48 KB
    const int cap = (int)((NR > 1 ? 2 : 1) * kP2LFuseBytes / (sizeof(double) * (size_t)NR * cols)) - 1;
    T = group * std::max(1, std::min(T, cap) / group);
  }
  const size_t tab_d = (size_t)a.dim * T * PREG + (size_t)NR * T + (FUSE ? (size_t)NR * cols * (T + 1) : 0);
  const size_t red_d = (size_t)nslices * a.P;
  const size_t smem = sizeof(double) * std::max(tab_d, red_d);
  if (smem > 48 * 1024)
    FB_CUDA(cudaFuncSetAttribute(k_p2l_grid<FAM, NR, PREG, FAST, FUSE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)smem));
  FB_LAUNCH((k_p2l_grid<FAM, NR, PREG, FAST, FUSE>), a.n_cells, nthreads, smem, s, a, nslices, cols, T);
}
template <int FAM, int NR, int PREG>
static void launch_p2l_grid(const P2LArgs &a, cudaStream_t s) {
  constexpr bool kFast = kernel_has_fast<FAM>();
  const bool fast = kFast && a.kp.fast;
  if (a.out) {  // fused M2P (targets = all sources)
    if (fast) launch_p2l_grid_impl<FAM, NR, PREG, kFast, true>(a, s);
    else launch_p2l_grid_impl<FAM, NR, PREG, false, true>(a, s);
  } else {
    if (fast) launch_p2l_grid_impl<FAM, NR, PREG, kFast, false>(a, s);
    else launch_p2l_grid_impl<FAM, NR, PREG, false, false>(a, s);
  }
}

// ---------------------------------------------------------------------------------- dispatch
template <int FAM>
static void p2l_fam(P2LArgs a, cudaStream_t s) {
  if (a.n_cells <= 0) return;
  int r = 0;
  while (r < a.nrhs) {
    a.rhs0 = r;
    const int left = a.nrhs - r;
    if (a.p <= 8) {  // p accumulators per right-hand side live in registers: 8 or 16 slots
      if (left >= 4) {
        launch_p2l_grid<FAM, 4, 8>(a, s);
        r += 4;
      } else if (left >= 2) {
        launch_p2l_grid<FAM, 2, 8>(a, s);
        r += 2;
      } else {
        launch_p2l_grid<FAM, 1, 8>(a, s);
        r += 1;
      }
    } else {
      if (left >= 2) {
        launch_p2l_grid<FAM, 2, 16>(a, s);
        r += 2;
      } else {
        launch_p2l_grid<FAM, 1, 16>(a, s);
        r += 1;
      }
    }
  }
}

void launch_p2l(const P2LArgs &a, cudaStream_t s) {
#define CALL(F) p2l_fam<F>(a, s)
  FB_FAM_SWITCH(a.kp.fam, CALL)
#undef CALL
}

}  // namespace fb
