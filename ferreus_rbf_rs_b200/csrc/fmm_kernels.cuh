// Device kernels of the FMM passes other than the direct sums (see direct.cu).
//   tree:      k_point_codes, k_gather_sorted, k_target_leaf ...       (morton.rs:35-119, linear_tree.rs:487-534)
//   upward:    k_p2m, k_m2m                                              (bbfmm.rs:666-772)
//   downward:  k_m2l, k_l2l                                              (bbfmm.rs:778-1086)
//   leaf:      k_l2p                                                     (bbfmm.rs:1358-1440)
#pragma once
#include "fmm.h"

namespace fb {

// ------------------------------------------------------------------------------------------ tree
__device__ __forceinline__ unsigned long long interleave_bits(unsigned a0, unsigned a1, unsigned a2, int dim) {
  unsigned long long code = 0;
  for (int bit = 0; bit < 16; ++bit) {
    code |= (unsigned long long)((a0 >> bit) & 1u) << (bit * dim);
    if (dim > 1) code |= (unsigned long long)((a1 >> bit) & 1u) << (bit * dim + 1);
    if (dim > 2) code |= (unsigned long long)((a2 >> bit) & 1u) << (bit * dim + 2);
  }
  return code;
}

// floor((x - disp) / side) as u64 with Rust `as` saturation (morton.rs:46): NaN/negative -> 0
__device__ __forceinline__ unsigned long long anchor_sat(double x, double disp, double side) {
  const double q = floor(__ddiv_rn(__dsub_rn(x, disp), side));
  if (!(q >= 0.0)) return 0ull;
  if (q >= 18446744073709551616.0) return 0xFFFFFFFFFFFFFFFFull;
  return (unsigned long long)q;
}

// level-16 interleaved code of every source point; err = first row outside the root cube (high side)
__global__ void k_point_codes(const double *pts, size_t n, int dim, double d0, double d1, double d2, double side16,
                              unsigned long long *codes, uint32_t *idx, unsigned long long *err) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double disp[3] = {d0, d1, d2};
  unsigned a[3] = {0, 0, 0};
  for (int j = 0; j < dim; ++j) {
    const unsigned long long v = anchor_sat(pts[i * dim + j], disp[j], side16);
    if (v >= 65536ull) atomicMin(err, (unsigned long long)i);
    a[j] = (unsigned)(v & 0xFFFFull);
  }
  codes[i] = interleave_bits(a[0], a[1], a[2], dim);
  idx[i] = (uint32_t)i;
}

__global__ void k_gather_sorted(const double *pts, const uint32_t *perm, size_t n, int dim, double *sx, double *sy,
                                double *sz, uint32_t *inv) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t s = perm[i];
  sx[i] = pts[(size_t)s * dim];
  sy[i] = dim > 1 ? pts[(size_t)s * dim + 1] : 0.0;
  sz[i] = dim > 2 ? pts[(size_t)s * dim + 2] : 0.0;
  if (inv) inv[s] = (uint32_t)i;
}

// weights [n][nrhs] row-major (user order) -> [rhs][n] sorted order
__global__ void k_sort_weights(const double *wu, const uint32_t *perm, size_t n, int nrhs, double *ws) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const size_t s = perm[i];
  for (int r = 0; r < nrhs; ++r) ws[(size_t)r * n + i] = wu[s * nrhs + r];
}

// leaf slot of every target (linear_tree.rs:487-520): key at level `depth`, then the enclosing leaf
__global__ void k_target_leaf(const double *tg, size_t m, int dim, int depth, double d0, double d1, double d2,
                              double side_depth, const unsigned long long *leaf_lo, const unsigned long long *leaf_hi,
                              int n_leaves, uint32_t *slot, uint32_t *idx, unsigned long long *err) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= m) return;
  const double disp[3] = {d0, d1, d2};
  unsigned a[3] = {0, 0, 0};
  bool outside = false;
  for (int j = 0; j < dim; ++j) {
    const unsigned long long v = anchor_sat(tg[i * dim + j], disp[j], side_depth) & 0xFFFFull;  // 16-bit LUT masking
    if (v >= (1ull << depth)) outside = true;
    a[j] = (unsigned)v;
  }
  idx[i] = (uint32_t)i;
  uint32_t s = 0;
  if (!outside) {
    const unsigned long long code = interleave_bits(a[0], a[1], a[2], dim) << (dim * (16 - depth));
    int lo = 0, hi = n_leaves;  // last leaf with leaf_lo <= code
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (leaf_lo[mid] <= code)
        lo = mid;
      else
        hi = mid;
    }
    if (n_leaves > 0 && leaf_lo[lo] <= code && code < leaf_hi[lo])
      s = (uint32_t)lo;
    else
      outside = true;
  }
  if (outside) atomicMin(err, (unsigned long long)i);
  slot[i] = s;
}

// flag != 0 when the two coordinate arrays differ in any bit
__global__ void k_points_differ(const double *a, const double *b, size_t count, unsigned long long *flag) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= count) return;
  if (__double_as_longlong(a[i]) != __double_as_longlong(b[i])) *flag = 1ull;
}

__global__ void k_subset_positions(const unsigned long long *idx, const uint32_t *inv, size_t m, size_t n,
                                   uint32_t *pos, uint32_t *val, unsigned long long *err) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= m) return;
  const unsigned long long s = idx[i];
  if (s >= n) {
    atomicMin(err, (unsigned long long)i);
    pos[i] = 0;
  } else {
    pos[i] = inv[s];
  }
  val[i] = (uint32_t)i;
}

// sorted source position -> output row of a subset-of-sources target set; dup != 0 when a position occurs twice
__global__ void k_subset_row_map(const uint32_t *pos_sorted, const uint32_t *rows, size_t m, uint32_t *row_of_pos,
                                 unsigned long long *dup) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= m) return;
  if (i + 1 < m && pos_sorted[i + 1] == pos_sorted[i]) *dup = 1ull;
  row_of_pos[pos_sorted[i]] = rows[i];
}
struct RowIsTarget {
  __host__ __device__ uint32_t operator()(uint32_t row) const { return row != 0xFFFFFFFFu ? 1u : 0u; }
};
__global__ void k_prefix_total(uint32_t *prefix, const uint32_t *row_of_pos, size_t n) {
  prefix[n] = n ? prefix[n - 1] + (row_of_pos[n - 1] != 0xFFFFFFFFu ? 1u : 0u) : 0u;
}

// per leaf slot: range of sorted targets whose key (leaf slot, or sorted source position) falls in the leaf
__global__ void k_leaf_ranges(const uint32_t *keys, size_t m, const int *key_lo, const int *key_hi, int n_leaves,
                              int *begin, int *end, int *tile_cnt) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= n_leaves) return;
  const uint32_t klo = key_lo ? (uint32_t)key_lo[l] : (uint32_t)l;
  const uint32_t khi = key_hi ? (uint32_t)key_hi[l] : (uint32_t)l + 1u;
  size_t lo = 0, hi = m;
  while (lo < hi) {
    const size_t mid = (lo + hi) >> 1;
    if (keys[mid] < klo) lo = mid + 1; else hi = mid;
  }
  const size_t b = lo;
  hi = m;
  while (lo < hi) {
    const size_t mid = (lo + hi) >> 1;
    if (keys[mid] < khi) lo = mid + 1; else hi = mid;
  }
  begin[l] = (int)b;
  end[l] = (int)lo;
  tile_cnt[l] = ((int)(lo - b) + kTile - 1) / kTile;
}

__global__ void k_fill_tiles(const int *tile_off_scan, const int *tile_cnt, int n_leaves, int *tile_leaf, int *tile_off,
                             int *n_tiles) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= n_leaves) return;
  const int base = tile_off_scan[l];
  for (int t = 0; t < tile_cnt[l]; ++t) {
    tile_leaf[base + t] = l;
    tile_off[base + t] = t * kTile;
  }
  if (l == n_leaves - 1) *n_tiles = base + tile_cnt[l];
}

__global__ void k_gather_targets(const double *tg, const uint32_t *order, size_t m, int dim, double *tx, double *ty,
                                 double *tz) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= m) return;
  const size_t s = order[i];
  tx[i] = tg[s * dim];
  ty[i] = dim > 1 ? tg[s * dim + 1] : 0.0;
  tz[i] = dim > 2 ? tg[s * dim + 2] : 0.0;
}

__global__ void k_gather_coords(const double *sx, const double *sy, const double *sz, const uint32_t *pos, size_t m,
                                double *tx, double *ty, double *tz) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= m) return;
  const size_t s = pos[i];
  tx[i] = sx[s];
  ty[i] = sy[s];
  tz[i] = sz[s];
}

// cells_with_targets = union of ancestors of leaves that hold targets (bbfmm.rs:467-478)
__global__ void k_flag_cells(const int *leaf_cell, const int *begin, const int *end, int n_leaves, const int *parent,
                             uint8_t *flag) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= n_leaves || end[l] <= begin[l]) return;
  int c = leaf_cell[l];
  while (c >= 0) {
    flag[c] = 1;
    c = parent[c];
  }
}

// --------------------------------------------------------------------------------------- Chebyshev
// S_n(x)[m] = (2 sum_k T_k(x) T_k(x_m) - 1) / p  (chebyshev.rs:114-127); optionally dS/dx (chebyshev.rs:130-142)
__device__ __forceinline__ void cheb_s(int p, double x, const double *tn, double *S, double *dS, double dscale) {
  double T[kMaxOrder], dT[kMaxOrder];
  T[0] = 1.0;
  dT[0] = 0.0;
  if (p > 1) {
    T[1] = x;
    dT[1] = 1.0;
  }
  for (int k = 2; k < p; ++k) {
    T[k] = 2.0 * x * T[k - 1] - T[k - 2];
    if (dS) dT[k] = 2.0 * T[k - 1] + 2.0 * x * dT[k - 1] - dT[k - 2];
  }
  const double pd = (double)p;
  for (int m = 0; m < p; ++m) {
    double s = 0.0, ds = 0.0;
    for (int k = 0; k < p; ++k) {
      const double t = tn[m * p + k];
      s += T[k] * t;
      if (dS) ds += dT[k] * t;
    }
    S[m] = (s * 2.0 - 1.0) / pd;
    if (dS) dS[m] = ds * (2.0 / pd) * dscale;
  }
}

// P2M: one CTA per source leaf (bbfmm.rs:691-739, chebyshev.rs:831-927)
constexpr int kP2MChunk = 64;
__global__ void __launch_bounds__(256) k_p2m(const int *leaves, const int *ptb, const int *pte, const double *sx,
                                             const double *sy, const double *sz, const double *w, size_t n,
                                             const double *ccx, const double *ccy, const double *ccz,
                                             const double *chalf, const double *tnodes, int p, int dim, int P, int nrhs,
                                             double *mult) {
  extern __shared__ double sm[];
  double *tn = sm;                       // p*p
  double *S = tn + p * p;                // [3][chunk][p]
  const int c = leaves[blockIdx.x];
  const int b = ptb[c], e = pte[c];
  const int tid = threadIdx.x;
  for (int i = tid; i < p * p; i += blockDim.x) tn[i] = tnodes[i];
  const double cc[3] = {ccx[c], ccy[c], ccz[c]};
  const double half = chalf[c];
  const int p1 = dim > 1 ? p : 1, p2 = dim > 2 ? p : 1;
  for (int c0 = b; c0 < e; c0 += kP2MChunk) {
    const int m = min(kP2MChunk, e - c0);
    __syncthreads();
    for (int t = tid; t < m * dim; t += blockDim.x) {
      const int pt = t / dim, d = t % dim;
      const double coord = d == 0 ? sx[c0 + pt] : (d == 1 ? sy[c0 + pt] : sz[c0 + pt]);
      const double x = (coord - cc[d]) / half;  // chebyshev.rs:841-845
      cheb_s(p, x, tn, &S[(d * kP2MChunk + pt) * p], nullptr, 0.0);
    }
    __syncthreads();
    for (int o = tid; o < P * nrhs; o += blockDim.x) {
      const int node = o % P, r = o / P;
      const int i2 = node % p2, i1 = (node / p2) % p1, i0 = node / (p1 * p2);
      const double *wr = w + (size_t)r * n + c0;
      double acc = 0.0;
      for (int pt = 0; pt < m; ++pt) {
        double s = S[(0 * kP2MChunk + pt) * p + i0];
        if (dim > 1) s *= S[(1 * kP2MChunk + pt) * p + i1];
        if (dim > 2) s *= S[(2 * kP2MChunk + pt) * p + i2];
        acc += s * wr[pt];
      }
      mult[((size_t)c * nrhs + r) * coef_stride(P) + node] += acc;
    }
  }
}

// One axis of the tensor-product transfer:  out[.. a ..] = sum_b A(a, b) in[.. b ..]
//   up   (M2M): A(m, i) = child_s[h][i][m]      down (L2L): A(i, m) = child_s[h][i][m]
__device__ __forceinline__ void tensor_axis(const double *in, double *out, const double *A, int p, int P, int stride,
                                            bool up, int tid, int nthreads) {
  for (int o = tid; o < P; o += nthreads) {
    const int a = (o / stride) % p;
    const int base = o - a * stride;
    double s = 0.0;
    for (int b = 0; b < p; ++b) s += (up ? A[b * p + a] : A[a * p + b]) * in[base + b * stride];
    out[o] = s;
  }
}

// M2M: one CTA per parent, one WARP per child (all children in flight: the pass is a chain of dependent shared-memory
// sweeps, latency not work — 42-59 us per level with the children taken one after the other, and the upward pass is a
// fixed cost of every partitioned matvec); M_parent += M2M[child_index] * M_child, sum-factorised over the axes, the
// children's contributions added in child order (bbfmm.rs:742-772; M2M[c] = (S_x (x) S_y (x) S_z)^T, chebyshev.rs:196-241)
__global__ void __launch_bounds__(256) k_m2m(const int *parents, const int *child_ptr, const int *child_idx,
                                             const int *cell_slot, const double *child_s, int p, int dim, int P,
                                             int nrhs, const uint8_t *flag, int cpar, double *mult) {
  extern __shared__ double sm[];
  double *A = sm;              // 2*p*p
  double *buf = A + 2 * p * p;  // [cpar children][2][P]
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int parent = parents[blockIdx.x];
  if (flag && !flag[parent]) return;  // sharded upward pass: no owned descendants, the multipole stays zero
  for (int i = tid; i < 2 * p * p; i += nt) A[i] = child_s[i];
  const int k0 = child_ptr[parent], nch = child_ptr[parent + 1] - k0;
  const int Ps = coef_stride(P);
  for (int r = 0; r < nrhs; ++r) {
    double *dst = mult + ((size_t)parent * nrhs + r) * Ps;
    for (int c0 = 0; c0 < nch; c0 += cpar) {  // cpar children at a time (all 2^dim unless p^d is too large for that)
      const int nb = min(cpar, nch - c0);
      __syncthreads();
      if (warp < nb) {
        const int ch = child_idx[k0 + c0 + warp];
        const int slot = cell_slot[ch];
        double *in = buf + (size_t)warp * 2 * P, *out = in + P;
        const double *src = mult + ((size_t)ch * nrhs + r) * Ps;
        for (int i = lane; i < P; i += 32) in[i] = src[i];
        __syncwarp();
        for (int d = 0; d < dim; ++d) {
          int stride = 1;
          for (int e = d + 1; e < dim; ++e) stride *= p;
          const int h = (slot >> d) & 1;  // bit d of the child index = half along axis d (chebyshev.rs:183-192)
          tensor_axis(in, out, A + h * p * p, p, P, stride, true, lane, 32);
          __syncwarp();
          double *t = in;
          in = out;
          out = t;
        }
      }
      __syncthreads();
      // the transformed child c sits in buf[c][dim & 1]
      for (int i = tid; i < P; i += nt) {
        double acc = 0.0;
        for (int c = 0; c < nb; ++c) acc += buf[((size_t)c * 2 + (dim & 1)) * P + i];
        dst[i] += acc;
      }
    }
  }
}

// L2L: one CTA per child cell of the level; L_child += M2M[child_index]^T L_parent (bbfmm.rs:1051-1086)
__global__ void __launch_bounds__(128) k_l2l(int cell0, const int *cell_parent, const int *cell_slot,
                                             const uint8_t *flag, const double *child_s, int p, int dim, int P, int nrhs,
                                             double *loc) {
  extern __shared__ double sm[];
  double *A = sm;
  double *b0 = A + 2 * p * p;
  double *b1 = b0 + P;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int c = cell0 + blockIdx.x;
  if (!flag[c]) return;
  const int parent = cell_parent[c];
  const int slot = cell_slot[c];
  for (int i = tid; i < 2 * p * p; i += nt) A[i] = child_s[i];
  for (int r = 0; r < nrhs; ++r) {
    __syncthreads();
    const double *src = loc + ((size_t)parent * nrhs + r) * coef_stride(P);
    for (int i = tid; i < P; i += nt) b0[i] = src[i];
    __syncthreads();
    double *in = b0, *out = b1;
    for (int d = 0; d < dim; ++d) {
      int stride = 1;
      for (int e = d + 1; e < dim; ++e) stride *= p;
      const int h = (slot >> d) & 1;
      tensor_axis(in, out, A + h * p * p, p, P, stride, false, tid, nt);
      __syncthreads();
      double *t = in;
      in = out;
      out = t;
    }
    double *dst = loc + ((size_t)c * nrhs + r) * coef_stride(P);
    for (int i = tid; i < P; i += nt) dst[i] += in[i];
  }
}

// ---- FP64 tensor-core helpers: mma.sync.aligned.m8n8k4 (SASS: DMMA.8x8x4) -------------------------------
// fragments: A[lane>>2][lane&3], B[lane&3][lane>>2], C/D[lane>>2][(lane&3)*2 + {0,1}]
__device__ __forceinline__ void dmma884(double &d0, double &d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}

// (entry, rhs) columns per CTA: NC = 32, 16 or 8 (chosen so the staged multipoles fit in shared memory);
// the row stride of Ys is NC + 4 == 4 or 12 (mod 16) -> conflict-free B fragments

constexpr int kM2LChunk = 4;  // rank tiles (8 rows each) accumulated per pass over the reduction
constexpr int kM2LPre = 8;    // k-steps of operator fragments prefetched per block in the second contraction

// M2L for one (level, reference vector) group (bbfmm.rs:864-986) as two dense contractions on the FP64 tensor
// cores.  A CTA owns NC (entry, rhs) columns:
//   Xs[c][j] = M_src[perm[j]]   permuted multipoles, staged once in shared memory (column stride Pp, Pp == 4 or
//                               12 mod 16 so the B fragments are bank-conflict free)
//   Ys = Vt Xs  (rank x NC)     8 warps = NC/8 column tiles x slices of the P-long reduction, summed in shared memory
//   Zs = U  Ys  (P x NC)        warps stride over the 8-row tiles of U; the accumulator fragments are parked in
//                               shared memory (over Xs, which is dead by then)
//   flush                       L_tgt[i] += sum over the columns of the same (target, rhs) of Zs[c][inv_perm_c[i]]:
//                               one coalesced RED per (target, node) instead of one scattered RED per (entry, node)
// Operators are stored in DMMA fragment order, zero padded: frag(mt, ks)[lane] = Op[mt*8 + lane/4][ks*4 + lane%4],
// so every A fragment is one coalesced 256-byte load.  ncu before this layout (profiles/r1_s2_ncu_full.txt): 47 % of
// the stalls were long-scoreboard waits on the per-element permutation loads of the scatter and on the fragment loads.
struct M2LGroupDev {  // one (level, reference vector) group of the fused M2L launch
  int cta_begin;        // first CTA of the group
  int rank_pad;
  long long entry_off;  // into the entry arrays
  long long n_entries;
  long long v_off, u_off;  // operator pool offsets (fragment order)
};

template <bool COMPRESSED, int NC>
__global__ void __launch_bounds__(256, NC == 32 ? 2 : 1) k_m2l(const M2LGroupDev *groups, const int *cta_group, const int *e_tgt_all,
                                                const int *e_src_all, const int *e_perm_all, const double *pool,
                                                const int *perm_tab, const int *inv_tab, int P, int P4, int Pp, int nrhs,
                                                const uint8_t *flag, const double *mult, double *loc) {
  // all levels and reference vectors run in ONE launch: M2L at different levels is independent
  const M2LGroupDev g = groups[cta_group[blockIdx.x]];
  const int *e_tgt = e_tgt_all + g.entry_off, *e_src = e_src_all + g.entry_off, *e_perm = e_perm_all + g.entry_off;
  const size_t n_entries = (size_t)g.n_entries;
  const int rank_pad = g.rank_pad;
  const double *VtF = pool + g.v_off, *UF = pool + g.u_off;
  const unsigned cta = blockIdx.x - g.cta_begin;
  extern __shared__ double sm[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t ncols = n_entries * (size_t)nrhs;
  constexpr int kM2LCols = NC, kM2LColsPad = NC + 4;
  constexpr int NW = 8;              // warps per CTA
  constexpr int kNT = NC / 8;        // 8-column tiles
  const size_t col0 = (size_t)cta * kM2LCols;
  const int nc = (int)min((size_t)kM2LCols, ncols - col0);
  double *Xs = sm;                                        // [NC][Pp]; reused as Zs after the first contraction
  double *Ys = Xs + (size_t)kM2LCols * Pp;                // [rank_pad][NC + 4]
  __shared__ int s_tgt[kM2LCols], s_rhs[kM2LCols], s_perm[kM2LCols], s_src[kM2LCols];
  __shared__ int s_list[kM2LCols], s_off[kM2LCols], s_len[kM2LCols];  // columns grouped by (target, rhs) run
  __shared__ int s_runs[kM2LCols], s_nruns;                          // first column of every run, number of runs
  __shared__ int s_any;
  if (tid == 0) s_any = 0;
  __syncthreads();
  if (tid < kM2LCols) {
    int tg = -1, sr = 0, pm = 0, rh = 0;
    if (tid < nc) {
      const size_t col = col0 + tid;
      const size_t e = col / nrhs;
      rh = (int)(col % nrhs);
      tg = e_tgt[e];
      sr = e_src[e];
      pm = e_perm[e];
      if (!flag[tg]) tg = -1; else s_any = 1;
    }
    s_tgt[tid] = tg;
    s_src[tid] = sr;
    s_perm[tid] = pm;
    s_rhs[tid] = rh;
  }
  __syncthreads();
  if (!s_any) return;
  if (warp == 0) {
    // runs of columns that add into the same (target, rhs): s_list holds the columns run by run; the first column
    // of a run carries the run's offset and length, every other column length 0
    const int col = lane;
    const bool valid = col < kM2LCols && s_tgt[col] >= 0;
    const int key = valid ? s_tgt[col] * nrhs + s_rhs[col] : -(lane + 1);
    const unsigned same = __match_any_sync(0xffffffffu, key);
    const int first = __ffs(same) - 1;
    const int rank_in_run = __popc(same & ((1u << lane) - 1u));
    int before = 0;  // columns of runs that start earlier
    for (int k = 0; k < 32; ++k) {
      const int fk = __shfl_sync(0xffffffffu, first, k);
      const int vk = __shfl_sync(0xffffffffu, (int)valid, k);
      before += (vk && fk < first) ? 1 : 0;
    }
    const bool is_first = valid && first == lane;
    const unsigned firsts = __ballot_sync(0xffffffffu, is_first);
    if (col < kM2LCols) {
      if (valid) s_list[before + rank_in_run] = col;
      s_off[col] = before;
      s_len[col] = is_first ? __popc(same) : 0;
      if (is_first) s_runs[__popc(firsts & ((1u << lane) - 1u))] = col;
    }
    if (lane == 0) s_nruns = __popc(firsts);
  }
  // stage permuted multipoles (zero padding up to P4 and for idle columns); 4 gathers in flight per lane
  for (int c = warp; c < kM2LCols; c += NW) {
    double *dst = Xs + (size_t)c * Pp;
    if (s_tgt[c] >= 0) {
      const double *src = mult + ((size_t)s_src[c] * nrhs + s_rhs[c]) * coef_stride(P);
      const int *pm = perm_tab + (size_t)s_perm[c] * P;
      for (int j0 = lane; j0 < P4; j0 += 128) {
        int idx[4];
        double v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) idx[u] = (j0 + 32 * u < P) ? __ldg(pm + j0 + 32 * u) : -1;
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = idx[u] >= 0 ? __ldg(src + idx[u]) : 0.0;
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (j0 + 32 * u < P4) dst[j0 + 32 * u] = v[u];
      }
    } else {
      for (int j = lane; j < P4; j += 32) dst[j] = 0.0;
    }
  }
  __syncthreads();
  const int ar = lane >> 2, ak = lane & 3;  // fragment coordinates
  if (COMPRESSED) {
    // ---- Ys = Vt * Xs: warp -> column tile nt, reduction slice kh; rank tiles in chunks of kM2LChunk
    constexpr int kKSplit = NW / kNT;  // warps sharing one column tile split the P-long reduction
    const int nt = warp % kNT, kh = warp / kNT;
    const int mtiles = rank_pad >> 3;
    const int ksteps = P4 >> 2;
    const int k_begin = (int)((long long)ksteps * kh / kKSplit), k_end = (int)((long long)ksteps * (kh + 1) / kKSplit);
    const double *bx = Xs + (size_t)(nt * 8 + ar) * Pp + ak;
    for (int m0 = 0; m0 < mtiles; m0 += kM2LChunk) {
      double acc[kM2LChunk][2];
#pragma unroll
      for (int i = 0; i < kM2LChunk; ++i) acc[i][0] = acc[i][1] = 0.0;
      const double *af = VtF + ((size_t)m0 * ksteps) * 32 + lane;
#pragma unroll 4
      for (int ks = k_begin; ks < k_end; ++ks) {
        const double b = bx[ks * 4];
#pragma unroll
        for (int i = 0; i < kM2LChunk; ++i)
          if (m0 + i < mtiles) dmma884(acc[i][0], acc[i][1], __ldg(af + ((size_t)i * ksteps + ks) * 32), b);
      }
      // the reduction slices take turns adding their partial products into the single Ys buffer
      for (int turn = 0; turn < kKSplit; ++turn) {
        if (turn == kh) {
#pragma unroll
          for (int i = 0; i < kM2LChunk; ++i)
            if (m0 + i < mtiles) {
              double *y = Ys + (size_t)((m0 + i) * 8 + ar) * kM2LColsPad + nt * 8 + ak * 2;
              if (turn == 0) {
                y[0] = acc[i][0];
                y[1] = acc[i][1];
              } else {
                y[0] += acc[i][0];
                y[1] += acc[i][1];
              }
            }
        }
        __syncthreads();
      }
    }
  }
  // ---- Zs = U * Ys (or K * Xs)
  const int mt_total = (P + 7) >> 3;
  const int ksteps2 = (COMPRESSED ? rank_pad : P4) >> 2;
  // operator fragments are read once per CTA (no reuse to hide their L2 latency behind): blocks of kM2LPre k-steps
  // are double buffered in registers, the next block's loads issued before the current block's DMMAs
  const int kblocks = (ksteps2 + kM2LPre - 1) / kM2LPre;
  const int my_tiles = mt_total > warp ? (mt_total - warp + NW - 1) / NW : 0;
  const int nblocks = my_tiles * kblocks;
  double a_cur[kM2LPre], a_nxt[kM2LPre];
  auto load_block = [&](int blk, double (&dst)[kM2LPre]) {
    const int mt = warp + NW * (blk / kblocks), ks0 = (blk % kblocks) * kM2LPre;
    const double *af = UF + ((size_t)mt * ksteps2 + ks0) * 32 + lane;
#pragma unroll
    for (int u = 0; u < kM2LPre; ++u) dst[u] = ks0 + u < ksteps2 ? __ldg(af + (size_t)u * 32) : 0.0;
  };
  if (nblocks > 0) load_block(0, a_cur);
  double z[kNT][2];
#pragma unroll
  for (int i = 0; i < kNT; ++i) z[i][0] = z[i][1] = 0.0;
  for (int blk = 0; blk < nblocks; ++blk) {
    if (blk + 1 < nblocks) load_block(blk + 1, a_nxt);
    const int mt = warp + NW * (blk / kblocks), kb = blk % kblocks, ks0 = kb * kM2LPre;
#pragma unroll
    for (int u = 0; u < kM2LPre; ++u) {
      const int ks = ks0 + u;
      if (ks < ksteps2) {
#pragma unroll
        for (int nt = 0; nt < kNT; ++nt) {
          const double b = COMPRESSED ? Ys[(size_t)(ks * 4 + ak) * kM2LColsPad + nt * 8 + ar]
                                      : Xs[(size_t)(nt * 8 + ar) * Pp + ks * 4 + ak];
          dmma884(z[nt][0], z[nt][1], a_cur[u], b);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < kM2LPre; ++u) a_cur[u] = a_nxt[u];
    if (kb + 1 < kblocks) continue;
    const int m = mt * 8 + ar;
    if (m < P) {
#pragma unroll
      for (int nt = 0; nt < kNT; ++nt)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int c = nt * 8 + ak * 2 + h;
          if (COMPRESSED) {
            Xs[(size_t)c * Pp + m] = z[nt][h];  // Zs: Xs is no longer read once Ys is complete
          } else {  // the dense operator still reads Xs: scatter straight from the fragments
            const int tg = s_tgt[c];
            if (tg < 0) continue;
            const int *pm = perm_tab + (size_t)s_perm[c] * P;
            atomicAdd(loc + ((size_t)tg * nrhs + s_rhs[c]) * coef_stride(P) + __ldg(pm + m), z[nt][h]);  // L[perm[m]] += y[m]
          }
        }
    }
#pragma unroll
    for (int i = 0; i < kNT; ++i) z[i][0] = z[i][1] = 0.0;
  }
  if (!COMPRESSED) return;
  __syncthreads();
  // ---- flush: L_tgt[i] += sum_{c in run} Zs[c][inv_perm_c[i]]; four gathers in flight per lane
  const int nchunks = (P + 31) >> 5;
  const int nitems = s_nruns * nchunks;  // (run, 32-node chunk) pairs, dealt round-robin to the warps
  for (int item = warp; item < nitems; item += NW) {
    const int run = item / nchunks, i = (item - run * nchunks) * 32 + lane;
    const int c0 = s_runs[run];
    const int len = s_len[c0];
    const int *lst = s_list + s_off[c0];
    if (i < P) {
      double v = 0.0;
      for (int k = 0; k < len; k += 4) {
        int cc[4], id[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          cc[u] = lst[min(k + u, len - 1)];
          id[u] = __ldg(inv_tab + (size_t)s_perm[cc[u]] * P + i);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const double x = Xs[(size_t)cc[u] * Pp + id[u]];
          if (k + u < len) v += x;
        }
      }
      atomicAdd(loc + ((size_t)s_tgt[c0] * nrhs + s_rhs[c0]) * coef_stride(P) + i, v);
    }
  }
}

// L2P: out[t] = S(x_t) . L_leaf (+ gradients); one CTA per target tile (bbfmm.rs:1358-1440)
__global__ void __launch_bounds__(kTile) k_l2p(const TargetSet ts, const int *leaf_cell, const double *loc,
                                               const double *ccx, const double *ccy, const double *ccz,
                                               const double *chalf, const double *tnodes, int p, int dim, int P,
                                               int nrhs, double *out, double *gout) {
  extern __shared__ double sm[];
  const int tile = blockIdx.x;
  if (tile >= *ts.n_tiles_dev) return;
  const int li = ts.tile_leaf[tile];
  const int tb = ts.leaf_begin[li] + ts.tile_off[tile];
  const int cnt = min(kTile, ts.leaf_end[li] - tb);
  const int tid = threadIdx.x;
  const int c = leaf_cell[li];
  double *tn = sm;                 // p*p
  double *L = tn + p * p;          // P (one rhs at a time)
  double *S = L + P;               // [kTile][dim][p]
  double *dS = S + kTile * dim * p;  // [kTile][dim][p] when gradients
  for (int i = tid; i < p * p; i += kTile) tn[i] = tnodes[i];
  __syncthreads();
  const bool active = tid < cnt;
  const double half = chalf[c];
  if (active) {
    const double cc[3] = {ccx[c], ccy[c], ccz[c]};
    const double xs[3] = {ts.x[tb + tid], ts.y[tb + tid], ts.z[tb + tid]};
    for (int d = 0; d < dim; ++d) {
      const double x = (xs[d] - cc[d]) / half;
      cheb_s(p, x, tn, &S[(tid * dim + d) * p], gout ? &dS[(tid * dim + d) * p] : nullptr, 1.0 / half);
    }
  }
  const int p1 = dim > 1 ? p : 1, p2 = dim > 2 ? p : 1;
  const size_t row = active ? ts.out_row[tb + tid] : 0;
  for (int r = 0; r < nrhs; ++r) {
    __syncthreads();
    const double *src = loc + ((size_t)c * nrhs + r) * coef_stride(P);
    for (int i = tid; i < P; i += kTile) L[i] = src[i];
    __syncthreads();
    if (!active) continue;
    const double *S0 = &S[(tid * dim + 0) * p];
    const double *S1 = dim > 1 ? &S[(tid * dim + 1) * p] : nullptr;
    const double *S2 = dim > 2 ? &S[(tid * dim + 2) * p] : nullptr;
    double v = 0.0, g0 = 0.0, g1 = 0.0, g2 = 0.0;
    for (int i0 = 0; i0 < p; ++i0) {
      double a1 = 0.0, a1d1 = 0.0, a1d2 = 0.0;
      for (int i1 = 0; i1 < p1; ++i1) {
        double a2 = 0.0, a2d = 0.0;
        const double *Lp = L + (i0 * p1 + i1) * p2;
        if (dim > 2) {
          for (int i2 = 0; i2 < p2; ++i2) {
            a2 += S2[i2] * Lp[i2];
            if (gout) a2d += dS[(tid * dim + 2) * p + i2] * Lp[i2];
          }
        } else {
          a2 = Lp[0];
        }
        const double s1 = dim > 1 ? S1[i1] : 1.0;
        a1 += s1 * a2;
        if (gout) {
          if (dim > 1) a1d1 += dS[(tid * dim + 1) * p + i1] * a2;
          a1d2 += s1 * a2d;
        }
      }
      v += S0[i0] * a1;
      if (gout) {
        g0 += dS[(tid * dim + 0) * p + i0] * a1;
        g1 += S0[i0] * a1d1;
        g2 += S0[i0] * a1d2;
      }
    }
    out[row * nrhs + r] += v;
    if (gout) {
      double *gp = gout + row * (size_t)(nrhs * dim) + (size_t)r * dim;
      gp[0] += g0;
      if (dim > 1) gp[1] += g1;
      if (dim > 2) gp[2] += g2;
    }
  }
}

}  // namespace fb
