// Symmetric P2P for the matvec case targets == sources, one right-hand side (the solver's and the bench's hot call).
// In a partitioned tree (comm.cu) a rank runs it for the chunks of its own Morton range [own_lo, own_hi) only: a chunk
// still takes ALL sources behind it, whoever owns them, and the source-side sums of foreign rows travel in the result
// all-reduce — every unordered pair of the whole cloud is evaluated exactly once across the ranks, nothing twice.
// Reference: particle_to_particle bbfmm.rs:1162-1251 — there every (target, source) pair of the U lists is evaluated;
// here each unordered pair is evaluated ONCE and serves both rows:
//     out[t] += k(t, s) w[s]      and      out[s] += k(t, s) w[t]        (all registry kernels are symmetric).
// U is a symmetric relation (adjacent leaves at any level + the leaf itself, linear_tree.rs:177-395 / :397-485), and the
// sources are stored in Morton order, so "each unordered pair once" = a warp owning the consecutive sorted positions
// [tb, tb + cnt) of a leaf takes the part of the leaf's merged U ranges that lies AFTER its own chunk (symmetric
// tiles), plus its own cnt x cnt diagonal block.  One right-hand side runs k_p2p_sym_blocked (a warp per 128-target
// tile, below); 2 - 4 right-hand sides, and one when FB_GENERIC_P2P=1, run k_p2p_sym (a warp per 64 targets).
//
// Cost model (tools/fp64_ubench.cu, tools/dmma_bench.cu): the FP64 pipe is the only resource (DMMA shares it, MUFU.RSQ64H
// serialises with it), 10 DFMA + 1 MUFU per evaluation = 7.2 clk per warp step on an SM.  The symmetric step adds one
// DMUL (k w[t]) and, amortised, one DADD of the source-side reduction: 8.3 clk for TWO pairs — 1.75x fewer pipe cycles
// per pair.  Source side: lane l parks k(t_l, s_j) w[t_l] in a warp-private shared-memory matrix part[j][l] (row stride
// 33: conflict-free both ways); after the tile, lane j sums row j in a fixed order and issues one RED to out[s_j].
// Target-side sums stay in registers and are added with one RED per target at the end (other warps' source-side REDs
// hit the same rows concurrently).  Values are the reference's own per-pair values; only the summation order differs.
#include "fmm.h"

#include <algorithm>
#include <atomic>
#include <cstdlib>

namespace fb {

constexpr int kSymWPC = 4;       // warps per CTA
constexpr int kSymStride = 33;   // row stride of the partial-sum matrix (doubles)

// NR right-hand sides per pass (1, 2 or 4): the kernel value of a pair is computed once and serves 2 NR accumulations.
// The source-side partial sums need NR matrices, so tiles shrink to 16 / 8 sources for NR = 2 / 4 (shared memory per
// warp: 10.5 / 11.4 / 12.5 KB; with 16-source tiles NR = 4 fitted two CTAs per SM and gained 9 % on the 2-D thin-plate
// config where the model says 40 %).
template <int NR>
struct SymWarpSmem {
  static constexpr int TS = NR == 1 ? 32 : (NR == 2 ? 16 : 8);  // sources per tile
  static constexpr int NV = 2 + NR / 2;         // double2 planes per source: {x, y}, {z, w0}, {w1, w2}, {w3, -}
  double2 st[2][NV][32];                        // double-buffered source tile (32 slots: the diagonal block uses them all)
  double part[NR * TS * kSymStride];            // part[r][j][l] = sum over the lane's targets of k(t, s_j) w_r[t]
};

template <int NR>
__device__ __forceinline__ void sym_unpack_w(const double2 (*t)[32], int j, double z_w0_y, double (&ws)[NR]) {
  ws[0] = z_w0_y;
  if (NR >= 2) {
    const double2 p2 = t[2][j];
    ws[1] = p2.x;
    if (NR >= 3) ws[2] = p2.y;
  }
  if (NR >= 4) ws[3] = t[3][j].x;
}

// A warp owns up to 64 consecutive sorted positions of a leaf, lane l the targets tb + l and (TWO) tb + 32 + l: every
// staged source then serves two evaluations per lane, which halves the shared-memory traffic per pair (source broadcasts,
// partial-sum stores and the row sums of the flush; ncu on the one-target version: l1tex 70 % busy, FP64 pipe 48 %) and
// doubles the independent chains in flight.  Chunks of <= 32 targets take the one-target instantiation.
// split > 1 (grids too small to fill the GPU, e.g. one rank's share): `split` warps share a chunk, warp `part` takes
// every split-th source tile (part 0 also the diagonal block); all sums leave through REDs, so nothing else changes.
template <int FAM, bool FAST, bool TWO, int NR>
__device__ __forceinline__ void p2p_sym_body(const DirectArgs &a, SymWarpSmem<NR> &sm, const int li, const int tb,
                                             const int cnt, const int lane, const int split, const int part) {
  constexpr int NT = TWO ? 2 : 1;
  constexpr int TS = SymWarpSmem<NR>::TS;
  constexpr double kScale = kernel_weight_scale<FAM, FAST>();
  const int a_end = tb + cnt;
  double xt[NT], yt[NT], zt[NT], wt[NT][NR], acc[NT][NR];
#pragma unroll
  for (int u = 0; u < NT; ++u) {
    const int i = 32 * u + lane;
    xt[u] = yt[u] = zt[u] = 0.0;
#pragma unroll
    for (int r = 0; r < NR; ++r) wt[u][r] = acc[u][r] = 0.0;
    if (i < cnt) {
      xt[u] = a.sx[tb + i];
      yt[u] = a.sy[tb + i];
      zt[u] = a.sz[tb + i];
#pragma unroll
      for (int r = 0; r < NR; ++r) wt[u][r] = a.w[(size_t)(a.rhs0 + r) * a.n + tb + i] * kScale;
    }
  }
  auto park = [&](int buf, double x, double y, double z, const double (&w)[NR]) {  // this lane's source slot of a tile
    sm.st[buf][0][lane] = make_double2(x, y);
    sm.st[buf][1][lane] = make_double2(z, w[0]);
    if (NR >= 2) sm.st[buf][2][lane] = make_double2(w[1], NR >= 3 ? w[2] : 0.0);
    if (NR >= 4) sm.st[buf][3][lane] = make_double2(w[3], 0.0);
  };
  // ---- diagonal block: the chunk against itself, every ordered pair (self term included, as the reference does)
#pragma unroll
  for (int h = 0; h < NT; ++h) park(h, xt[h], yt[h], zt[h], wt[h]);
  __syncwarp();
#pragma unroll
  for (int h = 0; h < NT; ++h) {
    const int mh = part == 0 ? min(32, cnt - 32 * h) : 0;
#pragma unroll 2
    for (int j = 0; j < mh; ++j) {
      const double2 p0 = sm.st[h][0][j], p1 = sm.st[h][1][j];
      double ws[NR];
      sym_unpack_w<NR>(sm.st[h], j, p1.y, ws);
#pragma unroll
      for (int u = 0; u < NT; ++u) {
        const double dx = xt[u] - p0.x, dy = yt[u] - p0.y, dz = zt[u] - p1.x;
        double r2 = dx * dx;
        r2 += dy * dy;
        r2 += dz * dz;
        const double v = kernel_mag<FAM, FAST, true>(r2, a.kp);
#pragma unroll
        for (int r = 0; r < NR; ++r) kernel_acc<FAM>(acc[u][r], v, ws[r]);
      }
    }
  }
  __syncwarp();

  // ---- symmetric tiles: the part of the merged U ranges behind the chunk
  long long e = a.u_ptr[li];
  const long long e_end = a.u_ptr[li + 1];
  int pos = 0, end = 0;  // current clipped range [pos, end)
  auto next_range = [&]() {
    while (e < e_end) {
      const int b = a.u_begin[e], n = a.u_count[e];
      ++e;
      pos = max(b, a_end);
      end = b + n;
      if (pos < end) return;
    }
    pos = end = 0;
  };
  next_range();
  double rx = 0, ry = 0, rz = 0, rw[NR];
#pragma unroll
  for (int r = 0; r < NR; ++r) rw[r] = 0.0;
  int base_next = 0;
  int skip = part;  // tiles to pass over before the next one of this warp
  auto fetch = [&](int &m) {  // this lane's element of the next tile of this warp, then advance
    for (;;) {
      m = min(TS, end - pos);
      if (m <= 0) {
        m = 0;
        return;
      }
      const bool mine = skip == 0;
      skip = mine ? split - 1 : skip - 1;
      if (mine) {
        base_next = pos;
        if (lane < m) {
          rx = a.sx[pos + lane];
          ry = a.sy[pos + lane];
          rz = a.sz[pos + lane];
#pragma unroll
          for (int r = 0; r < NR; ++r) rw[r] = a.w[(size_t)(a.rhs0 + r) * a.n + pos + lane] * kScale;
        }
      }
      pos += m;
      if (pos >= end) next_range();
      if (mine) return;
    }
  };
  int m_cur = 0, m_next = 0, buf = 0, base_cur = 0;
  fetch(m_cur);
  base_cur = base_next;
  if (lane < m_cur) park(0, rx, ry, rz, rw);
  __syncwarp();
  while (m_cur > 0) {
    fetch(m_next);  // global loads of the next tile overlap the arithmetic below
    const double2(*t)[32] = sm.st[buf];
    double *pl = sm.part + lane;
#pragma unroll 4
    for (int j = 0; j < m_cur; ++j) {
      const double2 p0 = t[0][j], p1 = t[1][j];
      double ws[NR], ps[NR];
      sym_unpack_w<NR>(t, j, p1.y, ws);
#pragma unroll
      for (int u = 0; u < NT; ++u) {
        const double dx = xt[u] - p0.x, dy = yt[u] - p0.y, dz = zt[u] - p1.x;
        double r2 = dx * dx;
        r2 += dy * dy;
        r2 += dz * dz;
        const double v = kernel_mag<FAM, FAST, true>(r2, a.kp);
#pragma unroll
        for (int r = 0; r < NR; ++r) {
          kernel_acc<FAM>(acc[u][r], v, ws[r]);
          ps[r] = u == 0 ? v * wt[0][r] : fma(v, wt[u][r], ps[r]);
        }
      }
#pragma unroll
      for (int r = 0; r < NR; ++r) pl[(r * TS + j) * kSymStride] = ps[r];
    }
    __syncwarp();
    // source side: row (r, j) of the partial sums, fixed order, one RED per (source, right-hand side)
    for (int q = lane; q < m_cur * NR; q += 32) {
      const int r = q / m_cur, j = q - r * m_cur;
      const double *pr = sm.part + (r * TS + j) * kSymStride;
      double sp[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) sp[k] = pr[k];
#pragma unroll
      for (int l = 8; l < 32; l += 8)
#pragma unroll
        for (int k = 0; k < 8; ++k) sp[k] += pr[l + k];
      const double s = ((sp[0] + sp[1]) + (sp[2] + sp[3])) + ((sp[4] + sp[5]) + (sp[6] + sp[7]));
      atomicAdd(a.out + (size_t)a.sym_row[base_cur + j] * a.nrhs + a.rhs0 + r, FAM == KF_LINEAR ? -s : s);
    }
    buf ^= 1;
    if (lane < m_next) park(buf, rx, ry, rz, rw);
    __syncwarp();
    m_cur = m_next;
    base_cur = base_next;
  }
#pragma unroll
  for (int u = 0; u < NT; ++u) {
    const int i = 32 * u + lane;
    if (i < cnt)
#pragma unroll
      for (int r = 0; r < NR; ++r) atomicAdd(a.out + (size_t)a.sym_row[tb + i] * a.nrhs + a.rhs0 + r, acc[u][r]);
  }
}

template <int FAM, bool FAST, int NR>
__global__ void __launch_bounds__(kSymWPC * 32, NR == 1 ? 5 : (NR == 2 ? 4 : 3)) k_p2p_sym(const DirectArgs a, const int split) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long gw = (long long)blockIdx.x * kSymWPC + warp;
  const long long chunk = gw / split;
  const int part = (int)(gw - chunk * split);
  const int tile = (int)(chunk >> 1), sub = (int)(chunk & 1);  // a tile holds <= kTile = 128 targets: two warps of <= 64
  if (tile >= *a.ts.n_tiles_dev) return;
  const int li = a.ts.tile_leaf[tile];
  // target i of the set is the source at the sorted position own_lo + i
  const int tb = a.ts.own_lo + a.ts.leaf_begin[li] + a.ts.tile_off[tile] + sub * 64;
  const int cnt = min(64, a.ts.own_lo + a.ts.leaf_end[li] - tb);
  if (cnt <= 0) return;
  extern __shared__ __align__(16) unsigned char dsm_raw[];
  SymWarpSmem<NR> &sm = reinterpret_cast<SymWarpSmem<NR> *>(dsm_raw)[warp];
  if (cnt > 32) p2p_sym_body<FAM, FAST, true, NR>(a, sm, li, tb, cnt, lane, split, part);
  else p2p_sym_body<FAM, FAST, false, NR>(a, sm, li, tb, cnt, lane, split, part);
}

// ---- one right-hand side: a warp per kTile = 128-target tile, NT = 1, 2 or 4 targets per lane -------------------------
// Lane l owns the targets 32 u + l (u < NT) of the tile, NT picked from the tile's count so that a short leaf does not
// run the four-target body on empty slots.  Per staged source: one broadcast of {x, y}, {z, w}, NT evaluations, the NT
// source-side terms combined in registers (one DMUL + NT - 1 DFMA) and ONE store to part[j][l]: with NT = 4 that is a
// quarter of the shared-memory stores, half the source broadcasts and a quarter of the flush per pair of the two-target
// body above.  Flush: lane j sums row j in a fixed order (LDS.128, rows 34 doubles apart: 8 lanes of a quarter-warp
// hit 8 distinct 16-byte bank groups) and issues one RED; no per-source loop, so no divergent collective.
// Source tiles are gathered across the merged U ranges (a tile ends only where the sources behind the tile end), so
// the inner loop runs 32 trips everywhere but in the last tile.
// split: as in k_p2p_sym, `split` warps share a tile and take every split-th source tile (part 0 also the diagonal).
// Order: with a warp per tile, a big leaf's tile (a depth-4 leaf of about 240 points in a 1M-point uniform cloud) holds
// about 15x the pairs of a small leaf's, so in tile order the pass ends in a tail of them (2.51-2.56 ms against 2.40 for
// k_p2p_sym on a B200).  The all-sources set lists its tiles by descending (targets x sources behind them), and the
// warps take them in that order (TargetSet::sym_tile_order): 1.89 ms (profiles/r5_p2p_order.json).  Giving the big
// tiles two warps instead reached 2.21 ms in tile order and 2.01 ms heaviest first.
// Diagonal: the tile's own block, sub-block pairs (u < g) of 32 x 32 once each (source block g is the targets 32 g + j,
// its source-side sums land in the owning lane's accumulator); only the 32 x 32 self-blocks run in full, self term
// included as the reference does.
constexpr int kBlkWPC = 4;       // warps per CTA
constexpr int kBlkStride = 34;   // row stride of the partial-sum matrix (doubles): even, for the LDS.128 row reads

struct BlkWarpSmem {
  double2 st[2][2][32];           // double-buffered source tile: {x, y}, {z, w}
  double part[32 * kBlkStride];   // part[j][l] = sum over lane l's targets of k(t, s_j) w[t]
};

// row j of the partial sums, fixed order
__device__ __forceinline__ double blk_row_sum(const BlkWarpSmem &sm, int j) {
  const double2 *pr = reinterpret_cast<const double2 *>(sm.part + j * kBlkStride);
  double2 q[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) q[k] = pr[k];
#pragma unroll
  for (int l = 4; l < 16; l += 4)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const double2 v = pr[l + k];
      q[k].x += v.x;
      q[k].y += v.y;
    }
  return ((q[0].x + q[0].y) + (q[1].x + q[1].y)) + ((q[2].x + q[2].y) + (q[3].x + q[3].y));
}

template <int FAM, bool FAST, int NT>
__device__ __forceinline__ void p2p_blk_body(const DirectArgs &a, BlkWarpSmem &sm, const int li, const int tb,
                                             const int cnt, const int lane, const int split, const int part) {
  constexpr double kScale = kernel_weight_scale<FAM, FAST>();
  const int a_end = tb + cnt;
  double xt[NT], yt[NT], zt[NT], wt[NT], acc[NT];
#pragma unroll
  for (int u = 0; u < NT; ++u) {
    const int i = 32 * u + lane;
    xt[u] = yt[u] = zt[u] = wt[u] = acc[u] = 0.0;
    if (i < cnt) {
      xt[u] = a.sx[tb + i];
      yt[u] = a.sy[tb + i];
      zt[u] = a.sz[tb + i];
      wt[u] = a.w[(size_t)a.rhs0 * a.n + tb + i] * kScale;
    }
  }
  double *pl = sm.part + lane;

  // ---- diagonal block (split part 0)
  if (part == 0) {
#pragma unroll
    for (int g = 0; g < NT; ++g) {
      const int mg = min(32, cnt - 32 * g);  // warp-uniform
      if (mg <= 0) break;
      sm.st[g & 1][0][lane] = make_double2(xt[g], yt[g]);
      sm.st[g & 1][1][lane] = make_double2(zt[g], wt[g]);
      __syncwarp();
      const double2(*t)[32] = sm.st[g & 1];
#pragma unroll 2
      for (int j = 0; j < mg; ++j) {
        const double2 p0 = t[0][j], p1 = t[1][j];
        double ps = 0.0;
#pragma unroll
        for (int u = 0; u <= g; ++u) {
          const double dx = xt[u] - p0.x, dy = yt[u] - p0.y, dz = zt[u] - p1.x;
          double r2 = dx * dx;
          r2 += dy * dy;
          r2 += dz * dz;
          const double v = kernel_mag<FAM, FAST, true>(r2, a.kp);
          kernel_acc<FAM>(acc[u], v, p1.y);
          if (u < g) ps = u == 0 ? v * wt[0] : fma(v, wt[u], ps);
        }
        if (g > 0) pl[j * kBlkStride] = ps;
      }
      if (g > 0) {
        __syncwarp();
        const double s = blk_row_sum(sm, lane);  // source side of target 32 g + lane: this lane's own row
        if (lane < mg) kernel_acc<FAM>(acc[g], s, 1.0);
        __syncwarp();
      }
    }
  }
  __syncwarp();

  // ---- symmetric tiles: the part of the merged U ranges behind the tile
  long long e = a.u_ptr[li];
  const long long e_end = a.u_ptr[li + 1];
  int pos = 0, end = 0;  // current clipped range [pos, end)
  auto next_range = [&]() {
    while (e < e_end) {
      const int b = a.u_begin[e], n = a.u_count[e];
      ++e;
      pos = max(b, a_end);
      end = b + n;
      if (pos < end) return;
    }
    pos = end = 0;
  };
  next_range();
  double rx = 0, ry = 0, rz = 0, rw = 0;
  int rp = 0;       // sorted position of this lane's source in the fetched tile
  int skip = part;  // tiles to pass over before the next one of this warp
  auto fetch = [&](int &m) {  // the next tile of this warp: up to 32 sources gathered across ranges, this lane's one
    for (;;) {
      m = 0;
      if (pos >= end) return;
      const bool mine = skip == 0;
      skip = mine ? split - 1 : skip - 1;
      while (m < 32 && pos < end) {
        const int k = min(32 - m, end - pos);
        if (mine && lane >= m && lane < m + k) {
          rp = pos + lane - m;
          rx = a.sx[rp];
          ry = a.sy[rp];
          rz = a.sz[rp];
          rw = a.w[(size_t)a.rhs0 * a.n + rp] * kScale;
        }
        m += k;
        pos += k;
        if (pos >= end) next_range();
      }
      if (mine) return;
    }
  };
  int m_cur = 0, m_next = 0, buf = 0;
  fetch(m_cur);
  int rp_cur = rp;
  if (lane < m_cur) {
    sm.st[0][0][lane] = make_double2(rx, ry);
    sm.st[0][1][lane] = make_double2(rz, rw);
  }
  __syncwarp();
  while (m_cur > 0) {
    fetch(m_next);  // global loads of the next tile overlap the arithmetic below
    const double2(*t)[32] = sm.st[buf];
#pragma unroll 2
    for (int j = 0; j < m_cur; ++j) {
      const double2 p0 = t[0][j], p1 = t[1][j];
      double ps;
#pragma unroll
      for (int u = 0; u < NT; ++u) {
        const double dx = xt[u] - p0.x, dy = yt[u] - p0.y, dz = zt[u] - p1.x;
        double r2 = dx * dx;
        r2 += dy * dy;
        r2 += dz * dz;
        const double v = kernel_mag<FAM, FAST, true>(r2, a.kp);
        kernel_acc<FAM>(acc[u], v, p1.y);
        ps = u == 0 ? v * wt[0] : fma(v, wt[u], ps);
      }
      pl[j * kBlkStride] = ps;
    }
    __syncwarp();
    const double s = blk_row_sum(sm, lane);  // source side: row `lane`, one RED per source
    if (lane < m_cur) atomicAdd(a.out + (size_t)a.sym_row[rp_cur] * a.nrhs + a.rhs0, FAM == KF_LINEAR ? -s : s);
    buf ^= 1;
    if (lane < m_next) {
      sm.st[buf][0][lane] = make_double2(rx, ry);
      sm.st[buf][1][lane] = make_double2(rz, rw);
    }
    __syncwarp();
    m_cur = m_next;
    rp_cur = rp;
  }
#pragma unroll
  for (int u = 0; u < NT; ++u) {
    const int i = 32 * u + lane;
    if (i < cnt) atomicAdd(a.out + (size_t)a.sym_row[tb + i] * a.nrhs + a.rhs0, acc[u]);
  }
}

// 20 warps per SM where the body fits 96 registers without spills (linear in both square-root modes, cubic with the
// second-order one), else 16
template <int FAM, bool FAST>
constexpr int blk_min_ctas() {
  return (FAM == KF_LINEAR || (FAM == KF_CUBIC && FAST)) ? 5 : 4;
}

template <int FAM, bool FAST>
__global__ void __launch_bounds__(kBlkWPC * 32, blk_min_ctas<FAM, FAST>())
    k_p2p_sym_blocked(const DirectArgs a, const int split) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long gw = (long long)blockIdx.x * kBlkWPC + warp;
  const int slot = (int)(gw / split);
  const int part = (int)(gw - (long long)slot * split);
  if (slot >= *a.ts.n_tiles_dev) return;
  // the all-sources set lists its tiles heaviest first (fmm.cu): the big leaves start at the head of the grid
  const int tile = a.ts.sym_tile_order ? a.ts.sym_tile_order[slot] : slot;
  const int li = a.ts.tile_leaf[tile];
  // target i of the set is the source at the sorted position own_lo + i
  const int tb = a.ts.own_lo + a.ts.leaf_begin[li] + a.ts.tile_off[tile];
  const int cnt = min(kTile, a.ts.own_lo + a.ts.leaf_end[li] - tb);
  if (cnt <= 0) return;
  extern __shared__ __align__(16) unsigned char dsm_raw[];
  BlkWarpSmem &sm = reinterpret_cast<BlkWarpSmem *>(dsm_raw)[warp];
  if (cnt > 64) p2p_blk_body<FAM, FAST, 4>(a, sm, li, tb, cnt, lane, split, part);
  else if (cnt > 32) p2p_blk_body<FAM, FAST, 2>(a, sm, li, tb, cnt, lane, split, part);
  else p2p_blk_body<FAM, FAST, 1>(a, sm, li, tb, cnt, lane, split, part);
}

std::atomic<unsigned long long> g_p2p_blocked_launches{0};

// FB_GENERIC_P2P=1 keeps one-column passes on k_p2p_sym (A/B baseline)
static bool p2p_force_generic() {
  static const bool on = [] {
    const char *v = std::getenv("FB_GENERIC_P2P");
    return v && v[0] == '1';
  }();
  return on;
}

template <int FAM>
static void p2p_blocked_launch(const DirectArgs &a, cudaStream_t s) {
  static_assert(kTile == 128, "four 32-target blocks per tile");
  const size_t smem = sizeof(BlkWarpSmem) * kBlkWPC;
  // about three waves of warps (148 SMs x 20 resident warps) keep the uneven tiles from leaving SMs idle at the end
  const long long tiles = std::max<long long>(1, (long long)(a.ts.m / kTile));
  const int split = (int)std::min<long long>(8, std::max<long long>(1, (148 * 20 * 3) / tiles));
  const unsigned grid = (unsigned)(((long long)a.ts.max_tiles * split + kBlkWPC - 1) / kBlkWPC);
  if (kernel_has_fast<FAM>() && a.kp.fast) {
    constexpr bool F = kernel_has_fast<FAM>();
    FB_CUDA(cudaFuncSetAttribute(k_p2p_sym_blocked<FAM, F>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    FB_LAUNCH((k_p2p_sym_blocked<FAM, F>), grid, kBlkWPC * 32, smem, s, a, split);
  } else {
    FB_CUDA(cudaFuncSetAttribute(k_p2p_sym_blocked<FAM, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    FB_LAUNCH((k_p2p_sym_blocked<FAM, false>), grid, kBlkWPC * 32, smem, s, a, split);
  }
  g_p2p_blocked_launches.fetch_add(1, std::memory_order_relaxed);
}

template <int FAM, int NR>
static void p2p_sym_launch(const DirectArgs &a, cudaStream_t s) {
  static_assert(kTile == 128, "two 64-target warps per tile");
  if (NR == 1 && !p2p_force_generic()) {
    p2p_blocked_launch<FAM>(a, s);
    return;
  }
  const size_t smem = sizeof(SymWarpSmem<NR>) * kSymWPC;
  // about three waves of warps (148 SMs x 20 resident warps) keep the uneven chunks from leaving SMs idle at the end
  const long long chunks = std::max<long long>(1, (long long)(a.ts.m / 64));
  const int split = (int)std::min<long long>(8, std::max<long long>(1, (148 * 20 * 3) / chunks));
  const unsigned grid = (unsigned)(((long long)a.ts.max_tiles * 2 * split + kSymWPC - 1) / kSymWPC);
  if (kernel_has_fast<FAM>() && a.kp.fast) {
    constexpr bool F = kernel_has_fast<FAM>();
    FB_CUDA(cudaFuncSetAttribute(k_p2p_sym<FAM, F, NR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    FB_LAUNCH((k_p2p_sym<FAM, F, NR>), grid, kSymWPC * 32, smem, s, a, split);
  } else {
    FB_CUDA(cudaFuncSetAttribute(k_p2p_sym<FAM, false, NR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    FB_LAUNCH((k_p2p_sym<FAM, false, NR>), grid, kSymWPC * 32, smem, s, a, split);
  }
}

// 1 .. 4 right-hand sides: one pass of 4, 2 or 1 columns at a time (3 = 2 + 1)
template <int FAM>
static void p2p_sym_fam(DirectArgs a, cudaStream_t s) {
  const int r_end = a.rhs0 + a.nrhs_pass;
  while (a.rhs0 < r_end) {
    const int left = r_end - a.rhs0;
    if (left >= 4) {
      p2p_sym_launch<FAM, 4>(a, s);
      a.rhs0 += 4;
    } else if (left >= 2) {
      p2p_sym_launch<FAM, 2>(a, s);
      a.rhs0 += 2;
    } else {
      p2p_sym_launch<FAM, 1>(a, s);
      a.rhs0 += 1;
    }
  }
}

// true when the symmetric kernel serves this call: values only, at most four right-hand sides (beyond that the kernel
// value is cheap next to the 2 K accumulations and the one-pass general kernel wins), targets = the tree's own sources
// or a rank's Morton-contiguous share of them
bool p2p_sym_applicable(const DirectArgs &a) {
  static const bool off = [] {
    const char *v = std::getenv("FB_P2P_SYM");
    return v && v[0] == '0';
  }();
  return !off && !a.gout && a.nrhs >= 1 && a.nrhs <= 4 && a.ts.own_hi > a.ts.own_lo && a.sym_row != nullptr && a.ts.max_tiles > 0 &&
         a.kp.fast != 3;
}

void launch_p2p_sym(const DirectArgs &a0, cudaStream_t s) {
  DirectArgs a = a0;
  a.rhs0 = 0;
  a.nrhs_pass = a.nrhs;
#define CALL(F) p2p_sym_fam<F>(a, s)
  FB_FAM_SWITCH(a.kp.fam, CALL)
#undef CALL
}

}  // namespace fb

uint64_t fb_p2p_blocked_launch_count(void) { return fb::g_p2p_blocked_launches.load(); }
