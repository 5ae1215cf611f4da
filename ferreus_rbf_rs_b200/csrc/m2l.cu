// Streaming M2L (bbfmm.rs:864-986): the compressed multipole-to-local translation as two dense contractions on the
// FP64 tensor cores, with every operand moved by the TMA engine.
//
// The reference applies 16 (3-D) / 7 (2-D) symmetric reference operators through a permutation of the source
// coefficients and the inverse permutation of the result.  Here the permutations are folded into the operators once at
// build time (k_m2l_expand: Vt_t[r][i] = Vt_ref[r][inv[i]], U_t[i][r] = U_ref[inv[i]][r] for each of the <= 316 transfer
// vectors t of a level — the same products in another summation order), so an entry of the V lists is
//       L_target += U_t (Vt_t M_source)
// with M_source and L_target contiguous P-long columns.  The work of a (level, t) group is a stream of such columns:
//   * a producer warp gathers 16 source columns per stage with cp.async.bulk (UBLKCP) into a 4-stage ring, completion
//     on an mbarrier (SYNCS);
//   * 8 MMA warps hold the group's operators in REGISTERS in DMMA fragment order — warp w owns the k-slice w of Vt_t
//     (first contraction, Y = Vt_t X, split over the P-long reduction) and the row tiles w, w + 8, .. of U_t (second
//     contraction, Z = U_t Y) — so the only shared-memory operand traffic is one B fragment per 3-6 DMMAs;
//   * the k-slice partial sums of Y are parked in the rows of the stage a warp alone reads, summed in a fixed order,
//     and Z overwrites the stage;
//   * the producer warp hands the finished columns to cp.reduce.async.bulk.add.f64 (UBLKRED): the TMA engine adds each
//     2.7 KB column into the locals in L2, no REDs are issued by the SM.
// Ranks above 24 are split into pieces of <= 24 (three 8-row tiles) so that the operator slices fit the register file.
// Measured ceilings of the data movement (tools/m2l_ubench.cu, profiles/r2_m2l_ubench.txt): UBLKCP ring 5.4-10 TB/s,
// UBLKRED f64 4.1-4.8 TB/s, against 2.5 GB each way per 1M-point matvec.
#include <algorithm>
#include <array>
#include <cstdlib>
#include <map>
#include <numeric>
#include <type_traits>

#include "fmm.h"

namespace fb {

constexpr int kStreamCols = 16;    // columns per stage
constexpr int kStreamStages = 4;
constexpr int kStreamMaxMt = 3;    // rank tiles (8 rows) per piece
constexpr int kStreamKsw = 8;      // k-steps of the first contraction per MMA warp
constexpr int kStreamMtw = 4;      // row tiles of the second contraction per MMA warp

struct M2LItemDev {
  long long entry_off;  // first entry (index into the stream entry arrays)
  int n_entries;
  int mt;               // rank tiles of the piece
  long long v_off, u_off;  // operator pool offsets (doubles), fragment order
};

struct M2LStreamArgs {
  const M2LItemDev *items;  // longest first
  int n_items;
  int *next_item;  // work counter, zeroed before the launch: CTAs pull items as they finish (no static tail)
  const int *e_tgt, *e_src;
  const double *pool;
  const uint8_t *flag;  // per cell: subtree has targets; null = every cell
  const double *mult;
  double *loc;
  int P, Ps, Pc, KS, MTU, nrhs;
};

// ---- PTX helpers ----------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *b, int cnt) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(cnt));
}
__device__ __forceinline__ void mbar_arrive_expect(unsigned long long *b, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long *b) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *b, unsigned parity) {
  asm volatile(
      "{\n.reg .pred p;\nWAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}\n" ::"r"(smem_u32(b)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_load(void *dst, const void *src, unsigned bytes, unsigned long long *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void bulk_red_add(double *dst, const void *src, unsigned bytes) {
  asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f64 [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void dmma(double &d0, double &d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}

// ---- operator expansion ---------------------------------------------------------------------------------------
struct M2LPieceDev {
  long long dense_u, dense_vt;  // offsets of the reference operator (column-major U P x rank, Vt rank x P)
  long long v_off, u_off;       // outputs
  int rank, r0, r1;             // the piece covers ranks [r0, r1)
  int perm;                     // symmetry permutation id
  int mt;
};

// one CTA per piece: Vt_t / U_t of the piece in DMMA fragment order, zero padded
//   VtF[(m * KS + ks) * 32 + lane] = Vt_t[r0 + m*8 + lane/4][ks*4 + lane%4]
//   UF [(t * KR + ks) * 32 + lane] = U_t [t*8 + lane/4][r0 + ks*4 + lane%4]          KR = 2 mt
__global__ void __launch_bounds__(256) k_m2l_expand(const M2LPieceDev *pieces, const double *dense, const int *inv_tab,
                                                    int P, int KS, int MTU, double *pool) {
  const M2LPieceDev pc = pieces[blockIdx.x];
  const int *inv = inv_tab + (size_t)pc.perm * P;
  const double *U = dense + pc.dense_u, *Vt = dense + pc.dense_vt;
  const int nv = pc.mt * KS * 32, KR = 2 * pc.mt, nu = MTU * KR * 32;
  for (int i = threadIdx.x; i < nv; i += blockDim.x) {
    const int lane = i & 31, f = i >> 5, ks = f % KS, m = f / KS;
    const int rr = pc.r0 + m * 8 + (lane >> 2), cc = ks * 4 + (lane & 3);
    pool[pc.v_off + i] = (rr < pc.r1 && cc < P) ? Vt[(size_t)inv[cc] * pc.rank + rr] : 0.0;
  }
  for (int i = threadIdx.x; i < nu; i += blockDim.x) {
    const int lane = i & 31, f = i >> 5, ks = f % KR, t = f / KR;
    const int row = t * 8 + (lane >> 2), rk = pc.r0 + ks * 4 + (lane & 3);
    pool[pc.u_off + i] = (row < P && rk < pc.r1) ? U[(size_t)rk * P + inv[row]] : 0.0;
  }
}

// ---- the streaming kernel -------------------------------------------------------------------------------------
// NW MMA warps + one producer warp.  Registers are allocated per 4 warps: 12 warps (NW = 11) or 9 warps (NW = 8, which
// the hardware rounds up to 12) leave 168 registers per thread, hence slices of <= 8 k-steps and <= 4 row tiles per warp:
// NW = 11 serves 261 <= P <= 352 (p = 7 in 3-D), NW = 8 serves 189 <= P <= 256 (p = 6 in 3-D).
template <int NW>
__global__ void __launch_bounds__((NW + 1) * 32, 1) k_m2l_stream(const M2LStreamArgs a) {
  constexpr int KSW = kStreamKsw, MTW = kStreamMtw;
  extern __shared__ __align__(128) double sm[];
  constexpr int S = kStreamStages, NC = kStreamCols, YS = NC + 4;
  const int Pc = a.Pc;
  double *stages = sm;                                  // [S][NC][Pc]
  double *Yb = stages + (size_t)S * NC * Pc;            // [2][24][YS]
  __shared__ unsigned long long full[S], zfull[S], pbar[2], ybar[2];
  __shared__ int s_ncols[S], s_item[S];
  __shared__ long long s_tgtoff[S][NC];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&zfull[s], NW);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&pbar[b], NW);
      mbar_init(&ybar[b], NW);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // stale shared memory must be finite: idle columns and pad rows are multiplied by zero operator entries
  for (int i = tid; i < S * NC * Pc + 2 * 24 * YS; i += blockDim.x) sm[i] = 0.0;
  __syncthreads();
  const unsigned col_bytes = (unsigned)a.Ps * 8u;

  if (warp == NW) {
    // ================================================================= producer warp: gathers and scatter-adds
    int j = 0;  // stages committed so far
    int have = 0;
    auto acquire = [&](int jj) {  // stage jj % S must be free: its previous occupant's Z goes out first
      if (jj < S) return;
      const int s = jj % S;
      mbar_wait(&zfull[s], (unsigned)((jj / S - 1) & 1));
      if (lane < s_ncols[s]) bulk_red_add(a.loc + s_tgtoff[s][lane], stages + ((size_t)s * NC + lane) * Pc, col_bytes);
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      __syncwarp();
    };
    auto commit = [&](int item, int ncols) {
      const int s = j % S;
      __syncwarp();
      if (lane == 0) {
        s_ncols[s] = ncols;
        s_item[s] = item;
        mbar_arrive_expect(&full[s], (unsigned)ncols * col_bytes);
      }
      __syncwarp();
      ++j;
    };
    for (;;) {
      int it = 0;
      if (lane == 0) it = atomicAdd(a.next_item, 1);
      it = __shfl_sync(0xffffffffu, it, 0);
      if (it >= a.n_items) break;
      const M2LItemDev im = a.items[it];
      const long long ncol_total = (long long)im.n_entries * a.nrhs;
      for (long long base = 0; base < ncol_total;) {
        const long long col = base + lane;
        bool valid = col < ncol_total;
        int tg = 0, r = 0;
        long long e = 0;
        if (valid) {
          e = col / a.nrhs;
          r = (int)(col - e * a.nrhs);
          tg = __ldg(a.e_tgt + im.entry_off + e);
          if (a.flag && !a.flag[tg]) valid = false;
        }
        const unsigned m = __ballot_sync(0xffffffffu, valid);
        const int need = NC - have;
        const int rank = __popc(m & ((1u << lane) - 1u));
        const bool take = valid && rank < need;
        const unsigned tm = __ballot_sync(0xffffffffu, take);
        const int ntake = __popc(tm);
        if (ntake > 0) {
          if (have == 0) acquire(j);
          const int s = j % S;
          if (take) {
            const int sr = __ldg(a.e_src + im.entry_off + e);
            s_tgtoff[s][have + rank] = ((long long)tg * a.nrhs + r) * a.Ps;
            bulk_load(stages + ((size_t)s * NC + have + rank) * Pc, a.mult + ((size_t)sr * a.nrhs + r) * a.Ps, col_bytes,
                      &full[s]);
          }
          have += ntake;
        }
        base += ((m & ~tm) == 0u) ? 32 : (32 - __clz(tm));
        if (have == NC) {
          commit(it, NC);
          have = 0;
        }
      }
      if (have > 0) {  // operators change with the item: close the partial stage
        commit(it, have);
        have = 0;
      }
    }
    // end of stream marker, then drain the stages still holding results
    acquire(j);
    commit(-1, 0);
    for (int jj = max(j, S); jj <= j - 2 + S; ++jj) acquire(jj);  // real stages j - 1 - S .. j - 2
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    return;
  }

  // =================================================================== MMA warps
  const int KS = a.KS, MTU = a.MTU;
  const int kb = (KS * warp) / NW, ke = (KS * (warp + 1)) / NW, kcnt = ke - kb;
  const int mcnt = MTU > warp ? (MTU - warp + NW - 1) / NW : 0;
  const int ar = lane >> 2, ak = lane & 3;
  double A1[kStreamMaxMt][KSW];      // Vt_t fragments of this warp's k-slice
  double A2[MTW][2 * kStreamMaxMt];  // U_t fragments of this warp's row tiles
  int item_g1 = -1, item_g2 = -1, mt1 = 0, mt2 = 0;
  auto load_a1 = [&](const M2LItemDev &im) {
    mt1 = im.mt;
    const double *vf = a.pool + im.v_off + lane;
#pragma unroll
    for (int m = 0; m < kStreamMaxMt; ++m)
#pragma unroll
      for (int q = 0; q < KSW; ++q)
        A1[m][q] = (m < im.mt && q < kcnt) ? __ldg(vf + ((size_t)m * KS + kb + q) * 32) : 0.0;
  };
  auto load_a2 = [&](const M2LItemDev &im) {
    mt2 = im.mt;
    const int KR = 2 * im.mt;
    const double *uf = a.pool + im.u_off + lane;
#pragma unroll
    for (int t = 0; t < MTW; ++t)
#pragma unroll
      for (int ks = 0; ks < 2 * kStreamMaxMt; ++ks)
        A2[t][ks] = (t < mcnt && ks < KR) ? __ldg(uf + ((size_t)(warp + NW * t) * KR + ks) * 32) : 0.0;
  };
  // first contraction of stage jj: partial Y over this warp's k-slice, parked in the rows of the stage it alone reads.
  // The bodies are specialised on the rank tiles MT of the piece and run all KSW k-steps / MTW row tiles (slices one
  // step short multiply zero fragments): a predicate around mma.sync costs a WARPSYNC + ISETP per pair of DMMAs, and
  // the instruction stream next to the DMMAs is what keeps the FP64 pipe from saturating (profiles/r2_m2l_*).
  auto gemm1 = [&](int jj, auto mt_c) {
    constexpr int MT = decltype(mt_c)::value;
    double *st = stages + (size_t)(jj % S) * NC * Pc;
    double y[MT][2][2];
#pragma unroll
    for (int m = 0; m < MT; ++m) y[m][0][0] = y[m][0][1] = y[m][1][0] = y[m][1][1] = 0.0;
    const double *bp = st + (size_t)ar * Pc + kb * 4 + ak;
#pragma unroll
    for (int q = 0; q < KSW; ++q) {
      // a slice one step short re-reads its last step (times a zero fragment) instead of the neighbour's first one, which
      // that warp may already be overwriting with its partial sums (harmless for the product, but a genuine WAR race)
      const int qq = q < kcnt ? q : kcnt - 1;
      const double b0 = bp[qq * 4], b1 = bp[(size_t)8 * Pc + qq * 4];
#pragma unroll
      for (int m = 0; m < MT; ++m) {
        dmma(y[m][0][0], y[m][0][1], A1[m][q], b0);
        dmma(y[m][1][0], y[m][1][1], A1[m][q], b1);
      }
    }
    __syncwarp();  // every lane is done reading the slice before it is overwritten
    double *pp = st + kb * 4;
#pragma unroll
    for (int m = 0; m < MT; ++m)
#pragma unroll
      for (int n = 0; n < 2; ++n)
#pragma unroll
        for (int h = 0; h < 2; ++h) pp[(size_t)(n * 8 + ak * 2 + h) * Pc + m * 8 + ar] = y[m][n][h];
  };
  // Y = sum of the NW partial products, in a fixed order
  auto reduce_y = [&](int jj, int mt) {
    const double *st = stages + (size_t)(jj % S) * NC * Pc;
    double *Y = Yb + (size_t)(jj & 1) * 24 * YS;
    const int rows = mt * 8, nel = rows * NC;
    for (int id = tid; id < nel; id += NW * 32) {
      const int rk = id % rows, c = id / rows;
      double v[NW];
#pragma unroll
      for (int w = 0; w < NW; ++w) v[w] = st[(size_t)c * Pc + ((KS * w) / NW) * 4 + rk];
#pragma unroll
      for (int span = 1; span < NW; span *= 2)  // pairwise: a fixed order, log2(NW) dependent additions
#pragma unroll
        for (int w = 0; w + span < NW; w += 2 * span) v[w] += v[w + span];
      Y[rk * YS + c] = v[0];
    }
  };
  // second contraction of stage jj: Z = U_t Y into the stage, then hand it to the producer
  auto gemm2 = [&](int jj, auto mt_c) {
    constexpr int MT = decltype(mt_c)::value;
    double *st = stages + (size_t)(jj % S) * NC * Pc;
    const double *Y = Yb + (size_t)(jj & 1) * 24 * YS;
    double z[MTW][2][2];
#pragma unroll
    for (int t = 0; t < MTW; ++t) z[t][0][0] = z[t][0][1] = z[t][1][0] = z[t][1][1] = 0.0;
#pragma unroll
    for (int ks = 0; ks < 2 * MT; ++ks) {
      const double b0 = Y[(ks * 4 + ak) * YS + ar], b1 = Y[(ks * 4 + ak) * YS + 8 + ar];
#pragma unroll
      for (int t = 0; t < MTW; ++t) {
        dmma(z[t][0][0], z[t][0][1], A2[t][ks], b0);
        dmma(z[t][1][0], z[t][1][1], A2[t][ks], b1);
      }
    }
#pragma unroll
    for (int t = 0; t < MTW; ++t)
      if (t < mcnt) {
        const int row = (warp + NW * t) * 8 + ar;
#pragma unroll
        for (int n = 0; n < 2; ++n)
#pragma unroll
          for (int h = 0; h < 2; ++h) st[(size_t)(n * 8 + ak * 2 + h) * Pc + row] = z[t][n][h];
      }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the TMA engine
    __syncwarp();
    if (lane == 0) mbar_arrive(&zfull[jj % S]);
  };
  // software pipeline: iteration i runs the first contraction of stage i + 1, the second of stage i and the partial-sum
  // reduction of stage i + 1.  The MMA warps meet only through mbarriers they arrive on early and wait on late
  // (pbar: partial sums of a stage complete; ybar: Y of a stage complete), so a warp that finishes its k-slice first
  // goes straight on to its row tiles of the previous stage instead of idling at a CTA barrier.
  auto run1 = [&](int jj) {
    if (mt1 == 3) gemm1(jj, std::integral_constant<int, 3>());
    else if (mt1 == 2) gemm1(jj, std::integral_constant<int, 2>());
    else gemm1(jj, std::integral_constant<int, 1>());
  };
  auto run2 = [&](int jj) {
    if (mt2 == 3) gemm2(jj, std::integral_constant<int, 3>());
    else if (mt2 == 2) gemm2(jj, std::integral_constant<int, 2>());
    else gemm2(jj, std::integral_constant<int, 1>());
  };
  auto warp_arrive = [&](unsigned long long *b) {
    __syncwarp();
    if (lane == 0) mbar_arrive(b);
  };
  mbar_wait(&full[0], 0);
  int cur = s_item[0];
  if (cur < 0) return;
  {
    const M2LItemDev im = a.items[cur];
    load_a1(im);
    item_g1 = cur;
  }
  run1(0);
  warp_arrive(&pbar[0]);
  mbar_wait(&pbar[0], 0);
  reduce_y(0, mt1);
  warp_arrive(&ybar[0]);
  for (int i = 0;; ++i) {
    const int jn = i + 1;
    mbar_wait(&full[jn % S], (unsigned)((jn / S) & 1));
    const int nxt = s_item[jn % S];
    if (nxt >= 0) {
      if (nxt != item_g1) {
        const M2LItemDev im = a.items[nxt];
        load_a1(im);
        item_g1 = nxt;
      }
      run1(jn);
      warp_arrive(&pbar[jn & 1]);
    }
    if (cur != item_g2) {
      const M2LItemDev im = a.items[cur];
      load_a2(im);
      item_g2 = cur;
    }
    mbar_wait(&ybar[i & 1], (unsigned)((i >> 1) & 1));
    run2(i);
    if (nxt < 0) break;
    mbar_wait(&pbar[jn & 1], (unsigned)((jn >> 1) & 1));
    reduce_y(jn, mt1);
    warp_arrive(&ybar[jn & 1]);
    cur = nxt;
  }
}

// ---- host side ------------------------------------------------------------------------------------------------
// work items of one launch for one (nrhs, target restriction)
struct M2LItemTable {
  DBuf<unsigned char> d_items;
  int n_items = 0, n_ctas = 0, nrhs = -1;
};

struct M2LStreamPlan {
  struct Group {
    int level, tix;
    long long entry_off;
    int n_entries;
    std::vector<int> pieces;  // indices into `pieces`
  };
  struct Piece {
    long long v_off, u_off;
    int mt;
  };
  std::vector<Group> groups;
  std::vector<Piece> pieces;
  std::vector<int> h_tgt;  // target cell of every entry (ascending inside a group): per-rank subranges are cut from it
  DBuf<int> d_tgt, d_src;
  DBuf<double> d_pool;
  DBuf<int> d_counter;
  M2LItemTable all;  // every entry
  int P = 0, Ps = 0, Pc = 0, KS = 0, MTU = 0, nw = 0;
  size_t smem = 0;
};

// MMA warps for order P, 0 = not served: the partial sums of a warp's k-slice (24 rows) must fit inside the slice
// (floor(KS / NW) >= 6) and the slices must fit the register file (ceil(KS / NW) <= 8, ceil(MTU / NW) <= 4)
static int m2l_stream_warps(int P) {
  const int KS = (P + 3) / 4, MTU = (P + 7) / 8;
  for (int nw : {8, 11})
    if (KS / nw >= 2 * kStreamMaxMt && (KS + nw - 1) / nw <= kStreamKsw && (MTU + nw - 1) / nw <= kStreamMtw) return nw;
  return 0;
}

// the dispatch rule alone (no environment override): uncompressed operators are never streamed
int m2l_stream_warps(int P, int compression) {
  if (compression == FB_COMPRESSION_NONE || P < 1) return 0;
  return m2l_stream_warps(P);
}

bool m2l_stream_supported(int P, int compression) {
  if (const char *v = std::getenv("FB_M2L_STREAM"))
    if (v[0] == '0') return false;
  return m2l_stream_warps(P, compression) != 0;
}

int m2l_stream_plan_warps(const M2LStreamPlan *p) { return p ? p->nw : 0; }

void m2l_stream_free(M2LStreamPlan *p) { delete p; }

// entries: (target cell, source cell, level, transfer index) of every V-list pair
M2LStreamPlan *m2l_stream_build(const HostTree &ht, const Operators &ops, int P, const int *d_inv_tab,
                                cudaStream_t stream) {
  auto *plan = new M2LStreamPlan();
  std::unique_ptr<M2LStreamPlan, void (*)(M2LStreamPlan *)> guard(plan, m2l_stream_free);
  const int dim = ht.dim;
  plan->P = P;
  plan->Ps = coef_stride(P);
  plan->KS = (P + 3) / 4;
  plan->MTU = (P + 7) / 8;
  plan->Pc = std::max(plan->Ps, plan->MTU * 8);
  while (plan->Pc % 16 != 4 && plan->Pc % 16 != 12) plan->Pc += 2;  // conflict-free B fragments, 16-byte columns
  plan->nw = m2l_stream_warps(P);
  plan->smem = sizeof(double) * ((size_t)kStreamStages * kStreamCols * plan->Pc + 2 * 24 * (kStreamCols + 4));
  // entries grouped by (level, transfer vector), targets ascending inside a group
  std::vector<int> e_tgt, e_src;
  std::vector<M2LPieceDev> hp;
  std::vector<double> dense;
  std::map<std::pair<int, int>, std::pair<long long, long long>> dense_off;  // (level, ref) -> (U, Vt)
  long long pool_size = 0;
  const int n_vec = (int)ops.ref_lookup.size();
  // transfer index of every V-list entry (calculate_m2l_transfer_index, bbfmm.rs:989-998), all cells at once
  const size_t ncell = ht.ncells();
  std::vector<uint32_t> anchors(3 * ncell);
#pragma omp parallel for schedule(static)
  for (long long c = 0; c < (long long)ncell; ++c) ht.anchor((int)c, &anchors[3 * (size_t)c]);
  const long long n_v = ht.v_ptr[ncell];
  std::vector<int> tix_of(n_v > 0 ? (size_t)n_v : 1);
#pragma omp parallel for schedule(dynamic, 256)
  for (long long c = 0; c < (long long)ncell; ++c) {
    const uint32_t *ac = &anchors[3 * (size_t)c];
    for (long long e = ht.v_ptr[c]; e < ht.v_ptr[c + 1]; ++e) {
      const uint32_t *as = &anchors[3 * (size_t)ht.v_idx[e]];
      int tix = 0;
      for (int d = 0; d < dim; ++d) tix = tix * 7 + ((int)ac[d] - (int)as[d] + 3);
      tix_of[e] = tix;
    }
  }
  for (int lvl = 2; lvl <= ht.depth; ++lvl) {
    // counting sort of the level's entries by transfer index; cells are visited in ascending order, so the targets of a
    // group come out ascending
    std::vector<long long> start(n_vec + 1, 0);
    for (int c = ht.level_ptr[lvl]; c < ht.level_ptr[lvl + 1]; ++c)
      for (long long e = ht.v_ptr[c]; e < ht.v_ptr[c + 1]; ++e) ++start[tix_of[e] + 1];
    for (int t = 0; t < n_vec; ++t) start[t + 1] += start[t];
    std::vector<std::array<int, 2>> sorted((size_t)start[n_vec]);
    {
      std::vector<long long> fill(start.begin(), start.end() - 1);
      for (int c = ht.level_ptr[lvl]; c < ht.level_ptr[lvl + 1]; ++c)
        for (long long e = ht.v_ptr[c]; e < ht.v_ptr[c + 1]; ++e) sorted[(size_t)fill[tix_of[e]]++] = {c, ht.v_idx[e]};
    }
    struct Span {
      const std::array<int, 2> *b, *e;
      bool empty() const { return b == e; }
      size_t size() const { return (size_t)(e - b); }
      const std::array<int, 2> *begin() const { return b; }
      const std::array<int, 2> *end() const { return e; }
    };
    std::vector<Span> per_t(n_vec);
    for (int t = 0; t < n_vec; ++t) per_t[t] = {sorted.data() + start[t], sorted.data() + start[t + 1]};
    for (int tix = 0; tix < n_vec; ++tix) {
      if (per_t[tix].empty()) continue;
      const int ref = ops.ref_lookup[tix];
      const M2LOperator &op = ops.m2l[lvl - 2][ref];
      auto key = std::make_pair(lvl, ref);
      if (!dense_off.count(key)) {
        const long long uo = (long long)dense.size();
        dense.insert(dense.end(), op.U.a.begin(), op.U.a.end());
        const long long vo = (long long)dense.size();
        dense.insert(dense.end(), op.Vt.a.begin(), op.Vt.a.end());
        dense_off[key] = {uo, vo};
      }
      M2LStreamPlan::Group g;
      g.level = lvl;
      g.tix = tix;
      g.entry_off = (long long)e_tgt.size();
      g.n_entries = (int)per_t[tix].size();
      for (auto &t : per_t[tix]) {
        e_tgt.push_back(t[0]);
        e_src.push_back(t[1]);
      }
      const int cap = 8 * kStreamMaxMt;
      for (int r0 = 0; r0 < std::max(op.rank, 1); r0 += cap) {
        const int r1 = std::min(op.rank, r0 + cap);
        M2LPieceDev pd;
        pd.dense_u = dense_off[key].first;
        pd.dense_vt = dense_off[key].second;
        pd.rank = op.rank;
        pd.r0 = r0;
        pd.r1 = r1;
        pd.perm = ops.perm_lookup[tix];
        pd.mt = std::max(1, (r1 - r0 + 7) / 8);
        pd.v_off = pool_size;
        pool_size += (long long)pd.mt * plan->KS * 32;
        pd.u_off = pool_size;
        pool_size += (long long)plan->MTU * 2 * pd.mt * 32;
        g.pieces.push_back((int)plan->pieces.size());
        plan->pieces.push_back({pd.v_off, pd.u_off, pd.mt});
        hp.push_back(pd);
      }
      plan->groups.push_back(std::move(g));
    }
  }
  if (plan->groups.empty()) return nullptr;
  plan->d_tgt.upload(e_tgt, stream);
  plan->h_tgt = e_tgt;
  plan->d_src.upload(e_src, stream);
  plan->d_pool.reserve((size_t)pool_size);
  DBuf<double> d_dense;
  d_dense.upload(dense, stream);
  DBuf<unsigned char> d_pieces;
  d_pieces.reserve(hp.size() * sizeof(M2LPieceDev));
  FB_CUDA(cudaMemcpyAsync(d_pieces.p, hp.data(), hp.size() * sizeof(M2LPieceDev), cudaMemcpyHostToDevice, stream));
  FB_LAUNCH(k_m2l_expand, (unsigned)hp.size(), 256, 0, stream, reinterpret_cast<const M2LPieceDev *>(d_pieces.p),
            d_dense.p, d_inv_tab, P, plan->KS, plan->MTU, plan->d_pool.p);
  FB_CUDA(cudaStreamSynchronize(stream));  // d_dense / d_pieces / hp go out of scope
  guard.release();
  return plan;
}

// work items of one launch: (piece, entry range), pulled by one persistent CTA per SM, longest first
// level_lo / level_hi (per level, or null): only entries whose target cell id lies in [lo, hi) of its level — the cells
// with targets of a Morton-contiguous leaf range form one such range per level, so a rank's share is a subrange of
// every group and needs no per-entry flag test
static void m2l_stream_items(M2LStreamPlan &pl, M2LItemTable &tab, int nrhs, int sms, const int *level_lo,
                             const int *level_hi, cudaStream_t stream) {
  struct Item {
    M2LItemDev d;
    double cost;
  };
  struct Span {
    int e0, e1;
  };
  std::vector<Span> spans(pl.groups.size());
  double total = 0;
  for (size_t gi = 0; gi < pl.groups.size(); ++gi) {
    const auto &g = pl.groups[gi];
    int e0 = 0, e1 = g.n_entries;
    if (level_lo) {
      const int *b = pl.h_tgt.data() + g.entry_off, *e = b + g.n_entries;
      e0 = (int)(std::lower_bound(b, e, level_lo[g.level]) - b);
      e1 = (int)(std::lower_bound(b, e, level_hi[g.level]) - b);
      e1 = std::max(e1, e0);  // a level without owned cells has lo > hi
    }
    spans[gi] = {e0, e1};
    for (int pi : g.pieces) total += (double)(e1 - e0) * nrhs * pl.pieces[pi].mt;
  }
  std::vector<Item> items;
  // an item should be long enough to amortise the operator load (~50 fragment loads per thread) and short enough to
  // balance the tail: at most 1/6 of a CTA's share
  const double max_cost = std::max(total / (6.0 * sms), 3.0 * 64.0);
  for (size_t gi = 0; gi < pl.groups.size(); ++gi) {
    const auto &g = pl.groups[gi];
    for (int pi : g.pieces) {
      const auto &pc = pl.pieces[pi];
      const double per_entry = (double)nrhs * pc.mt;
      const int chunk = std::max(1, (int)(max_cost / per_entry));
      for (int e0 = spans[gi].e0; e0 < spans[gi].e1; e0 += chunk) {
        const int ne = std::min(chunk, spans[gi].e1 - e0);
        Item it;
        it.d.entry_off = g.entry_off + e0;
        it.d.n_entries = ne;
        it.d.mt = pc.mt;
        it.d.v_off = pc.v_off;
        it.d.u_off = pc.u_off;
        it.cost = ne * per_entry + 48.0;  // + the operator load
        items.push_back(it);
      }
    }
  }
  // longest first: the CTAs pull items from a counter as they finish
  std::stable_sort(items.begin(), items.end(), [](const Item &x, const Item &y) { return x.cost > y.cost; });
  std::vector<M2LItemDev> flat;
  for (auto &it : items) flat.push_back(it.d);
  tab.n_items = (int)flat.size();
  tab.n_ctas = std::max(1, std::min<int>(sms, tab.n_items));
  tab.d_items.reserve(flat.size() * sizeof(M2LItemDev));
  FB_CUDA(cudaMemcpyAsync(tab.d_items.p, flat.data(), flat.size() * sizeof(M2LItemDev), cudaMemcpyHostToDevice, stream));
  pl.d_counter.reserve(1);
  FB_CUDA(cudaStreamSynchronize(stream));
  tab.nrhs = nrhs;
}

static int device_sms() {
  int dev = 0, sms = 148;
  FB_CUDA(cudaGetDevice(&dev));
  FB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  return sms;
}

M2LItemTable *m2l_stream_table_new(M2LStreamPlan *plan, int nrhs, const int *level_lo, const int *level_hi,
                                   cudaStream_t stream) {
  auto *t = new M2LItemTable();
  try {
    m2l_stream_items(*plan, *t, nrhs, device_sms(), level_lo, level_hi, stream);
  } catch (...) {
    delete t;
    throw;
  }
  return t;
}
int m2l_stream_table_nrhs(const M2LItemTable *t) { return t->nrhs; }
void m2l_stream_table_free(M2LItemTable *t) { delete t; }

void m2l_stream_launch(M2LStreamPlan *plan, int nrhs, const uint8_t *flag_or_null, const M2LItemTable *table_or_null,
                       const double *mult, double *loc, cudaStream_t stream) {
  M2LStreamPlan &pl = *plan;
  const M2LItemTable *tp = table_or_null;
  if (!tp) {
    if (pl.all.nrhs != nrhs) m2l_stream_items(pl, pl.all, nrhs, device_sms(), nullptr, nullptr, stream);
    tp = &pl.all;
  }
  FB_REQUIRE(tp->nrhs == nrhs, "M2L item table built for another number of right-hand sides");
  if (tp->n_items == 0) return;
  const M2LItemTable &tb = *tp;
  M2LStreamArgs a{};
  a.items = reinterpret_cast<const M2LItemDev *>(tb.d_items.p);
  a.n_items = tb.n_items;
  a.next_item = pl.d_counter.p;
  FB_CUDA(cudaMemsetAsync(pl.d_counter.p, 0, sizeof(int), stream));
  a.e_tgt = pl.d_tgt.p;
  a.e_src = pl.d_src.p;
  a.pool = pl.d_pool.p;
  a.flag = table_or_null ? nullptr : flag_or_null;  // a restricted table is already exact
  a.mult = mult;
  a.loc = loc;
  a.P = pl.P;
  a.Ps = pl.Ps;
  a.Pc = pl.Pc;
  a.KS = pl.KS;
  a.MTU = pl.MTU;
  a.nrhs = nrhs;
#define FB_STREAM_LAUNCH(NWV)                                                                                     \
  do {                                                                                                            \
    FB_CUDA(cudaFuncSetAttribute(k_m2l_stream<NWV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));  \
    FB_LAUNCH((k_m2l_stream<NWV>), tb.n_ctas, ((NWV) + 1) * 32, pl.smem, stream, a);                              \
  } while (0)
  if (pl.nw == 8)
    FB_STREAM_LAUNCH(8);
  else
    FB_STREAM_LAUNCH(11);
#undef FB_STREAM_LAUNCH
}

}  // namespace fb
