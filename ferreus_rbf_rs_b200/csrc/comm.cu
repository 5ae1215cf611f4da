// Multi-GPU BBFMM matvec: one process per GPU, the tree partitioned by Morton-contiguous leaf ranges (SURVEY.md §8e),
// NCCL over NVLink for the two exchange steps.  The reference is single-process rayon (bbfmm.rs:669, 682, 788, 841,
// 1122 are its parallel loops); this file is what replaces "one rayon pool" when the tree spans several B200s.
//
//   ownership   leaves in Morton order, cut into `world` contiguous ranges of nearly equal estimated work; a rank owns
//               the points of its range.  Tree topology and point coordinates are replicated (24 B per point), the
//               work is not: every kernel evaluation of the unpartitioned matvec is made by exactly one rank.
//   upward      P2M over the OWNED leaves only, M2M over the cells that have owned descendants: every rank holds the
//               exact multipoles of the cells inside its range and a partial sum for the cells that span ranks;
//   exchange 1  ncclAllReduce(sum) of the multipole array completes the spanning cells and hands every rank the halo
//               multipoles its V / W lists need; the exchange and the downward pass run on the high-priority main
//               stream, the near-field pass (it needs no multipoles) beside them on a low-priority one;
//   near field  symmetric P2P (p2p_sym.cu) for the chunks of the owned range against ALL sources behind them: the
//               source-side sums of rows another rank owns are added into this rank's copy of the full-length result;
//   downward    M2L / L2L / L2P for the cells / targets of the share; the fused W/X kernel (p2l.cu) for the cells with
//               owned targets — its M2P half, applied by the owner of the cell's first point, also reaches foreign rows;
//   exchange 2  ncclAllReduce(sum) of the full-length result (8 N nrhs bytes): owned rows + the symmetric halves other
//               ranks computed for them = the full A w, replicated, in the caller's row order — the next Krylov vector
//               needs exactly that.
// NCCL is loaded at run time (dlopen of the copy already in the process, else libnccl.so.2): the single-GPU drop-in
// has no link-time dependency on it.
#include <dlfcn.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <numeric>

#include <nccl.h>

#include "fmm.h"

namespace fb {

// ---- NCCL entry points, resolved once ------------------------------------------------------------------------------
struct NcclApi {
  void *handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
};

static NcclApi &nccl() {
  static NcclApi api = [] {
    NcclApi a;
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    // the copy already mapped into this process (torch ships its own) wins: two NCCLs in one process is asking for it
    for (const char *nm : names)
      if (!a.handle) a.handle = dlopen(nm, RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);
    if (const char *p = std::getenv("FB_NCCL_LIB"))
      if (!a.handle) a.handle = dlopen(p, RTLD_NOW | RTLD_GLOBAL);
    for (const char *nm : names)
      if (!a.handle) a.handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
    if (!a.handle) return a;
#define FB_SYM(field, name) a.field = reinterpret_cast<decltype(a.field)>(dlsym(a.handle, name))
    FB_SYM(GetUniqueId, "ncclGetUniqueId");
    FB_SYM(CommInitRank, "ncclCommInitRank");
    FB_SYM(CommDestroy, "ncclCommDestroy");
    FB_SYM(AllReduce, "ncclAllReduce");
    FB_SYM(AllGather, "ncclAllGather");
    FB_SYM(GetErrorString, "ncclGetErrorString");
#undef FB_SYM
    return a;
  }();
  return api;
}

static void require_nccl() {
  NcclApi &a = nccl();
  if (!a.handle || !a.GetUniqueId || !a.CommInitRank || !a.AllReduce || !a.AllGather)
    throw Error(FB_ERR_CUDA, "NCCL (libnccl.so.2) could not be loaded; set FB_NCCL_LIB to its path");
}

#define FB_NCCL(expr)                                                                                        \
  do {                                                                                                       \
    ncclResult_t r_ = (expr);                                                                                \
    if (r_ != ncclSuccess)                                                                                   \
      throw fb::Error(FB_ERR_CUDA, std::string(#expr) + ": " +                                               \
                                       (fb::nccl().GetErrorString ? fb::nccl().GetErrorString(r_) : "NCCL error")); \
  } while (0)

// contiguous ranges of nearly equal work: boundaries into the leaf sequence (the same cut sharding.py makes)
void partition_by_work(const double *work, size_t n, int parts, uint64_t *bounds) {
  bounds[0] = 0;
  bounds[parts] = n;
  if (parts <= 1) return;
  if (n == 0) {
    for (int k = 1; k < parts; ++k) bounds[k] = 0;
    return;
  }
  std::vector<double> csum(n);
  double run = 0;
  for (size_t i = 0; i < n; ++i) csum[i] = (run += work[i]);
  const double total = csum[n - 1];
  for (int k = 1; k < parts; ++k) {
    const double target = total * (double)k / (double)parts;
    const size_t cut = (size_t)(std::lower_bound(csum.begin(), csum.end(), target) - csum.begin()) + 1;
    bounds[k] = std::max<uint64_t>(std::min(cut, n), bounds[k - 1]);
  }
}

__global__ void k_iota_u64(const uint32_t *perm, size_t begin, size_t count, unsigned long long *out) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i < count) out[i] = perm[begin + i];
}

}  // namespace fb

using namespace fb;

struct fb_comm {
  ncclComm_t comm = nullptr;
  int rank = 0, world = 1, device = 0;
  cudaStream_t stream = nullptr;  // collectives that run under compute
  cudaEvent_t ev_ready = nullptr, ev_done = nullptr;
  ~fb_comm() {
    if (comm && nccl().CommDestroy) nccl().CommDestroy(comm);
    if (ev_ready) cudaEventDestroy(ev_ready);
    if (ev_done) cudaEventDestroy(ev_done);
    if (stream) cudaStreamDestroy(stream);
  }
};

// per-tree state of the partition (fb_tree::shard)
struct fb_shard {
  fb_comm *comm = nullptr;
  int fork_mode = 0;                  // where the near field forks off the main stream: chosen in fb_tree_shard
  bool full_upward = false;           // emulated share with every multipole formed locally: the owned rows come out exact
  int rank = 0, world = 1;            // the share this process computes: the communicator's, or an emulated one (fb_tree_shard_as)
  std::vector<uint64_t> leaf_bounds;  // world + 1 boundaries into the Morton leaf sequence
  std::vector<int> pos;               // world + 1 boundaries into the sorted point order
  DBuf<int> d_owned_leaves;           // cells of the owned leaves that hold sources (P2M grid)
  int n_owned_leaves = 0;
  TargetBuffers tb;
  TargetSet ts{};
  DBuf<unsigned long long> d_rows;
  std::vector<int> level_lo, level_hi;  // per level: the cells with owned targets are the ids [lo, hi)
  M2LItemTable *m2l_table = nullptr;    // M2L work items of that share
  double last_ms[4] = {0, 0, 0, 0};   // upward pass + multipole all-reduce, downward pass, (rest of the near field +) L2P, result all-reduce
  cudaEvent_t ev[5] = {};
  ~fb_shard() {
    for (auto &e : ev)
      if (e) cudaEventDestroy(e);
    if (m2l_table) m2l_stream_table_free(m2l_table);
  }
};

void fb_shard_free(fb_shard *s) { delete s; }

extern "C" {

int fb_partition_by_work(const double *work, size_t n_leaves, int parts, uint64_t *bounds_out) {
  if (!work || !bounds_out || parts < 1) return FB_ERR_INVALID_ARGUMENT;
  partition_by_work(work, n_leaves, parts, bounds_out);
  return FB_OK;
}

int fb_comm_unique_id(uint8_t *id_out128) {
  return guarded([&] {
    FB_REQUIRE(id_out128, "null argument");
    require_nccl();
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    FB_NCCL(nccl().GetUniqueId(&id));
    std::memcpy(id_out128, &id, sizeof(id));
  });
}

int fb_comm_init(const uint8_t *id128, int rank, int world_size, fb_comm **out) {
  if (!out) return FB_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  fb_comm *c = nullptr;
  const int rc = guarded([&] {
    FB_REQUIRE(id128 && world_size >= 1 && rank >= 0 && rank < world_size, "fb_comm_init: bad rank / world size");
    require_nccl();
    c = new fb_comm();
    c->rank = rank;
    c->world = world_size;
    FB_CUDA(cudaGetDevice(&c->device));
    ncclUniqueId id;
    std::memcpy(&id, id128, sizeof(id));
    FB_NCCL(nccl().CommInitRank(&c->comm, world_size, id, rank));
    // highest priority: the collective's CTAs must become resident while the near-field kernel it runs under is still
    // feeding the SMs, not after that kernel's last wave (a default-priority stream measured exactly that: 0.68 ms for
    // 0.48 ms of P2P at 8 ranks)
    int prio_lo = 0, prio_hi = 0;
    FB_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    FB_CUDA(cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, prio_hi));
    FB_CUDA(cudaEventCreateWithFlags(&c->ev_ready, cudaEventDisableTiming));
    FB_CUDA(cudaEventCreateWithFlags(&c->ev_done, cudaEventDisableTiming));
  });
  if (rc != FB_OK) {
    delete c;
    return rc;
  }
  *out = c;
  return FB_OK;
}

void fb_comm_free(fb_comm *c) {
  if (!c) return;
  cudaSetDevice(c->device);
  delete c;
}

int fb_comm_rank(const fb_comm *c) { return c ? c->rank : -1; }
int fb_comm_world_size(const fb_comm *c) { return c ? c->world : -1; }

// Estimated work of every leaf under the ownership rules above, in units of one direct-sum kernel evaluation
// (calibrated on the 1M-point headline workload: symmetric P2P 1.16 ps, W/X 0.74 ps per evaluation, M2L 1.75 ns per entry
// at P = 343): the P2P evaluations of a leaf are the pairs with the sources BEHIND it (one RHS: p2p_sym.cu) or all its
// ordered pairs; a cell's X-list work and M2L entries are pushed down to its leaves.
constexpr double kShortNearMs = 0.45;  // estimated near-field time of a rank below which it forks after the upward pass

static double share_work(const fb_tree &t, int world, uint64_t *leaf_ptr, double *work) {
  const HostTree &ht = t.ht;
  const size_t nl = ht.leaves.size(), nc = ht.ncells();
  const bool sym = t.nrhs == 1;
  std::vector<double> down(nc, 0.0);
  for (size_t c = 1; c < nc; ++c) {
    double nx = 0;
    for (long long e = ht.x_ptr[c]; e < ht.x_ptr[c + 1]; ++e) nx += ht.pt_end[ht.x_idx[e]] - ht.pt_begin[ht.x_idx[e]];
    down[c] += nx * t.P + (double)(ht.v_ptr[c + 1] - ht.v_ptr[c]) * 7.0 * t.P;
    const int nch = ht.child_ptr[c + 1] - ht.child_ptr[c];
    for (int k = ht.child_ptr[c]; k < ht.child_ptr[c + 1]; ++k) down[ht.child_idx[k]] += down[c] / nch;
  }
  std::vector<double> near(nl, 0.0);
  double near_total = 0.0;
  for (size_t l = 0; l < nl; ++l) {
    const int c = ht.leaves[l];
    leaf_ptr[l] = (uint64_t)ht.pt_begin[c];
    const double nt = ht.pt_end[c] - ht.pt_begin[c];
    double nsrc = 0;
    for (long long e = ht.u_ptr[c]; e < ht.u_ptr[c + 1]; ++e) {
      const int u = ht.u_idx[e];
      if (!sym || ht.pt_begin[u] >= ht.pt_begin[c]) nsrc += ht.pt_end[u] - ht.pt_begin[u];
    }
    near[l] = (sym ? 1.6 : 1.0) * nt * nsrc;
    near_total += near[l];
    // (the M2P evaluations of the leaf's W list ride on the X-list evaluations of those cells)
    work[l] = down[c] + 0.3 * nt * t.P + 1.0;
  }
  leaf_ptr[nl] = (uint64_t)t.n;
  // A SHORT near field (forked after the upward pass, see fb_tree_shard) runs beside exchange 1 and in the tails of the
  // downward kernels: about 0.35 ms of it per rank cost nothing on the critical path at 8 ranks on the headline workload,
  // and a cut that counted it in full left the ranks with few direct pairs waiting on the ones with many far-field
  // evaluations.  Only the part beyond that slack is weighed.  A long near field (forked before the upward pass) is
  // weighed in full: beside it the upward pass and the exchange stretch by about what it saves (measured at 2 / 4 ranks).
  const double unit_ms = 0.74e-9 * (1.0 + 0.15 * (t.nrhs - 1));  // one evaluation unit, B200, from the stage timings
  const double near_ms = near_total * unit_ms;
  const bool short_near = near_ms / world < kShortNearMs;
  const double alpha = short_near && near_ms > 0 ? std::min(1.0, std::max(0.25, 1.0 - 0.35 * world / near_ms)) : 1.0;
  for (size_t l = 0; l < nl; ++l) work[l] += alpha * near[l];
  return near_ms / world;  // estimated near-field time of a rank
}

// as_world > 0: take the share of rank `as_rank` of `as_world` ranks with a world-1 communicator — the per-rank kernel
// times of an N-GPU partition measured on one GPU (tools/shard_emulate.py); the collectives degenerate to copies, so
// the owned rows are exact only with `exact` != 0 (every multipole formed locally: the upward time is then the unpartitioned one)
static int shard_impl(fb_tree *t, fb_comm *comm, int as_rank, int as_world, int exact) {
  return guarded([&] {
    FB_REQUIRE(t, "null tree");
    FB_CUDA(cudaSetDevice(t->device));
    if (t->shard) {
      fb_shard_free(t->shard);
      t->shard = nullptr;
    }
    if (!comm) return;
    FB_REQUIRE(comm->device == t->device, "the communicator and the tree live on different devices");
    std::unique_ptr<fb_shard> sh(new fb_shard());
    sh->comm = comm;
    sh->rank = comm->rank;
    sh->world = comm->world;
    if (as_world > 0) {
      FB_REQUIRE(comm->world == 1 && as_rank >= 0 && as_rank < as_world, "emulated shares need a world-1 communicator");
      sh->rank = as_rank;
      sh->world = as_world;
      sh->full_upward = exact != 0;
    }
    const int world = sh->world, rank = sh->rank;
    const HostTree &ht = t->ht;
    const size_t nl = ht.leaves.size();
    std::vector<uint64_t> leaf_ptr(nl + 1);
    std::vector<double> work(nl);
    const double near_rank_ms = share_work(*t, world, leaf_ptr.data(), work.data());
    // Fork point of the near field (see fb_tree_matvec_sharded).  The downward kernels fill the register file (M2L: one
    // 384-thread CTA per SM, W/X: three CTAs per SM), so a P2P grid that is still running when they start only gets their
    // tails: a LONG near field is better off starting beside the upward pass (2 / 4 ranks on the headline workload: 5.42
    // / 2.78 ms against 5.56 / 2.91), a SHORT one after it, where it no longer stretches the latency-bound upward chain
    // and the exchange behind it (8 ranks: 1.65 against 1.73 ms).
    sh->fork_mode = near_rank_ms < kShortNearMs ? 1 : 0;
    if (const char *v = std::getenv("FB_SHARD_FORK")) sh->fork_mode = v[0] == '1' ? 1 : 0;
    sh->leaf_bounds.resize(world + 1);
    partition_by_work(work.data(), nl, world, sh->leaf_bounds.data());
    sh->pos.resize(world + 1);
    for (int r = 0; r <= world; ++r) sh->pos[r] = (int)leaf_ptr[sh->leaf_bounds[r]];
    std::vector<int> owned;
    for (uint64_t l = sh->leaf_bounds[rank]; l < sh->leaf_bounds[rank + 1]; ++l) {
      const int c = ht.leaves[l];
      if (ht.pt_end[c] > ht.pt_begin[c]) owned.push_back(c);
    }
    // ancestors of a contiguous leaf range are one contiguous id range per level
    sh->level_lo.assign(ht.depth + 1, INT32_MAX);
    sh->level_hi.assign(ht.depth + 1, 0);
    for (int c0 : owned)
      for (int c = c0; c >= 0; c = ht.parent[c]) {
        const int lv = ht.level[c];
        if (c >= sh->level_lo[lv] && c < sh->level_hi[lv]) break;  // the rest of the chain is already inside
        sh->level_lo[lv] = std::min(sh->level_lo[lv], c);
        sh->level_hi[lv] = std::max(sh->level_hi[lv], c + 1);
      }
    sh->n_owned_leaves = (int)owned.size();
    sh->d_owned_leaves.upload(owned, t->stream);
    // owned rows (Morton order) as the target subset: cell flags, leaf tiles, fused W/X row map
    const size_t p0 = (size_t)sh->pos[rank], cnt = (size_t)sh->pos[rank + 1] - p0;
    FB_REQUIRE(cnt > 0, "a rank owns no points: more ranks than leaves with work");
    sh->d_rows.reserve(cnt);
    FB_LAUNCH(k_iota_u64, (unsigned)((cnt + 255) / 256), 256, 0, t->stream, t->d_perm.p, p0, cnt, sh->d_rows.p);
    sh->ts = t->subset_target_set_dev(sh->d_rows.p, cnt, sh->tb);
    // the rows were listed in Morton order, so target i of the set is the source at sorted position p0 + i; the result
    // buffer of a partitioned matvec has a row for every source (foreign rows receive the symmetric halves), so the
    // set's row maps are the global ones
    const TargetSet all = t->source_target_set();
    sh->ts.own_lo = (int)p0;
    sh->ts.own_hi = (int)(p0 + cnt);
    sh->ts.out_row = all.out_row + p0;
    sh->ts.row_of_pos = all.row_of_pos;
    sh->ts.tgt_prefix = nullptr;
    for (auto &e : sh->ev) FB_CUDA(cudaEventCreate(&e));
    FB_CUDA(cudaStreamSynchronize(t->stream));
    t->shard = sh.release();
  });
}

int fb_tree_shard(fb_tree *t, fb_comm *comm) { return shard_impl(t, comm, 0, 0, 0); }
int fb_tree_shard_as(fb_tree *t, fb_comm *comm, int rank, int world, int exact) {
  return shard_impl(t, comm, rank, world, exact);
}

int fb_tree_shard_fork_mode(fb_tree *t, int mode) {
  if (!t || !t->shard || mode < 0 || mode > 1) return FB_ERR_INVALID_ARGUMENT;
  t->shard->fork_mode = mode;
  return FB_OK;
}

int fb_tree_shard_rows(const fb_tree *t, int rank, uint64_t *begin_pos, uint64_t *end_pos) {
  if (!t || !t->shard || rank < 0 || rank >= t->shard->world) return FB_ERR_INVALID_ARGUMENT;
  if (begin_pos) *begin_pos = (uint64_t)t->shard->pos[rank];
  if (end_pos) *end_pos = (uint64_t)t->shard->pos[rank + 1];
  return FB_OK;
}

// one partitioned matvec; weights (all N rows, replicated) were uploaded with fb_tree_upload_weights
int fb_tree_matvec_sharded(fb_tree *t) {
  return guarded([&] {
    FB_REQUIRE(t && t->shard, "fb_tree_shard must be called first");
    FB_CUDA(cudaSetDevice(t->device));
    FB_REQUIRE(t->d_w_user.cap >= t->n * (size_t)t->nrhs, "fb_tree_upload_weights must be called first");
    fb_shard &sh = *t->shard;
    fb_comm &cm = *sh.comm;
    cudaStream_t s = t->stream;
    const size_t nc = t->ht.ncells();
    const size_t out_count = t->n * (size_t)t->nrhs;
    FB_CUDA(cudaEventRecord(sh.ev[0], s));
    t->sort_weights();
    // The near-field pass needs the sorted weights and nothing else: it goes to the tree's LOW-priority side stream, the
    // upward pass (P2M, then one small M2M launch per level: latency-bound on a rank's share) and exchange 1 stay on the
    // high-priority main stream, so their CTAs are placed ahead of the P2P kernel's pending ones.  (Two streams of equal
    // priority measured 0.33 ms for the 0.08 ms M2M chain at 8 ranks: its launches queued behind the P2P grid.)
    const bool fuse = t->ht.adaptive && t->n_x_cells > 0;
    const size_t mult_count = nc * (size_t)t->nrhs * coef_stride(t->P);
    cudaStream_t s2 = t->stream2;
    // fork point of the near field: 0 = right after the weight sort (beside the upward pass too), 1 = after the upward
    // pass (beside exchange 1 and the downward pass only: the upward pass then has the SMs to itself); chosen by
    // fb_tree_shard from the estimated length of the near field (FB_SHARD_FORK / fb_tree_shard_fork_mode override it)
    if (sh.fork_mode == 1) {
      if (sh.full_upward) t->upward();
      else t->upward(sh.d_owned_leaves.p, sh.n_owned_leaves, sh.ts.cell_flag);
    }
    // this rank's copy of the full-length result: owned rows + the symmetric halves it computes for foreign rows.  Zeroed
    // on the main stream in front of the fork: both the near field (side stream) and the fused W/X pass (main stream) add
    // into it
    t->d_out.zero(out_count, s);
    FB_CUDA(cudaEventRecord(t->ev_fork, s));
    FB_CUDA(cudaStreamWaitEvent(s2, t->ev_fork, 0));
    if (t->timing) FB_CUDA(cudaEventRecord(t->ev[10], s2));
    t->launch_p2p(sh.ts, false, true, s2, true);  // U lists only; REDs: the fused W/X pass adds to the same rows
    if (t->timing) FB_CUDA(cudaEventRecord(t->ev[11], s2));
    FB_CUDA(cudaEventRecord(t->ev_join, s2));
    if (sh.fork_mode != 1) {
      if (sh.full_upward) t->upward();
      else t->upward(sh.d_owned_leaves.p, sh.n_owned_leaves, sh.ts.cell_flag);
    }
    if (cm.world > 1) {
      FB_NCCL(nccl().AllReduce(t->d_mult.p, t->d_mult.p, mult_count, ncclDouble, ncclSum, cm.comm, s));
      g_launches.fetch_add(1);
    }
    FB_CUDA(cudaEventRecord(sh.ev[1], s));
    if (t->m2l_plan && (!sh.m2l_table || m2l_stream_table_nrhs(sh.m2l_table) != t->nrhs)) {
      if (sh.m2l_table) m2l_stream_table_free(sh.m2l_table);
      sh.m2l_table = nullptr;
      sh.m2l_table = m2l_stream_table_new(t->m2l_plan, t->nrhs, sh.level_lo.data(), sh.level_hi.data(), s);
    }
    t->downward(sh.ts.cell_flag, fuse ? &sh.ts : nullptr, true, sh.m2l_table);
    FB_CUDA(cudaEventRecord(sh.ev[2], s));
    FB_CUDA(cudaStreamWaitEvent(s, t->ev_join, 0));  // the near field joins in front of L2P (plain read-modify-write)
    if (t->timing) FB_CUDA(cudaEventRecord(t->ev[7], s));
    t->launch_l2p(sh.ts, false);
    if (t->timing) FB_CUDA(cudaEventRecord(t->ev[8], s));
    if (!fuse && t->n_w_entries > 0) t->launch_p2p(sh.ts, false, false, s, false, true);  // W lists on their own
    FB_CUDA(cudaEventRecord(sh.ev[3], s));
    // exchange 2: partial full-length results -> A w on every rank
    if (cm.world > 1) {
      FB_NCCL(nccl().AllReduce(t->d_out.p, t->d_out.p, out_count, ncclDouble, ncclSum, cm.comm, s));
      g_launches.fetch_add(1);
    }
    FB_CUDA(cudaEventRecord(sh.ev[4], s));
    FB_CUDA(cudaStreamSynchronize(s));
    for (int k = 0; k < 4; ++k) {
      float ms = 0;
      FB_CUDA(cudaEventElapsedTime(&ms, sh.ev[k], sh.ev[k + 1]));
      sh.last_ms[k] = ms;
    }
    t->last_out_rows = t->n;
    if (t->timing) {  // per-kernel times of this rank's share, same slots as fb_tree_last_timing
      auto ms = [&](int a, int b) {
        float v = 0;
        cudaEventElapsedTime(&v, t->ev[a], t->ev[b]);
        return (double)v;
      };
      t->last_ms[0] = ms(0, 1);
      t->last_ms[1] = ms(1, 2);
      t->last_ms[2] = ms(3, 4);
      t->last_ms[3] = ms(4, 5);
      t->last_ms[4] = ms(5, 6);
      t->last_ms[5] = ms(7, 8);
      t->last_ms[6] = ms(10, 11);
      t->last_ms[7] = sh.last_ms[0] + sh.last_ms[1] + sh.last_ms[2] + sh.last_ms[3];
    }
  });
}

int fb_tree_sharded_timing(const fb_tree *t, double *ms_out4) {
  if (!t || !t->shard || !ms_out4) return FB_ERR_INVALID_ARGUMENT;
  for (int k = 0; k < 4; ++k) ms_out4[k] = t->shard->last_ms[k];
  return FB_OK;
}

int fb_tree_sharded_result_device(const fb_tree *t, const double **dev_ptr) {
  if (!t || !t->shard || !dev_ptr) return FB_ERR_INVALID_ARGUMENT;
  *dev_ptr = t->d_out.p;
  return FB_OK;
}

int fb_tree_sharded_download(fb_tree *t, double *out_vals) {
  return guarded([&] {
    FB_REQUIRE(t && t->shard && out_vals, "null argument");
    FB_CUDA(cudaSetDevice(t->device));
    FB_CUDA(cudaMemcpyAsync(out_vals, t->d_out.p, t->n * (size_t)t->nrhs * sizeof(double), cudaMemcpyDeviceToHost,
                            t->stream));
    FB_CUDA(cudaStreamSynchronize(t->stream));
  });
}

}  // extern "C"
