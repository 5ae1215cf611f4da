// fb_tree: device-resident BBFMM evaluator (build, upward, downward, leaf pass) and its C ABI.
#include "fmm.h"

#include <algorithm>
#include <array>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <thread>
#include <unordered_map>

#include <cub/cub.cuh>
#include <thrust/iterator/transform_iterator.h>

#include "fmm_kernels.cuh"

namespace fb {

std::atomic<uint64_t> g_launches{0};
static int initial_sqrt_mode() {
  const char *v = std::getenv("FB_SQRT");
  return (v && std::string(v) == "exact") ? 0 : 1;
}
std::atomic<int> g_sqrt_mode{initial_sqrt_mode()};
static thread_local std::string t_last_error;
void set_last_error(const std::string &msg) { t_last_error = msg; }

static inline unsigned nblocks(size_t n, int bs) { return (unsigned)((n + bs - 1) / bs); }

// ---- device memory cache (see common.h) ------------------------------------------------------------------------------
namespace {
struct DevCache {
  std::mutex mu;
  std::multimap<size_t, void *> free_blocks[16];            // per device: size -> block
  std::unordered_map<void *, std::pair<size_t, int>> live;  // block -> (size, device)
  size_t cached_bytes = 0;
};
DevCache &dev_cache() {
  static DevCache *c = new DevCache();  // never destroyed: blocks may be released during static destruction
  return *c;
}
size_t round_block(size_t bytes) {
  if (bytes <= (1u << 20)) return (bytes + 511) & ~(size_t)511;
  return (bytes + ((size_t)2 << 20) - 1) & ~(((size_t)2 << 20) - 1);
}
void trim_locked(DevCache &c) {
  for (auto &m : c.free_blocks) {
    for (auto &kv : m) cudaFree(kv.second);
    m.clear();
  }
  c.cached_bytes = 0;
}
}  // namespace

void *dev_alloc(size_t bytes) {
  DevCache &c = dev_cache();
  const size_t want = round_block(bytes);
  int dev = 0;
  FB_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(c.mu);
  auto &m = c.free_blocks[dev & 15];
  auto it = m.lower_bound(want);
  // reuse a cached block unless it would waste more than a quarter of itself
  if (it != m.end() && it->first - want <= it->first / 4) {
    void *p = it->second;
    c.cached_bytes -= it->first;
    c.live[p] = {it->first, dev};
    m.erase(it);
    return p;
  }
  void *p = nullptr;
  cudaError_t e = cudaMalloc(&p, want);
  if (e != cudaSuccess) {  // out of memory: give the cache back and try once more
    cudaGetLastError();
    trim_locked(c);
    e = cudaMalloc(&p, want);
  }
  if (e != cudaSuccess)
    throw Error(FB_ERR_CUDA, std::string("cudaMalloc of ") + std::to_string(want) + " bytes: " + cudaGetErrorString(e));
  c.live[p] = {want, dev};
  return p;
}

void dev_free(void *p) {
  if (!p) return;
  DevCache &c = dev_cache();
  cudaDeviceSynchronize();  // nothing queued may still touch the block (the semantics of the cudaFree this replaces)
  std::lock_guard<std::mutex> lock(c.mu);
  auto it = c.live.find(p);
  if (it == c.live.end()) {
    cudaFree(p);
    return;
  }
  const size_t sz = it->second.first;
  const int dev = it->second.second;
  c.live.erase(it);
  static const bool off = [] {
    const char *v = std::getenv("FB_NO_MEMORY_CACHE");
    return v && v[0] == '1';
  }();
  if (off) {
    cudaFree(p);
    return;
  }
  c.free_blocks[dev & 15].emplace(sz, p);
  c.cached_bytes += sz;
}

size_t dev_cache_trim() {
  DevCache &c = dev_cache();
  cudaDeviceSynchronize();
  std::lock_guard<std::mutex> lock(c.mu);
  const size_t b = c.cached_bytes;
  trim_locked(c);
  return b;
}

// Host threads of the staging copies / comparisons below.  torchrun exports OMP_NUM_THREADS=1 to every rank, which would
// serialise the 8-24 MB copies on the end-to-end path; they take an explicit team instead: FB_IO_THREADS, else the
// machine's hardware threads divided among the ranks of this node (LOCAL_WORLD_SIZE), at most 16.
int io_threads() {  // referenced from OpenMP clauses only (not static: the device front end would call it unused)
  static const int n = [] {
    if (const char *v = std::getenv("FB_IO_THREADS")) return std::max(1, std::atoi(v));
    int ranks = 1;
    if (const char *v = std::getenv("LOCAL_WORLD_SIZE")) ranks = std::max(1, std::atoi(v));
    const int hw = (int)std::max(1u, std::thread::hardware_concurrency());
    return std::max(1, std::min(16, hw / ranks));
  }();
  return n;
}

// bytewise equality of two host buffers, all host threads (24 MB in ~0.3 ms: cheaper than moving them over PCIe)
static bool same_bytes(const void *a, const void *b, size_t bytes) {
  // two different vectors differ in their first few values: settle that case before the thread team starts
  const size_t head = std::min<size_t>(bytes, 4096);
  if (std::memcmp(a, b, head) != 0) return false;
  const size_t chunk = 1 << 18;
  const long nchunks = (long)((bytes + chunk - 1) / chunk);
  std::atomic<int> differ{0};
#pragma omp parallel for schedule(static) num_threads(io_threads())
  for (long c = 0; c < nchunks; ++c) {
    if (differ.load(std::memory_order_relaxed)) continue;
    const size_t off = (size_t)c * chunk, len = std::min(chunk, bytes - off);
    if (std::memcmp((const char *)a + off, (const char *)b + off, len) != 0) differ.store(1, std::memory_order_relaxed);
  }
  return differ.load() == 0;
}
static void copy_bytes(void *dst, const void *src, size_t bytes) {
  const size_t chunk = 1 << 18;
  const long nchunks = (long)((bytes + chunk - 1) / chunk);
#pragma omp parallel for schedule(static) num_threads(io_threads())
  for (long c = 0; c < nchunks; ++c) {
    const size_t off = (size_t)c * chunk, len = std::min(chunk, bytes - off);
    std::memcpy((char *)dst + off, (const char *)src + off, len);
  }
}

template <class K>
static void set_smem(K kernel, size_t bytes) {
  if (bytes > 48 * 1024)
    FB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
}

}  // namespace fb

using namespace fb;

fb_tree::~fb_tree() {
  for (auto &e : ev)
    if (e) cudaEventDestroy(e);
  for (auto &e : ev_mv)
    if (e) cudaEventDestroy(e);
  if (ev_fork) cudaEventDestroy(ev_fork);
  if (ev_join) cudaEventDestroy(ev_join);
  if (stream2) cudaStreamDestroy(stream2);
  if (stream) cudaStreamDestroy(stream);
  if (m2l_plan) m2l_stream_free(m2l_plan);
  if (shard) fb_shard_free(shard);
}

// ------------------------------------------------------------------------------------------- build
void fb_tree::build(const double *points, size_t n_, int dim_, ptrdiff_t rs, ptrdiff_t cs, int order_,
                    const fb_kernel_params *k, int adaptive, int sparse, const double *extents,
                    const fb_fmm_params *params) {
  FB_REQUIRE(points && n_ > 0, "source_points must be a non-empty n x dim matrix");
  FB_REQUIRE(dim_ >= 1 && dim_ <= 3, "Unsupported number of dimensions: " + std::to_string(dim_));
  FB_REQUIRE(order_ >= 1 && order_ <= kMaxOrder, "interpolation_order must be in 1.." + std::to_string(kMaxOrder));
  FB_REQUIRE(n_ < (1ull << 31), "at most 2^31-1 source points per tree");
  FB_REQUIRE(k != nullptr, "kernel params required");
  // kernel_helpers.rs:72-73 asserts live in KernelParamsBuilder::build (mirrored by the Python KernelParams class);
  // FmmTree::new itself accepts any KernelParams
  FB_REQUIRE(make_kparams(*k, kp), "unknown kernel_type");
  kp.fast = g_sqrt_mode.load();
  kparams_c = *k;
  n = n_;
  dim = dim_;
  order = order_;
  P = 1;
  for (int d = 0; d < dim; ++d) P *= order;
  if (params) {
    fparams = *params;
  } else {  // FmmParams::new_defaults, bbfmm.rs:95-104
    fparams.max_points_per_cell = 256;
    fparams.compression_type = FB_COMPRESSION_ACA;
    fparams.epsilon = std::pow(10.0, -(double)order);
    fparams.eval_chunk_size = 1024;
  }
  FB_REQUIRE(fparams.compression_type >= 0 && fparams.compression_type <= 2, "unknown compression type");

  const bool verbose = std::getenv("FB_TIMING") != nullptr;
  auto t_lap = std::chrono::steady_clock::now();
  auto lap = [&](const char *what) {
    if (verbose)
      fprintf(stderr, "[fb_tree] %-28s %8.3f s\n", what,
              std::chrono::duration<double>(std::chrono::steady_clock::now() - t_lap).count());
    t_lap = std::chrono::steady_clock::now();
  };
  FB_CUDA(cudaGetDevice(&device));
  {
    int prio_lo = 0, prio_hi = 0;
    FB_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    FB_CUDA(cudaStreamCreateWithPriority(&stream, cudaStreamNonBlocking, prio_hi));
    FB_CUDA(cudaStreamCreateWithPriority(&stream2, cudaStreamNonBlocking, prio_lo));
    FB_CUDA(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
    FB_CUDA(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
    const char *ov = std::getenv("FB_OVERLAP");
    overlap_p2p = ov && ov[0] == '1';  // measured slower on B200 (15.1 vs 13.6 ms), kept as an opt-in experiment
  }
  for (auto &e : ev) FB_CUDA(cudaEventCreate(&e));
  for (auto &e : ev_mv) FB_CUDA(cudaEventCreate(&e));

  host_points.resize(n * dim);
  for (size_t i = 0; i < n; ++i)
    for (int d = 0; d < dim; ++d) host_points[i * dim + d] = points[(ptrdiff_t)i * rs + (ptrdiff_t)d * cs];

  // extents: given [mins..., maxs...] or from the data (bbfmm.rs:281-284, utils.rs:22-54)
  double ext[6];
  if (extents) {
    for (int d = 0; d < 2 * dim; ++d) ext[d] = extents[d];
  } else {
    for (int d = 0; d < dim; ++d) ext[d] = ext[dim + d] = host_points[d];
    for (size_t i = 0; i < n; ++i)
      for (int d = 0; d < dim; ++d) {
        const double v = host_points[i * dim + d];
        if (v < ext[d]) ext[d] = v;
        if (v > ext[dim + d]) ext[dim + d] = v;
      }
  }
  // calculate_tree_center_and_radius, morton.rs:349-373
  double center[3] = {0, 0, 0}, radius = -INFINITY;
  for (int d = 0; d < dim; ++d) {
    const double lo = std::floor(ext[d]), hi = std::ceil(ext[dim + d]);
    center[d] = (lo + hi) / 2.0;
    radius = std::max(radius, (hi - lo) / 2.0 + 1e-3);
  }
  FB_REQUIRE(std::isfinite(radius) && radius > 0, "invalid extents");

  // ---- device radix sort of the level-16 Morton codes
  DBuf<double> &d_pts = d_pts_user;  // kept: evaluate() recognises targets that are exactly the source points
  d_pts.reserve(n * dim);
  FB_CUDA(cudaMemcpyAsync(d_pts.p, host_points.data(), n * dim * sizeof(double), cudaMemcpyHostToDevice, stream));
  DBuf<unsigned long long> d_codes, d_codes2;
  DBuf<uint32_t> d_idx;
  d_codes.reserve(n);
  d_codes2.reserve(n);
  d_idx.reserve(n);
  d_perm.reserve(n);
  d_inv.reserve(n);
  d_err.reserve(1);
  FB_CUDA(cudaMemsetAsync(d_err.p, 0xFF, sizeof(unsigned long long), stream));
  const double side16 = 2.0 * radius / 65536.0;  // morton.rs:29-32 at level 16
  FB_LAUNCH(k_point_codes, nblocks(n, 256), 256, 0, stream, d_pts.p, n, dim, center[0] - radius, center[1] - radius,
            center[2] - radius, side16, d_codes.p, d_idx.p, d_err.p);
  size_t cub_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, d_codes.p, d_codes2.p, d_idx.p, d_perm.p, (int)n, 0, 16 * dim,
                                  stream);
  d_cub.reserve(cub_bytes);
  FB_CUDA(cub::DeviceRadixSort::SortPairs(d_cub.p, cub_bytes, d_codes.p, d_codes2.p, d_idx.p, d_perm.p, (int)n, 0,
                                          16 * dim, stream));
  g_launches.fetch_add(4);
  d_sx.reserve(n);
  d_sy.reserve(n);
  d_sz.reserve(n);
  FB_LAUNCH(k_gather_sorted, nblocks(n, 256), 256, 0, stream, d_pts.p, d_perm.p, n, dim, d_sx.p, d_sy.p, d_sz.p,
            d_inv.p);
  std::vector<unsigned long long> h_codes(n);
  unsigned long long h_err = 0;
  FB_CUDA(cudaMemcpyAsync(h_codes.data(), d_codes2.p, n * sizeof(unsigned long long), cudaMemcpyDeviceToHost, stream));
  FB_CUDA(cudaMemcpyAsync(&h_err, d_err.p, sizeof(h_err), cudaMemcpyDeviceToHost, stream));
  FB_CUDA(cudaStreamSynchronize(stream));
  if (h_err != ~0ull)
    throw Error(FB_ERR_INVALID_ARGUMENT,
                "source point at row " + std::to_string(h_err) + " lies outside the given tree extents", h_err);

  lap("copy + device sort");
  // ---- host: adaptive/uniform subdivision over the sorted codes + interaction lists
  ht.build((const uint64_t *)h_codes.data(), n, dim, center, radius, (size_t)fparams.max_points_per_cell, !sparse,
           adaptive != 0);
  const size_t nc = ht.ncells();
  const int nl = (int)ht.leaves.size();

  lap("tree + lists (host)");
  // ---- host: operators
  ops.build_cached(order, dim, radius, ht.depth, kp, fparams.compression_type, fparams.epsilon);
  lap("operators (host)");

  // ---- upload cells
  std::vector<double> ccx(nc), ccy(nc), ccz(nc), chalf(nc);
  std::vector<int> slot(nc);
  for (size_t c = 0; c < nc; ++c) {
    double cc[3] = {0, 0, 0}, side;
    ht.cell_center((int)c, cc, side);
    ccx[c] = cc[0];
    ccy[c] = dim > 1 ? cc[1] : 0.0;
    ccz[c] = dim > 2 ? cc[2] : 0.0;
    chalf[c] = side * 0.5;
    slot[c] = (int)(ht.prefix[c] & ((1u << dim) - 1u));  // morton.rs:300-305
  }
  d_ccx.upload(ccx, stream);
  d_ccy.upload(ccy, stream);
  d_ccz.upload(ccz, stream);
  d_chalf.upload(chalf, stream);
  d_cell_slot.upload(slot, stream);
  d_cell_parent.upload(ht.parent, stream);
  d_cell_ptb.upload(ht.pt_begin, stream);
  d_cell_pte.upload(ht.pt_end, stream);
  d_child_ptr.upload(ht.child_ptr, stream);
  d_child_idx.upload(ht.child_idx, stream);
  std::vector<uint8_t> ones(nc, 1);
  d_flag_all.upload(ones, stream);

  // leaves
  std::vector<int> cell_to_leaf(nc, -1);
  std::vector<unsigned long long> llo(nl), lhi(nl);
  std::vector<int> src_leaves, tl_b(nl), tl_e(nl);
  for (int l = 0; l < nl; ++l) {
    const int c = ht.leaves[l];
    cell_to_leaf[c] = l;
    const int sh = dim * (16 - ht.level[c]);
    llo[l] = ht.prefix[c] << sh;
    lhi[l] = llo[l] + (1ull << sh);
    tl_b[l] = ht.pt_begin[c];
    tl_e[l] = ht.pt_end[c];
    if (ht.pt_end[c] > ht.pt_begin[c]) src_leaves.push_back(c);
  }
  d_leaf_cell.upload(ht.leaves, stream);
  d_leaf_lo.upload(llo, stream);
  d_leaf_hi.upload(lhi, stream);
  d_src_leaves.upload(src_leaves, stream);
  n_src_leaves = (int)src_leaves.size();
  d_src_tl_begin.upload(tl_b, stream);
  d_src_tl_end.upload(tl_e, stream);
  // non-leaf cells per level (M2M grids)
  h_parents.assign(ht.depth + 1, {});
  for (size_t c = 0; c < nc; ++c)
    if (ht.child_ptr[c + 1] > ht.child_ptr[c]) h_parents[ht.level[c]].push_back((int)c);
  {
    std::vector<int> flat;
    parents_off.assign(ht.depth + 2, 0);
    for (int l = 0; l <= ht.depth; ++l) {
      parents_off[l] = (int)flat.size();
      flat.insert(flat.end(), h_parents[l].begin(), h_parents[l].end());
    }
    parents_off[ht.depth + 1] = (int)flat.size();
    d_parents.upload(flat, stream);
  }
  // all-sources target set: tiles per leaf
  {
    std::vector<int> t_leaf, t_off;
    for (int l = 0; l < nl; ++l)
      for (int o = 0; o < tl_e[l] - tl_b[l]; o += kTile) {
        t_leaf.push_back(l);
        t_off.push_back(o);
      }
    src_tiles = (int)t_leaf.size();
    d_src_tile_leaf.upload(t_leaf, stream);
    d_src_tile_off.upload(t_off, stream);
    std::vector<int> nt{src_tiles};
    d_src_ntiles.upload(nt, stream);
  }

  // ---- leaf lists: U as merged contiguous source ranges, W as cells; X per cell as ranges
  {
    std::vector<long long> u_ptr(nl + 1, 0), w_ptr(nl + 1, 0);
    std::vector<int> u_b, u_c, w_c;
    p2p_pairs = m2p_pairs = p2l_pairs = 0;
    std::vector<std::pair<int, int>> rng;
    for (int l = 0; l < nl; ++l) {
      const int c = ht.leaves[l];
      rng.clear();
      uint64_t nsrc = 0;
      for (long long e = ht.u_ptr[c]; e < ht.u_ptr[c + 1]; ++e) {
        const int u = ht.u_idx[e];
        if (ht.pt_end[u] > ht.pt_begin[u]) {
          rng.emplace_back(ht.pt_begin[u], ht.pt_end[u]);
          nsrc += ht.pt_end[u] - ht.pt_begin[u];
        }
      }
      std::sort(rng.begin(), rng.end());
      for (size_t i = 0; i < rng.size(); ++i) {
        if (!u_b.empty() && (long long)u_b.size() > u_ptr[l] && u_b.back() + u_c.back() == rng[i].first)
          u_c.back() += rng[i].second - rng[i].first;
        else {
          u_b.push_back(rng[i].first);
          u_c.push_back(rng[i].second - rng[i].first);
        }
      }
      u_ptr[l + 1] = (long long)u_b.size();
      const uint64_t nt = ht.pt_end[c] - ht.pt_begin[c];
      p2p_pairs += nt * nsrc;
      for (long long e = ht.w_ptr[c]; e < ht.w_ptr[c + 1]; ++e) w_c.push_back(ht.w_idx[e]);
      w_ptr[l + 1] = (long long)w_c.size();
      m2p_pairs += nt * (uint64_t)(ht.w_ptr[c + 1] - ht.w_ptr[c]);
    }
    d_u_ptr.upload(u_ptr, stream);
    d_u_begin.upload(u_b, stream);
    d_u_count.upload(u_c, stream);
    d_w_ptr.upload(w_ptr, stream);
    d_w_ptr_none.upload(std::vector<long long>(nl + 1, 0), stream);
    d_w_cell.upload(w_c, stream);
    n_w_entries = (long long)w_c.size();
    // one CTA per X cell (p2l.cu), dispatched in blockIdx order: the cells are listed by descending source count so that
    // the long lists start first and the short ones fill the tail of the grid (a rank's share of a partitioned tree is
    // only a couple of waves deep)
    std::vector<int> x_cells, x_b, x_c;
    std::vector<long long> x_ptr{0};
    {
      struct XCell {
        int cell;
        long long count;
        std::vector<std::pair<int, int>> ranges;
      };
      std::vector<XCell> xs;
      for (size_t c = 0; c < nc; ++c) {
        if (ht.x_ptr[c + 1] == ht.x_ptr[c]) continue;
        rng.clear();
        long long cnt = 0;
        for (long long e = ht.x_ptr[c]; e < ht.x_ptr[c + 1]; ++e) {
          const int x = ht.x_idx[e];
          if (ht.pt_end[x] > ht.pt_begin[x]) {
            rng.emplace_back(ht.pt_begin[x], ht.pt_end[x]);
            cnt += ht.pt_end[x] - ht.pt_begin[x];
          }
        }
        if (rng.empty()) continue;
        p2l_pairs += (uint64_t)cnt;
        std::sort(rng.begin(), rng.end());
        XCell xc{(int)c, cnt, {}};
        for (auto &r : rng) {
          if (!xc.ranges.empty() && xc.ranges.back().first + xc.ranges.back().second == r.first)
            xc.ranges.back().second += r.second - r.first;
          else
            xc.ranges.emplace_back(r.first, r.second - r.first);
        }
        xs.push_back(std::move(xc));
      }
      std::stable_sort(xs.begin(), xs.end(), [](const XCell &a, const XCell &b) { return a.count > b.count; });
      for (const XCell &xc : xs) {
        for (auto &r : xc.ranges) {
          x_b.push_back(r.first);
          x_c.push_back(r.second);
        }
        x_cells.push_back(xc.cell);
        x_ptr.push_back((long long)x_b.size());
      }
    }
    n_x_cells = (int)x_cells.size();
    d_x_cells.upload(x_cells, stream);
    d_x_ptr.upload(x_ptr, stream);
    d_x_begin.upload(x_b, stream);
    d_x_count.upload(x_c, stream);
  }

  // ---- operators to device
  d_nodes.upload(ops.nodes, stream);
  d_tnodes.upload(ops.tnodes, stream);
  d_child_s.upload(ops.child_s, stream);
  {
    std::vector<int> pt(ops.perm.begin(), ops.perm.end());
    d_perm_tab.upload(pt, stream);
    std::vector<int> it(ops.inv_perm.begin(), ops.inv_perm.end());
    d_inv_tab.upload(it, stream);
  }
  // M2L: the streaming kernel (m2l.cu) when the order fits its register-resident operator slices ...
  lap("leaf list packing + upload");
  if (m2l_stream_supported(P, fparams.compression_type) && ht.depth >= 2)
    m2l_plan = m2l_stream_build(ht, ops, P, d_inv_tab.p, stream);
  lap("M2L stream plan");
  // ... else groups of entries (target, source, permutation) per (level, reference vector), sorted by target
  if (!m2l_plan) {
    m2l_groups.clear();
    std::vector<double> pool;
    std::vector<int> e_tgt, e_src, e_perm;
    const bool compressed = fparams.compression_type != FB_COMPRESSION_NONE;
    const int P4 = ((P + 3) / 4) * 4, P8 = ((P + 7) / 8) * 8;
    for (int lvl = 2; lvl <= ht.depth; ++lvl) {
      std::vector<std::vector<std::array<int, 3>>> per_ref(ops.n_ref);
      for (int c = ht.level_ptr[lvl]; c < ht.level_ptr[lvl + 1]; ++c) {
        uint32_t ac[3];
        ht.anchor(c, ac);
        for (long long e = ht.v_ptr[c]; e < ht.v_ptr[c + 1]; ++e) {
          const int s = ht.v_idx[e];
          uint32_t as[3];
          ht.anchor(s, as);
          int tix = 0;  // calculate_m2l_transfer_index, bbfmm.rs:989-998: t = round((c_target - c_source)/side)
          for (int d = 0; d < dim; ++d) tix = tix * 7 + ((int)ac[d] - (int)as[d] + 3);
          per_ref[ops.ref_lookup[tix]].push_back({c, s, ops.perm_lookup[tix]});
        }
      }
      for (int r = 0; r < ops.n_ref; ++r) {
        if (per_ref[r].empty()) continue;
        const M2LOperator &op = ops.m2l[lvl - 2][r];
        M2LGroup g;
        g.level = lvl;
        g.ref = r;
        g.rank = op.rank;
        g.rank_pad = compressed ? std::max(8, ((op.rank + 7) / 8) * 8) : P4;
        g.n_entries = per_ref[r].size();
        g.entry_off = e_tgt.size();
        for (auto &t : per_ref[r]) {
          e_tgt.push_back(t[0]);
          e_src.push_back(t[1]);
          e_perm.push_back(t[2]);
        }
        // operators in DMMA fragment order: frag(mt, ks)[lane] = Op[mt*8 + lane/4][ks*4 + lane%4], zero padded
        auto pack = [&](int rows, int cols, int rows_pad, int cols_pad, auto get) {
          const size_t off = pool.size();
          const int mtn = rows_pad / 8, ksn = cols_pad / 4;
          pool.resize(off + (size_t)mtn * ksn * 32, 0.0);
          for (int mt = 0; mt < mtn; ++mt)
            for (int ks = 0; ks < ksn; ++ks)
              for (int l = 0; l < 32; ++l) {
                const int rr = mt * 8 + l / 4, cc = ks * 4 + l % 4;
                if (rr < rows && cc < cols) pool[off + ((size_t)mt * ksn + ks) * 32 + l] = get(rr, cc);
              }
          return off;
        };
        if (compressed) {
          g.v_off = pack(op.rank, P, g.rank_pad, P4, [&](int rr, int cc) { return op.Vt(rr, cc); });
          g.u_off = pack(P, op.rank, P8, g.rank_pad, [&](int rr, int cc) { return op.U(rr, cc); });
        } else {
          g.v_off = 0;
          g.u_off = pack(P, P, P8, P4, [&](int rr, int cc) { return op.U(rr, cc); });
        }
        m2l_groups.push_back(g);
      }
    }
    d_oppool.upload(pool, stream);
    d_m2l_tgt.upload(e_tgt, stream);
    d_m2l_src.upload(e_src, stream);
    d_m2l_perm.upload(e_perm, stream);
    int max_rp = 8;
    for (auto &g : m2l_groups) max_rp = std::max(max_rp, compressed ? g.rank_pad : 0);
    m2l_P4 = P4;
    m2l_Pp = P4;
    while (m2l_Pp % 16 != 4 && m2l_Pp % 16 != 12) m2l_Pp += 4;  // bank-conflict-free B fragments
    m2l_nc = 0;
    const char *nc_env = std::getenv("FB_M2L_NC");  // experiment knob: cap the column tile
    const int nc_cap = nc_env ? std::atoi(nc_env) : 32;
    for (int nc : {64, 32, 16, 8}) {  // columns per CTA: the largest tile that fits in shared memory
      if (nc > nc_cap) continue;
      const size_t need = sizeof(double) * ((size_t)nc * m2l_Pp + (size_t)max_rp * (nc + 4));
      if (need <= 220 * 1024) {
        m2l_nc = nc;
        m2l_smem = need;
        break;
      }
    }
    FB_REQUIRE(m2l_nc != 0, "interpolation order too large for the M2L shared-memory tile (p^d <= ~3300)");
  }
  FB_CUDA(cudaStreamSynchronize(stream));
  lap("list packing + upload");
  have_weights = have_locals = false;
}

// --------------------------------------------------------------------------------------- weights
bool fb_tree::upload_weights(const double *w, size_t n_rows, size_t nrhs_, ptrdiff_t rs, ptrdiff_t cs) {
  FB_REQUIRE(w != nullptr, "weights required");
  FB_REQUIRE(n_rows >= n, "weights must have at least one row per source point");
  FB_REQUIRE(nrhs_ >= 1, "weights need at least one column");
  const size_t cnt = n * nrhs_;
  const bool contiguous = cs == 1 && rs == (ptrdiff_t)nrhs_;
  // The reference API passes the weights twice per matvec (set_weights(w), then evaluate(w, ..): bbfmm.rs:383, 444);
  // the second copy is recognised on the host and neither re-uploaded nor re-sorted.
  if (contiguous && w_cache_valid && (int)nrhs_ == nrhs && h_w_last_cnt == cnt && d_w.cap >= cnt &&
      same_bytes(w, h_w_last.p, cnt * sizeof(double)))
    return false;
  // fb_tree_set_weights returns without waiting for its transfer and upward pass: make sure nothing is still reading
  // the staging buffers before they are rewritten (or reallocated)
  FB_CUDA(cudaStreamSynchronize(stream));
  d_w_user.reserve(cnt);
  if (contiguous) {
    // user memory is pageable: gather it into the pinned cache with all host threads and send it from there
    h_w_last.reserve(cnt);
    // in pieces: the transfer of one piece runs under the host copy of the next
    const size_t piece = std::max<size_t>((cnt + 3) / 4, (size_t)1 << 17);
    for (size_t off = 0; off < cnt; off += piece) {
      const size_t len = std::min(piece, cnt - off);
      copy_bytes(h_w_last.p + off, w + off, len * sizeof(double));
      FB_CUDA(cudaMemcpyAsync(d_w_user.p + off, h_w_last.p + off, len * sizeof(double), cudaMemcpyHostToDevice, stream));
    }
    h_w_last_cnt = cnt;
    w_cache_valid = true;
  } else {
    w_cache_valid = false;
    h_stage.reserve(cnt);
    for (size_t i = 0; i < n; ++i)
      for (size_t r = 0; r < nrhs_; ++r) h_stage.p[i * nrhs_ + r] = w[(ptrdiff_t)i * rs + (ptrdiff_t)r * cs];
    FB_CUDA(cudaMemcpyAsync(d_w_user.p, h_stage.p, cnt * sizeof(double), cudaMemcpyHostToDevice, stream));
  }
  nrhs = (int)nrhs_;
  sort_weights();
  last_w_ptr = contiguous ? w : nullptr;
  return true;
}

void fb_tree::sort_weights() {
  d_w.reserve(n * (size_t)nrhs);
  FB_LAUNCH(k_sort_weights, nblocks(n, 256), 256, 0, stream, d_w_user.p, d_perm.p, n, nrhs, d_w.p);
}

// ---------------------------------------------------------------------------------------- upward
void fb_tree::upward(const int *leaves, int n_leaves, const uint8_t *cell_flag) {
  const size_t nc = ht.ncells();
  d_mult.zero(nc * (size_t)nrhs * coef_stride(P), stream);
  const int p = order;
  if (timing) FB_CUDA(cudaEventRecord(ev[0], stream));
  const int nsl = leaves ? n_leaves : n_src_leaves;
  const int *leaf_list = leaves ? leaves : d_src_leaves.p;
  if (nsl > 0 && !launch_p2m_fast(nsl, leaf_list, d_cell_ptb.p, d_cell_pte.p, d_sx.p, d_sy.p, d_sz.p, d_w.p, n,
                                  d_ccx.p, d_ccy.p, d_ccz.p, d_chalf.p, d_tnodes.p, p, dim, nrhs, d_mult.p, stream)) {
    const size_t smem = sizeof(double) * ((size_t)p * p + 3 * (size_t)kP2MChunk * p);
    set_smem(k_p2m, smem);
    FB_LAUNCH(k_p2m, nsl, 256, smem, stream, leaf_list, d_cell_ptb.p, d_cell_pte.p, d_sx.p, d_sy.p, d_sz.p,
              d_w.p, n, d_ccx.p, d_ccy.p, d_ccz.p, d_chalf.p, d_tnodes.p, p, dim, P, nrhs, d_mult.p);
  }
  if (timing) FB_CUDA(cudaEventRecord(ev[1], stream));
  int cpar = 1 << dim;  // children in flight per parent: all of them unless p^d is too large for shared memory
  while (cpar > 1 && sizeof(double) * (2 * (size_t)p * p + 2 * (size_t)cpar * P) > 200 * 1024) cpar >>= 1;
  const size_t smem = sizeof(double) * (2 * (size_t)p * p + 2 * (size_t)cpar * P);
  set_smem(k_m2m, smem);
  // bbfmm.rs:675-687 goes up to the level-1 parents; their multipoles are never read (V, W and X lists only hold cells
  // of level >= 2: every level-1 cell touches every other), so the last, eight-cell launch is left out
  for (int lvl = ht.depth - 1; lvl >= 2; --lvl) {
    const int np = parents_off[lvl + 1] - parents_off[lvl];
    if (np <= 0) continue;
    FB_LAUNCH(k_m2m, np, 256, smem, stream, d_parents.p + parents_off[lvl], d_child_ptr.p, d_child_idx.p,
              d_cell_slot.p, d_child_s.p, p, dim, P, nrhs, cell_flag, cpar, d_mult.p);
  }
  if (timing) FB_CUDA(cudaEventRecord(ev[2], stream));
  have_weights = true;
}

// -------------------------------------------------------------------------------------- downward
void fb_tree::downward(const uint8_t *flags, const TargetSet *fuse_m2p, bool out_zeroed, bool m2l_one_cta_per_sm,
                       const M2LItemTable *m2l_table) {
  const size_t nc = ht.ncells();
  const int p = order;
  d_loc.zero(nc * (size_t)nrhs * coef_stride(P), stream);
  if (fuse_m2p && !out_zeroed) d_out.zero(fuse_m2p->m * (size_t)nrhs, stream);
  if (timing) FB_CUDA(cudaEventRecord(ev[3], stream));
  // M2L (loop A of bbfmm.rs:781-832)
  const bool compressed = fparams.compression_type != FB_COMPRESSION_NONE;
  if (m2l_plan) {
    m2l_stream_launch(m2l_plan, nrhs, flags == d_flag_all.p ? nullptr : flags, m2l_table, d_mult.p, d_loc.p, stream);
  } else if (!m2l_groups.empty()) {
    if (m2l_table_nrhs != nrhs) {  // CTA ranges depend on the number of right-hand sides
      std::vector<M2LGroupDev> tab;
      std::vector<int> cta_group;
      long long cta = 0;
      for (const M2LGroup &g : m2l_groups) {
        M2LGroupDev t;
        t.cta_begin = (int)cta;
        t.rank_pad = g.rank_pad;
        t.entry_off = (long long)g.entry_off;
        t.n_entries = (long long)g.n_entries;
        t.v_off = (long long)g.v_off;
        t.u_off = (long long)g.u_off;
        const long long nct = (long long)((g.n_entries * (size_t)nrhs + m2l_nc - 1) / m2l_nc);
        cta_group.insert(cta_group.end(), (size_t)nct, (int)tab.size());
        tab.push_back(t);
        cta += nct;
      }
      FB_REQUIRE(cta < (1ll << 31), "too many M2L tiles");
      m2l_ctas = (unsigned)cta;
      d_m2l_table.reserve(tab.size() * sizeof(M2LGroupDev));
      FB_CUDA(cudaMemcpyAsync(d_m2l_table.p, tab.data(), tab.size() * sizeof(M2LGroupDev), cudaMemcpyHostToDevice,
                              stream));
      d_m2l_cta_group.upload(cta_group, stream);
      FB_CUDA(cudaStreamSynchronize(stream));
      m2l_table_nrhs = nrhs;
    }
    const M2LGroupDev *tab = reinterpret_cast<const M2LGroupDev *>(d_m2l_table.p);
    // sharing the SM with the concurrent P2P kernel: ask for more than half of the shared memory so that one CTA
    // (half of the registers) is resident per SM and the P2P CTAs fit beside it
    const size_t m2l_smem_launch = m2l_one_cta_per_sm ? std::max(m2l_smem, (size_t)116 * 1024) : m2l_smem;
#define FB_M2L_LAUNCH(COMP, NCV)                                                                                   \
  do {                                                                                                             \
    set_smem(k_m2l<COMP, NCV>, m2l_smem_launch);                                                                   \
    FB_LAUNCH((k_m2l<COMP, NCV>), m2l_ctas, (NCV) == 64 ? 512 : 256, m2l_smem_launch, stream, tab, d_m2l_cta_group.p, d_m2l_tgt.p,   \
              d_m2l_src.p, d_m2l_perm.p, d_oppool.p, d_perm_tab.p, d_inv_tab.p, P, m2l_P4, m2l_Pp, nrhs, flags,    \
              d_mult.p, d_loc.p);                                                                                  \
  } while (0)
    if (compressed) {
      if (m2l_nc == 64) FB_M2L_LAUNCH(true, 64);
      else if (m2l_nc == 32) FB_M2L_LAUNCH(true, 32);
      else if (m2l_nc == 16) FB_M2L_LAUNCH(true, 16);
      else FB_M2L_LAUNCH(true, 8);
    } else {
      if (m2l_nc == 64) FB_M2L_LAUNCH(false, 64);
      else if (m2l_nc == 32) FB_M2L_LAUNCH(false, 32);
      else if (m2l_nc == 16) FB_M2L_LAUNCH(false, 16);
      else FB_M2L_LAUNCH(false, 8);
    }
#undef FB_M2L_LAUNCH
  }
  if (timing) FB_CUDA(cudaEventRecord(ev[4], stream));
  // P2L (adaptive only)
  if (ht.adaptive && n_x_cells > 0) {
    P2LArgs a{};
    a.cells = d_x_cells.p;
    a.n_cells = n_x_cells;
    a.x_ptr = d_x_ptr.p;
    a.x_begin = d_x_begin.p;
    a.x_count = d_x_count.p;
    a.cell_flag = flags;
    a.sx = d_sx.p;
    a.sy = d_sy.p;
    a.sz = d_sz.p;
    a.w = d_w.p;
    a.n = n;
    a.loc = d_loc.p;
    a.ccx = d_ccx.p;
    a.ccy = d_ccy.p;
    a.ccz = d_ccz.p;
    a.chalf = d_chalf.p;
    a.nodes = d_nodes.p;
    a.p = p;
    a.dim = dim;
    a.P = P;
    a.nrhs = nrhs;
    a.rhs0 = 0;
    a.kp = kp;
    if (fuse_m2p) {
      a.mult = d_mult.p;
      a.out = d_out.p;
      a.out_row = fuse_m2p->row_of_pos;
      a.tgt_prefix = fuse_m2p->tgt_prefix;
      if (fuse_m2p->own_hi > fuse_m2p->own_lo && !fuse_m2p->all_sources) {  // a rank's share of a partitioned tree
        a.cell_ptb = d_cell_ptb.p;
        a.own_lo = fuse_m2p->own_lo;
        a.own_hi = fuse_m2p->own_hi;
      }
    }
    launch_p2l(a, stream);
  }
  if (timing) FB_CUDA(cudaEventRecord(ev[5], stream));
  // L2L (loop B of bbfmm.rs:834-856): children at levels 2..depth
  const size_t smem = sizeof(double) * (2 * (size_t)p * p + 2 * (size_t)P);
  set_smem(k_l2l, smem);
  // (level-1 locals are identically zero — no M2L or P2L reaches that level — so the children of level 2 have nothing
  // to inherit and the loop starts one level further down)
  for (int lvl = 3; lvl <= ht.depth; ++lvl) {
    const int c0 = ht.level_ptr[lvl], cnt = ht.level_ptr[lvl + 1] - c0;
    if (cnt <= 0) continue;
    FB_LAUNCH(k_l2l, cnt, 128, smem, stream, c0, d_cell_parent.p, d_cell_slot.p, flags, d_child_s.p, p, dim, P, nrhs,
              d_loc.p);
  }
  if (timing) FB_CUDA(cudaEventRecord(ev[6], stream));
  have_locals = true;
}

// ------------------------------------------------------------------------------------- leaf pass
void fb_tree::launch_l2p(const TargetSet &ts, bool grads) {
  const int p = order;
  if (ts.max_tiles <= 0) return;
  if (!grads && launch_l2p_fast(ts, d_leaf_cell.p, d_loc.p, d_ccx.p, d_ccy.p, d_ccz.p, d_chalf.p, d_tnodes.p, p, dim,
                                nrhs, d_out.p, stream))
    return;
  const size_t smem = sizeof(double) * ((size_t)p * p + P + (size_t)kTile * dim * p * (grads ? 2 : 1));
  set_smem(k_l2p, smem);
  FB_LAUNCH(k_l2p, ts.max_tiles, kTile, smem, stream, ts, d_leaf_cell.p, d_loc.p, d_ccx.p, d_ccy.p, d_ccz.p,
            d_chalf.p, d_tnodes.p, p, dim, P, nrhs, d_out.p, grads ? d_gout.p : nullptr);
}

void fb_tree::launch_p2p(const TargetSet &ts, bool grads, bool m2p_done, cudaStream_t s, bool atomic_out,
                         bool w_only) {
  DirectArgs a{};
  a.ts = ts;
  a.u_ptr = d_u_ptr.p;
  a.u_begin = d_u_begin.p;
  a.u_count = d_u_count.p;
  a.w_ptr = m2p_done ? d_w_ptr_none.p : d_w_ptr.p;  // fused: the W lists were applied by the P2L kernel
  a.w_cell = d_w_cell.p;
  a.sx = d_sx.p;
  a.sy = d_sy.p;
  a.sz = d_sz.p;
  a.w = d_w.p;
  a.n = n;
  a.mult = d_mult.p;
  a.ccx = d_ccx.p;
  a.ccy = d_ccy.p;
  a.ccz = d_ccz.p;
  a.chalf = d_chalf.p;
  a.nodes = d_nodes.p;
  a.p = order;
  a.dim = dim;
  a.P = P;
  a.nrhs = nrhs;
  a.rhs0 = 0;
  a.atomic_out = atomic_out ? 1 : 0;
  a.has_w = (!m2p_done && n_w_entries > 0) ? 1 : 0;
  a.skip_p2p = w_only ? 1 : 0;
  a.sym_row = ts.own_hi > ts.own_lo ? d_src_out_row.p : nullptr;  // filled by source_target_set()
  a.out = d_out.p;
  a.gout = grads ? d_gout.p : nullptr;
  a.kp = kp;
  launch_leaf_direct(a, s);
}

void fb_tree::leaf_pass(const TargetSet &ts, bool grads, bool m2p_done) {
  if (!m2p_done) d_out.zero(ts.m * (size_t)nrhs, stream);
  if (grads) d_gout.zero(ts.m * (size_t)nrhs * dim, stream);
  if (timing) FB_CUDA(cudaEventRecord(ev[7], stream));
  launch_l2p(ts, grads);
  if (timing) FB_CUDA(cudaEventRecord(ev[8], stream));
  launch_p2p(ts, grads, m2p_done, stream, false);
  if (timing) FB_CUDA(cudaEventRecord(ev[9], stream));
  last_overlapped = false;
}

// ----------------------------------------------------------------------------------- target sets
TargetSet fb_tree::source_target_set() {
  if (d_src_out_row.cap < n) {  // out_row = source row of each sorted position
    d_src_out_row.reserve(n);
    FB_CUDA(cudaMemcpyAsync(d_src_out_row.p, d_perm.p, n * sizeof(uint32_t), cudaMemcpyDeviceToDevice, stream));
  }
  TargetSet ts;
  ts.m = n;
  ts.x = d_sx.p;
  ts.y = d_sy.p;
  ts.z = d_sz.p;
  ts.out_row = d_src_out_row.p;
  ts.leaf_begin = d_src_tl_begin.p;
  ts.leaf_end = d_src_tl_end.p;
  ts.tile_leaf = d_src_tile_leaf.p;
  ts.tile_off = d_src_tile_off.p;
  ts.n_tiles_dev = d_src_ntiles.p;
  ts.max_tiles = src_tiles;
  ts.cell_flag = d_flag_all.p;
  ts.all_sources = true;
  ts.own_lo = 0;
  ts.own_hi = (int)n;
  ts.row_of_pos = d_src_out_row.p;
  return ts;
}

// targets = all sources: X is the transpose of W, so the P2L kernel applies the M2P half as well
void fb_tree::evaluate_sources_fused(const TargetSet &ts) {
  const bool fuse = ht.adaptive && n_x_cells > 0 && ts.row_of_pos != nullptr;
  if (!(fuse && overlap_p2p && !m2l_groups.empty())) {
    downward(ts.cell_flag, fuse ? &ts : nullptr);
    leaf_pass(ts, false, fuse);
    return;
  }
  // Experiment (FB_OVERLAP=1): P2P needs only the sorted weights; M2L runs on the FP64 tensor pipe, P2P on the FP64
  // FMA pipe, so the P2P kernel goes to a low-priority side stream and shares the SMs with M2L; its results and the
  // fused M2P half are added with REDs, L2P joins last.  Result on B200: M2L at one CTA per SM (needed to leave
  // registers for the P2P CTAs) slows from 2.9 to 4.8 ms and P2P then competes with the W/X pass for the FMA pipe:
  // 15.1 ms against 13.6 ms for the serial order, so the serial order stays the default.
  d_out.zero(ts.m * (size_t)nrhs, stream);
  FB_CUDA(cudaEventRecord(ev_fork, stream));
  FB_CUDA(cudaStreamWaitEvent(stream2, ev_fork, 0));
  if (timing) FB_CUDA(cudaEventRecord(ev[10], stream2));
  launch_p2p(ts, false, true, stream2, true);
  if (timing) FB_CUDA(cudaEventRecord(ev[11], stream2));
  FB_CUDA(cudaEventRecord(ev_join, stream2));
  downward(ts.cell_flag, &ts, true, true);
  FB_CUDA(cudaStreamWaitEvent(stream, ev_join, 0));
  if (timing) FB_CUDA(cudaEventRecord(ev[7], stream));
  launch_l2p(ts, false);
  if (timing) {
    FB_CUDA(cudaEventRecord(ev[8], stream));
    FB_CUDA(cudaEventRecord(ev[9], stream));
  }
  last_overlapped = true;
}

// shared tail of bin_targets / subset_target_set: keys (leaf slot or sorted source position) -> TargetSet
TargetSet fb_tree::finish_target_set(TargetBuffers &tb, size_t m, int key_bits, bool keys_are_positions) {
  fb_tree &t = *this;
  const int nl = (int)t.ht.leaves.size();
  size_t cub_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, tb.key.p, tb.key2.p, tb.val.p, tb.val2.p, (int)m, 0, key_bits,
                                  t.stream);
  size_t scan_bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, tb.tile_cnt.p, tb.tile_cnt.p, nl, t.stream);
  t.d_cub.reserve(std::max(cub_bytes, scan_bytes));
  FB_CUDA(cub::DeviceRadixSort::SortPairs(t.d_cub.p, cub_bytes, tb.key.p, tb.key2.p, tb.val.p, tb.val2.p, (int)m, 0,
                                          key_bits, t.stream));
  g_launches.fetch_add(3);
  tb.tl_begin.reserve(nl);
  tb.tl_end.reserve(nl);
  tb.tile_cnt.reserve(2 * (size_t)nl);
  FB_LAUNCH(k_leaf_ranges, nblocks(nl, 128), 128, 0, t.stream, tb.key2.p, m,
            keys_are_positions ? t.d_src_tl_begin.p : nullptr, keys_are_positions ? t.d_src_tl_end.p : nullptr, nl,
            tb.tl_begin.p, tb.tl_end.p, tb.tile_cnt.p);
  int *scan_out = tb.tile_cnt.p + nl;
  FB_CUDA(cub::DeviceScan::ExclusiveSum(t.d_cub.p, scan_bytes, tb.tile_cnt.p, scan_out, nl, t.stream));
  g_launches.fetch_add(1);
  const int max_tiles = (int)std::min<size_t>((m + kTile - 1) / kTile + (size_t)nl, m);
  tb.tile_leaf.reserve(max_tiles);
  tb.tile_off.reserve(max_tiles);
  tb.ntiles.reserve(1);
  FB_LAUNCH(k_fill_tiles, nblocks(nl, 128), 128, 0, t.stream, scan_out, tb.tile_cnt.p, nl, tb.tile_leaf.p,
            tb.tile_off.p, tb.ntiles.p);
  tb.flag.reserve(t.ht.ncells());
  FB_CUDA(cudaMemsetAsync(tb.flag.p, 0, t.ht.ncells(), t.stream));
  FB_LAUNCH(k_flag_cells, nblocks(nl, 128), 128, 0, t.stream, t.d_leaf_cell.p, tb.tl_begin.p, tb.tl_end.p, nl,
            t.d_cell_parent.p, tb.flag.p);
  TargetSet ts;
  ts.m = m;
  ts.x = tb.tx.p;
  ts.y = tb.ty.p;
  ts.z = tb.tz.p;
  ts.out_row = tb.val2.p;
  ts.leaf_begin = tb.tl_begin.p;
  ts.leaf_end = tb.tl_end.p;
  ts.tile_leaf = tb.tile_leaf.p;
  ts.tile_off = tb.tile_off.p;
  ts.n_tiles_dev = tb.ntiles.p;
  ts.max_tiles = max_tiles;
  ts.cell_flag = tb.flag.p;
  return ts;
}

static int bits_for(size_t v) {
  int b = 1;
  while (b < 32 && (1ull << b) <= v) ++b;
  return b;
}

TargetSet fb_tree::bin_targets(const double *targets, size_t m, ptrdiff_t rs, ptrdiff_t cs, uint64_t *bad) {
  FB_REQUIRE(targets != nullptr && m > 0, "target_points must be a non-empty m x dim matrix");
  FB_REQUIRE(m < (1ull << 31), "at most 2^31-1 targets per call");
  const int nl = (int)ht.leaves.size();
  // targets bit-identical to the source points, in the same order (what ferreus_rbf's solver passes on every
  // matvec, rbf.rs:1357-1364): compared on the host, nothing is uploaded or binned
  if (m == n && cs == 1 && rs == (ptrdiff_t)dim && same_bytes(targets, host_points.data(), n * dim * sizeof(double)))
    return source_target_set();
  d_t_user.reserve(m * dim);
  if (cs == 1 && rs == (ptrdiff_t)dim) {
    FB_CUDA(cudaMemcpyAsync(d_t_user.p, targets, m * dim * sizeof(double), cudaMemcpyHostToDevice, stream));
  } else {
    h_stage.reserve(m * dim);
    for (size_t i = 0; i < m; ++i)
      for (int d = 0; d < dim; ++d) h_stage.p[i * dim + d] = targets[(ptrdiff_t)i * rs + (ptrdiff_t)d * cs];
    FB_CUDA(cudaMemcpyAsync(d_t_user.p, h_stage.p, m * dim * sizeof(double), cudaMemcpyHostToDevice, stream));
  }
  TargetBuffers &tb = tb_scratch;
  tb.key.reserve(m);
  tb.key2.reserve(m);
  tb.val.reserve(m);
  tb.val2.reserve(m);
  tb.tx.reserve(m);
  tb.ty.reserve(m);
  tb.tz.reserve(m);
  d_err.reserve(2);  // [0] first target outside the tree, [1] != 0 when the targets differ from the source points
  FB_CUDA(cudaMemsetAsync(d_err.p, 0xFF, sizeof(unsigned long long), stream));
  FB_CUDA(cudaMemsetAsync(d_err.p + 1, 0, sizeof(unsigned long long), stream));
  const bool maybe_sources = m == n && d_pts_user.cap >= n * (size_t)dim;
  if (maybe_sources)
    FB_LAUNCH(k_points_differ, nblocks(n * dim, 256), 256, 0, stream, d_t_user.p, d_pts_user.p, n * (size_t)dim,
              d_err.p + 1);
  const double side_depth = 2.0 * ht.radius / (double)(1ull << ht.depth);  // linear_tree.rs:495
  FB_LAUNCH(k_target_leaf, nblocks(m, 256), 256, 0, stream, d_t_user.p, m, dim, ht.depth, ht.disp[0], ht.disp[1],
            ht.disp[2], side_depth, d_leaf_lo.p, d_leaf_hi.p, nl, tb.key.p, tb.val.p, d_err.p);
  unsigned long long h_flags[2] = {0, 0};
  FB_CUDA(cudaMemcpyAsync(h_flags, d_err.p, sizeof(h_flags), cudaMemcpyDeviceToHost, stream));
  FB_CUDA(cudaStreamSynchronize(stream));
  const unsigned long long h_err = h_flags[0];
  // targets bit-identical to the source points, in the same order (what ferreus_rbf's solver passes on every
  // matvec, rbf.rs:1357-1364): reuse the source binning; evaluate() can then run the fused W/X pass
  if (maybe_sources && h_flags[1] == 0 && h_err == ~0ull) return source_target_set();
  if (h_err != ~0ull) {
    if (bad) *bad = h_err;
    throw Error(FB_ERR_POINT_OUTSIDE_TREE,
                "FMM evaluation failed: target point at row " + std::to_string(h_err) +
                    " lies outside the tree extents",
                h_err);
  }
  TargetSet ts = finish_target_set(tb, m, bits_for((size_t)nl), false);
  FB_LAUNCH(k_gather_targets, nblocks(m, 256), 256, 0, stream, d_t_user.p, tb.val2.p, m, dim, tb.tx.p, tb.ty.p,
            tb.tz.p);
  return ts;
}

TargetSet fb_tree::subset_target_set(const uint64_t *idx, size_t m) {
  FB_REQUIRE(idx != nullptr && m > 0 && m < (1ull << 31), "index list must be non-empty");
  d_idx64.reserve(m);
  FB_CUDA(cudaMemcpyAsync(d_idx64.p, idx, m * sizeof(uint64_t), cudaMemcpyHostToDevice, stream));
  return subset_target_set_dev(d_idx64.p, m, tb_scratch);
}

TargetSet fb_tree::subset_target_set_dev(const unsigned long long *d_idx, size_t m, TargetBuffers &tb) {
  tb.key.reserve(m);
  tb.key2.reserve(m);
  tb.val.reserve(m);
  tb.val2.reserve(m);
  tb.tx.reserve(m);
  tb.ty.reserve(m);
  tb.tz.reserve(m);
  d_err.reserve(1);
  FB_CUDA(cudaMemsetAsync(d_err.p, 0xFF, sizeof(unsigned long long), stream));
  FB_LAUNCH(k_subset_positions, nblocks(m, 256), 256, 0, stream, d_idx, d_inv.p, m, n, tb.key.p, tb.val.p, d_err.p);
  unsigned long long h_err = 0;
  FB_CUDA(cudaMemcpyAsync(&h_err, d_err.p, sizeof(h_err), cudaMemcpyDeviceToHost, stream));
  FB_CUDA(cudaStreamSynchronize(stream));
  FB_REQUIRE(h_err == ~0ull, "source index out of range at position " + std::to_string(h_err));
  TargetSet ts = finish_target_set(tb, m, bits_for(n), true);
  FB_LAUNCH(k_gather_coords, nblocks(m, 256), 256, 0, stream, d_sx.p, d_sy.p, d_sz.p, tb.key2.p, m, tb.tx.p, tb.ty.p,
            tb.tz.p);
  // sorted position -> output row map and target counts (fused W/X pass); a subset that names a source twice keeps
  // the separate M2P / P2L kernels
  tb.row_of_pos.reserve(n);
  tb.tgt_prefix.reserve(n + 1);
  tb.dup.reserve(1);
  FB_CUDA(cudaMemsetAsync(tb.row_of_pos.p, 0xFF, n * sizeof(uint32_t), stream));
  FB_CUDA(cudaMemsetAsync(tb.dup.p, 0, sizeof(unsigned long long), stream));
  FB_LAUNCH(k_subset_row_map, nblocks(m, 256), 256, 0, stream, tb.key2.p, tb.val2.p, m, tb.row_of_pos.p, tb.dup.p);
  size_t scan_bytes = 0;
  RowIsTarget is_target;
  auto flags_in = thrust::make_transform_iterator(tb.row_of_pos.p, is_target);
  cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, flags_in, tb.tgt_prefix.p, (int)n, stream);
  d_cub.reserve(scan_bytes);
  // n + 1 outputs: scan the n flags and append the total
  FB_CUDA(cub::DeviceScan::ExclusiveSum(d_cub.p, scan_bytes, flags_in, tb.tgt_prefix.p, (int)n, stream));
  FB_LAUNCH(k_prefix_total, 1, 1, 0, stream, tb.tgt_prefix.p, tb.row_of_pos.p, n);
  g_launches.fetch_add(1);
  unsigned long long h_dup = 0;
  FB_CUDA(cudaMemcpyAsync(&h_dup, tb.dup.p, sizeof(h_dup), cudaMemcpyDeviceToHost, stream));
  FB_CUDA(cudaStreamSynchronize(stream));
  if (h_dup == 0) {
    ts.row_of_pos = tb.row_of_pos.p;
    ts.tgt_prefix = tb.tgt_prefix.p;
  }
  return ts;
}

// weights already in d_w_user: upward pass, downward pass restricted to the target set, leaf pass -> d_out.
// The near-field pass (U lists) needs the sorted weights and nothing else: it is forked to the low-priority side stream
// right away, so the upward pass — P2M plus one small, latency-bound M2M launch per level — runs beside it instead of in
// front of it; the high-priority main stream's CTAs are placed ahead of the P2P kernel's pending ones.  Every writer of
// the result rows adds with REDs until the two streams join in front of L2P.  On one GPU the whole matvec is bound by
// the one FP64 pipe, so this only moves work around (measured 9.96 against 10.03 ms at the 1M-point headline) and it
// blurs the per-stage times: opt-in with FB_NEAR_OVERLAP=1.  A rank's share of a partitioned tree (comm.cu), where the
// upward pass is latency-bound and an all-reduce follows it, always runs this way.
void fb_tree::matvec_dev(const TargetSet &ts) {
  static const bool serial = [] {
    const char *v = std::getenv("FB_NEAR_OVERLAP");
    return !(v && v[0] == '1');
  }();
  sort_weights();
  if (serial) {
    upward();
    evaluate_sources_fused(ts);
    return;
  }
  const bool fuse = ht.adaptive && n_x_cells > 0 && ts.row_of_pos != nullptr;
  d_out.zero(ts.m * (size_t)nrhs, stream);  // in front of the fork: both streams add into it
  FB_CUDA(cudaEventRecord(ev_fork, stream));
  FB_CUDA(cudaStreamWaitEvent(stream2, ev_fork, 0));
  if (timing) FB_CUDA(cudaEventRecord(ev[10], stream2));
  launch_p2p(ts, false, true, stream2, true);  // U lists only
  if (timing) FB_CUDA(cudaEventRecord(ev[11], stream2));
  FB_CUDA(cudaEventRecord(ev_join, stream2));
  upward();
  downward(ts.cell_flag, fuse ? &ts : nullptr, true);
  FB_CUDA(cudaStreamWaitEvent(stream, ev_join, 0));
  if (timing) FB_CUDA(cudaEventRecord(ev[7], stream));
  launch_l2p(ts, false);
  if (timing) FB_CUDA(cudaEventRecord(ev[8], stream));
  if (!fuse && n_w_entries > 0) launch_p2p(ts, false, false, stream, false, true);  // W lists on their own
  if (timing) FB_CUDA(cudaEventRecord(ev[9], stream));
  last_overlapped = true;
}

void fb_tree::fetch_output(size_t m, bool grads, double *out_vals, double *out_grads, ptrdiff_t o_rs,
                           ptrdiff_t o_cs) {
  auto is_pinned = [](const void *p) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
      cudaGetLastError();
      return false;
    }
    return at.type == cudaMemoryTypeHost;
  };
  auto fetch = [&](const double *dsrc, size_t cols, double *dst) {
    const size_t cnt = m * cols;
    if (o_cs == 1 && o_rs == (ptrdiff_t)cols && cnt >= (1u << 14) && is_pinned(dst)) {  // fb_host_alloc'ed result
      FB_CUDA(cudaMemcpyAsync(dst, dsrc, cnt * sizeof(double), cudaMemcpyDeviceToHost, stream));
      FB_CUDA(cudaStreamSynchronize(stream));
    } else if (o_cs == 1 && o_rs == (ptrdiff_t)cols) {  // device -> pinned staging -> user buffer (all host threads)
      h_stage.reserve(cnt);
      FB_CUDA(cudaMemcpyAsync(h_stage.p, dsrc, cnt * sizeof(double), cudaMemcpyDeviceToHost, stream));
      FB_CUDA(cudaStreamSynchronize(stream));
      copy_bytes(dst, h_stage.p, cnt * sizeof(double));
    } else {
      h_stage.reserve(cnt);
      FB_CUDA(cudaMemcpyAsync(h_stage.p, dsrc, cnt * sizeof(double), cudaMemcpyDeviceToHost, stream));
      FB_CUDA(cudaStreamSynchronize(stream));
      // strides describe the value matrix (m x nrhs); gradients use o_rs * dim, o_cs (same orientation)
      const ptrdiff_t rs = (cols == (size_t)nrhs) ? o_rs : (o_cs == 1 ? (ptrdiff_t)cols : 1);
      const ptrdiff_t cs2 = (cols == (size_t)nrhs) ? o_cs : (o_cs == 1 ? 1 : (ptrdiff_t)m);
      for (size_t i = 0; i < m; ++i)
        for (size_t c = 0; c < cols; ++c) dst[(ptrdiff_t)i * rs + (ptrdiff_t)c * cs2] = h_stage.p[i * cols + c];
    }
  };
  fetch(d_out.p, (size_t)nrhs, out_vals);
  if (grads && out_grads) {
    if (o_cs == 1 && o_rs == (ptrdiff_t)nrhs) {  // row-major values => row-major gradients
      FB_CUDA(cudaMemcpyAsync(out_grads, d_gout.p, m * (size_t)nrhs * dim * sizeof(double), cudaMemcpyDeviceToHost,
                              stream));
      FB_CUDA(cudaStreamSynchronize(stream));
    } else {
      fetch(d_gout.p, (size_t)nrhs * dim, out_grads);
    }
  }
}

// ------------------------------------------------------------------------------------------ C ABI
template <class F>
static int guarded(F &&f, uint64_t *bad = nullptr) {
  try {
    f();
    return FB_OK;
  } catch (const fb::Error &e) {
    set_last_error(e.what());
    if (bad && e.code == FB_ERR_POINT_OUTSIDE_TREE) *bad = e.index;
    return e.code;
  } catch (const std::exception &e) {
    set_last_error(e.what());
    return FB_ERR_CUDA;
  }
}

static void collect_timing(fb_tree *t) {
  if (!t->timing) return;
  auto ms = [&](int a, int b) {
    float v = 0;
    cudaEventElapsedTime(&v, t->ev[a], t->ev[b]);
    return (double)v;
  };
  t->last_ms[0] = ms(0, 1);  // p2m
  t->last_ms[1] = ms(1, 2);  // m2m
  t->last_ms[2] = ms(3, 4);  // m2l
  t->last_ms[3] = ms(4, 5);  // p2l
  t->last_ms[4] = ms(5, 6);  // l2l
  t->last_ms[5] = ms(7, 8);  // l2p
  t->last_ms[6] = t->last_overlapped ? ms(10, 11) : ms(8, 9);  // p2p (+ m2p); overlapped: its own span on the side stream
  t->last_ms[7] = ms(0, 9);  // total
}

extern "C" {

const char *fb_last_error(void) { return t_last_error.c_str(); }
uint64_t fb_kernel_launch_count(void) { return g_launches.load(); }
int fb_set_sqrt_mode(int fast) {
  g_sqrt_mode.store(fast == 3 ? 3 : (fast ? 1 : 0));
  return FB_OK;
}
int fb_get_sqrt_mode(void) { return g_sqrt_mode.load(); }
uint64_t fb_trim_memory(void) { return (uint64_t)fb::dev_cache_trim(); }
int fb_set_device(int device) {
  return guarded([&] { FB_CUDA(cudaSetDevice(device)); });
}
void *fb_host_alloc(size_t bytes) {
  void *p = nullptr;
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}
void fb_host_free(void *p) {
  if (p) cudaFreeHost(p);
}

int fb_tree_new(const double *points, size_t n, int dim, ptrdiff_t row_stride, ptrdiff_t col_stride,
                int interpolation_order, const fb_kernel_params *kernel, int adaptive_tree, int sparse,
                const double *extents_or_null, const fb_fmm_params *params_or_null, fb_tree **out) {
  if (!out) return FB_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  fb_tree *t = nullptr;
  const int rc = guarded([&] {
    t = new fb_tree();
    t->build(points, n, dim, row_stride, col_stride, interpolation_order, kernel, adaptive_tree, sparse,
             extents_or_null, params_or_null);
  });
  if (rc != FB_OK) {
    delete t;
    return rc;
  }
  *out = t;
  return FB_OK;
}

void fb_tree_free(fb_tree *t) {
  if (!t) return;
  cudaSetDevice(t->device);
  cudaStreamSynchronize(t->stream);
  delete t;
}

int fb_tree_set_weights(fb_tree *t, const double *w, size_t n_rows, size_t nrhs, ptrdiff_t rs, ptrdiff_t cs) {
  return guarded([&] {
    FB_REQUIRE(t, "null tree");
    FB_CUDA(cudaSetDevice(t->device));
    t->upload_weights(w, n_rows, nrhs, rs, cs);
    t->upward();
    // no synchronisation here: the weights were copied out of the caller's memory above, and the transfer + upward pass
    // (0.5 ms at 1M points) run under the host-side work of the evaluate call that follows (target recognition);
    // every call that hands results back synchronises the stream
  });
}

int fb_tree_set_local_coefficients(fb_tree *t, const double *w, size_t n_rows, size_t nrhs, ptrdiff_t rs,
                                   ptrdiff_t cs) {
  return guarded([&] {
    FB_REQUIRE(t, "null tree");
    FB_CUDA(cudaSetDevice(t->device));
    FB_REQUIRE(t->have_weights, "set_weights must be called before set_local_coefficients");
    FB_REQUIRE((int)nrhs == t->nrhs, "weights must have the column count given to set_weights");
    const int keep = t->nrhs;
    t->upload_weights(w, n_rows, nrhs, rs, cs);
    t->nrhs = keep;
    t->downward(t->d_flag_all.p);
    FB_CUDA(cudaStreamSynchronize(t->stream));
  });
}

static int eval_common(fb_tree *t, const double *w, size_t n_rows, size_t nrhs, ptrdiff_t w_rs, ptrdiff_t w_cs,
                       const double *targets, size_t m, ptrdiff_t t_rs, ptrdiff_t t_cs, double *out_vals,
                       double *out_grads, ptrdiff_t o_rs, ptrdiff_t o_cs, uint64_t *bad, bool leaves_only) {
  return guarded(
      [&] {
        FB_REQUIRE(t, "null tree");
        FB_CUDA(cudaSetDevice(t->device));
        FB_REQUIRE(out_vals, "output buffer required");
        FB_REQUIRE(t->have_weights, "set_weights must be called before evaluate");
        FB_REQUIRE((int)nrhs == t->nrhs, "weights must have the column count given to set_weights");
        if (leaves_only) FB_REQUIRE(t->have_locals, "set_local_coefficients must be called before evaluate_leaves");
        // The solver's call (rbf.rs:1357-1364) hands over the vector it has just given to set_weights and the source
        // points themselves, every time; both facts are established by comparing the caller's buffers with the library's
        // copies on the host — 32 MB of memcmp at 1M points, longer than the upward pass it used to hide behind.  When
        // the same two pointers arrive as in the last call that was confirmed to be that case, the device work is queued
        // BEFORE the comparisons; if one of them fails after all, the call simply continues on the general path below
        // (same stream: the speculative kernels finish first and their results are overwritten).
        bool speculated = false;
        if (!leaves_only && out_grads == nullptr && targets != nullptr && targets == t->spec_targets && w == t->last_w_ptr &&
            m == t->n && t_cs == 1 && t_rs == (ptrdiff_t)t->dim && w_cs == 1 && w_rs == (ptrdiff_t)nrhs && t->w_cache_valid) {
          t->evaluate_sources_fused(t->source_target_set());
          speculated = true;
        }
        TargetSet ts = t->bin_targets(targets, m, t_rs, t_cs, bad);  // before touching weights: errors leave state intact
        const bool reuploaded = t->upload_weights(w, n_rows, nrhs, w_rs, w_cs);
        const bool solver_call = ts.all_sources && !leaves_only && out_grads == nullptr;
        t->spec_targets = (solver_call && !reuploaded) ? targets : nullptr;
        if (speculated && solver_call && !reuploaded) {
          // confirmed: the queued pass is the answer
        } else if (solver_call) {
          t->evaluate_sources_fused(ts);
        } else {
          if (!leaves_only) t->downward(ts.cell_flag);
          t->leaf_pass(ts, out_grads != nullptr);
        }
        t->fetch_output(m, out_grads != nullptr, out_vals, out_grads, o_rs, o_cs);
      },
      bad);
}

int fb_tree_evaluate(fb_tree *t, const double *w, size_t n_rows, size_t nrhs, ptrdiff_t w_rs, ptrdiff_t w_cs,
                     const double *targets, size_t m, ptrdiff_t t_rs, ptrdiff_t t_cs, double *out_vals,
                     double *out_grads_or_null, ptrdiff_t o_rs, ptrdiff_t o_cs, uint64_t *bad_index) {
  return eval_common(t, w, n_rows, nrhs, w_rs, w_cs, targets, m, t_rs, t_cs, out_vals, out_grads_or_null, o_rs, o_cs,
                     bad_index, false);
}

int fb_tree_evaluate_leaves(fb_tree *t, const double *w, size_t n_rows, size_t nrhs, ptrdiff_t w_rs, ptrdiff_t w_cs,
                            const double *targets, size_t m, ptrdiff_t t_rs, ptrdiff_t t_cs, double *out_vals,
                            double *out_grads_or_null, ptrdiff_t o_rs, ptrdiff_t o_cs, uint64_t *bad_index) {
  return eval_common(t, w, n_rows, nrhs, w_rs, w_cs, targets, m, t_rs, t_cs, out_vals, out_grads_or_null, o_rs, o_cs,
                     bad_index, true);
}

int fb_tree_evaluate_at_sources(fb_tree *t, const double *w, size_t n_rows, size_t nrhs, ptrdiff_t w_rs,
                                ptrdiff_t w_cs, const uint64_t *idx_or_null, size_t n_idx, double *out_vals,
                                ptrdiff_t o_rs, ptrdiff_t o_cs) {
  return guarded([&] {
    FB_REQUIRE(t, "null tree");
    FB_CUDA(cudaSetDevice(t->device));
    FB_REQUIRE(out_vals, "output buffer required");
    FB_REQUIRE(t->have_weights, "set_weights must be called before evaluate");
    FB_REQUIRE((int)nrhs == t->nrhs, "weights must have the column count given to set_weights");
    TargetSet ts = idx_or_null ? t->subset_target_set(idx_or_null, n_idx) : t->source_target_set();
    t->upload_weights(w, n_rows, nrhs, w_rs, w_cs);
    t->evaluate_sources_fused(ts);
    t->fetch_output(ts.m, false, out_vals, nullptr, o_rs, o_cs);
  });
}

int fb_tree_upload_weights(fb_tree *t, const double *w, size_t n_rows, size_t nrhs, ptrdiff_t rs, ptrdiff_t cs) {
  return guarded([&] {
    FB_REQUIRE(t, "null tree");
    FB_CUDA(cudaSetDevice(t->device));
    t->upload_weights(w, n_rows, nrhs, rs, cs);
    FB_CUDA(cudaStreamSynchronize(t->stream));
  });
}

int fb_tree_matvec_resident(fb_tree *t) {
  return guarded([&] {
    FB_REQUIRE(t, "null tree");
    FB_CUDA(cudaSetDevice(t->device));
    FB_REQUIRE(t->d_w_user.cap >= t->n * (size_t)t->nrhs, "fb_tree_upload_weights must be called first");
    FB_CUDA(cudaEventRecord(t->ev_mv[0], t->stream));
    TargetSet ts = t->have_subset ? t->ts_subset : t->source_target_set();
    t->matvec_dev(ts);
    t->last_out_rows = ts.m;
    FB_CUDA(cudaEventRecord(t->ev_mv[1], t->stream));
    FB_CUDA(cudaStreamSynchronize(t->stream));
    float mv_ms = 0;
    FB_CUDA(cudaEventElapsedTime(&mv_ms, t->ev_mv[0], t->ev_mv[1]));
    t->last_matvec_ms = mv_ms;
    collect_timing(t);
  });
}

int fb_tree_download_result(fb_tree *t, double *out_vals, ptrdiff_t o_rs, ptrdiff_t o_cs) {
  return guarded([&] {
    FB_REQUIRE(t && out_vals, "null argument");
    FB_CUDA(cudaSetDevice(t->device));
    t->fetch_output(t->have_subset ? t->ts_subset.m : t->n, false, out_vals, nullptr, o_rs, o_cs);
  });
}

int fb_tree_leaf_work(const fb_tree *t, uint64_t *leaf_ptr, double *work) {
  if (!t) return FB_ERR_INVALID_ARGUMENT;
  const fb::HostTree &ht = t->ht;
  const size_t nl = ht.leaves.size();
  // M2L entries of every cell, accumulated down the tree so a leaf carries its ancestors' share
  std::vector<double> v_share(ht.ncells(), 0.0);
  for (size_t c = 1; c < ht.ncells(); ++c) {
    const double own = (double)(ht.v_ptr[c + 1] - ht.v_ptr[c]) * 4.0 * 24.0 * t->P;  // ~4 r P flops per entry
    const int nch = std::max(1, ht.child_ptr[c + 1] - ht.child_ptr[c]);
    v_share[c] += own;
    for (int k = ht.child_ptr[c]; k < ht.child_ptr[c + 1]; ++k) v_share[ht.child_idx[k]] += v_share[c] / nch;
  }
  for (size_t l = 0; l < nl; ++l) {
    const int c = ht.leaves[l];
    if (leaf_ptr) leaf_ptr[l] = (uint64_t)ht.pt_begin[c];
    if (work) {
      const double nt = ht.pt_end[c] - ht.pt_begin[c];
      double nsrc = 0;
      for (long long e = ht.u_ptr[c]; e < ht.u_ptr[c + 1]; ++e) nsrc += ht.pt_end[ht.u_idx[e]] - ht.pt_begin[ht.u_idx[e]];
      const double nw = (double)(ht.w_ptr[c + 1] - ht.w_ptr[c]);
      double nx = 0;
      for (long long e = ht.x_ptr[c]; e < ht.x_ptr[c + 1]; ++e) nx += ht.pt_end[ht.x_idx[e]] - ht.pt_begin[ht.x_idx[e]];
      work[l] = 12.0 * (nt * (nsrc + nw * t->P) + nx * t->P) + v_share[c] + 1.0;
    }
  }
  if (leaf_ptr) leaf_ptr[nl] = (uint64_t)t->n;
  return FB_OK;
}

int fb_tree_morton_order(const fb_tree *t, uint64_t *order) {
  if (!t || !order) return FB_ERR_INVALID_ARGUMENT;
  return guarded([&] {
    std::vector<uint32_t> perm(t->n);
    FB_CUDA(cudaSetDevice(t->device));
    FB_CUDA(cudaMemcpy(perm.data(), t->d_perm.p, t->n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < t->n; ++i) order[i] = perm[i];
  });
}

int fb_tree_set_target_subset(fb_tree *t, const uint64_t *idx, size_t n_idx) {
  return guarded([&] {
    FB_REQUIRE(t, "null tree");
    FB_CUDA(cudaSetDevice(t->device));
    if (n_idx == 0 || idx == nullptr) {
      t->have_subset = false;
      return;
    }
    FB_REQUIRE(n_idx < (1ull << 31), "subset too large");
    t->d_subset_idx.reserve(n_idx);
    FB_CUDA(cudaMemcpyAsync(t->d_subset_idx.p, idx, n_idx * sizeof(uint64_t), cudaMemcpyHostToDevice, t->stream));
    t->ts_subset = t->subset_target_set_dev(t->d_subset_idx.p, n_idx, t->tb_subset);
    FB_CUDA(cudaStreamSynchronize(t->stream));
    t->have_subset = true;
  });
}

int fb_tree_result_device(fb_tree *t, const double **dev_ptr, uint64_t *n_rows, uint64_t *n_cols) {
  if (!t || !dev_ptr) return FB_ERR_INVALID_ARGUMENT;
  *dev_ptr = t->d_out.p;
  if (n_rows) *n_rows = t->last_out_rows;
  if (n_cols) *n_cols = (uint64_t)t->nrhs;
  return FB_OK;
}

int fb_tree_last_matvec_ms(fb_tree *t, double *ms_out) {
  if (!t || !ms_out) return FB_ERR_INVALID_ARGUMENT;
  *ms_out = t->last_matvec_ms;
  return FB_OK;
}

// FP64 FMA-pipe peak of the current device: 16 independent DFMA chains per thread, CUDA-event timed
__global__ void k_dfma_peak(double *out, int iters, double a, double b) {
  double x[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) x[i] = (double)(threadIdx.x + i) * 1e-3;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 16; ++i) x[i] = fma(x[i], a, b);
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += x[i];
  if (s == 12345.678) out[0] = s;
}

int fb_measure_fp64_tflops(double *tflops_out) {
  return guarded([&] {
    FB_REQUIRE(tflops_out, "null argument");
    int dev = 0, sms = 0;
    FB_CUDA(cudaGetDevice(&dev));
    FB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    fb::DBuf<double> out;
    out.reserve(1);
    cudaEvent_t e0, e1;
    FB_CUDA(cudaEventCreate(&e0));
    FB_CUDA(cudaEventCreate(&e1));
    const int iters = 16384, blocks = sms * 8, threads = 256;
    double best = 0;
    for (int rep = 0; rep < 8; ++rep) {  // the first repetitions also bring the clocks up
      FB_CUDA(cudaEventRecord(e0, 0));
      FB_LAUNCH(k_dfma_peak, blocks, threads, 0, 0, out.p, iters, 0.999999, 1e-9);
      FB_CUDA(cudaEventRecord(e1, 0));
      FB_CUDA(cudaEventSynchronize(e1));
      float ms = 0;
      FB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
      const double fl = 2.0 * 16.0 * iters * (double)blocks * threads;
      if (rep >= 2) best = std::max(best, fl / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *tflops_out = best;
  });
}

// algorithmic FLOPs of one M2L pass per right-hand side (SURVEY.md 8(d)): sum over the V-list entries of 4 r P for the
// compressed operators (2 P^2 uncompressed), r the rank of the entry's (level, reference vector) operator
int fb_tree_m2l_flops(const fb_tree *t, double *flops_out) {
  if (!t || !flops_out) return FB_ERR_INVALID_ARGUMENT;
  const fb::HostTree &ht = t->ht;
  const bool compressed = t->fparams.compression_type != FB_COMPRESSION_NONE;
  double fl = 0.0;
  for (int lvl = 2; lvl <= ht.depth; ++lvl)
    for (int c = ht.level_ptr[lvl]; c < ht.level_ptr[lvl + 1]; ++c) {
      uint32_t ac[3];
      ht.anchor(c, ac);
      for (long long e = ht.v_ptr[c]; e < ht.v_ptr[c + 1]; ++e) {
        uint32_t as[3];
        ht.anchor(ht.v_idx[e], as);
        int tix = 0;
        for (int d = 0; d < t->dim; ++d) tix = tix * 7 + ((int)ac[d] - (int)as[d] + 3);
        const int r = t->ops.m2l[lvl - 2][t->ops.ref_lookup[tix]].rank;
        fl += compressed ? 4.0 * r * t->P : 2.0 * (double)t->P * t->P;
      }
    }
  *flops_out = fl;
  return FB_OK;
}

// FP64 tensor-instruction peak of the current device (mma.sync m8n8k4, 6 independent chains per warp)
__global__ void k_dmma_peak(double *out, int iters) {
  double c[6][2];
#pragma unroll
  for (int i = 0; i < 6; ++i) c[i][0] = c[i][1] = 0.0;
  const double a = threadIdx.x * 1e-3, b = threadIdx.x * 2e-3;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 6; ++i)
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                   : "+d"(c[i][0]), "+d"(c[i][1])
                   : "d"(a), "d"(b));
  }
  double s = 0;
#pragma unroll
  for (int i = 0; i < 6; ++i) s += c[i][0] + c[i][1];
  if (s == 12345.678) out[0] = s;
}

int fb_measure_fp64_dmma_tflops(double *tflops_out) {
  return guarded([&] {
    FB_REQUIRE(tflops_out, "null argument");
    int dev = 0, sms = 0;
    FB_CUDA(cudaGetDevice(&dev));
    FB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    fb::DBuf<double> out;
    out.reserve(1);
    cudaEvent_t e0, e1;
    FB_CUDA(cudaEventCreate(&e0));
    FB_CUDA(cudaEventCreate(&e1));
    const int iters = 16384, blocks = sms * 4, threads = 256;
    double best = 0;
    for (int rep = 0; rep < 8; ++rep) {  // the first repetitions also bring the clocks up
      FB_CUDA(cudaEventRecord(e0, 0));
      FB_LAUNCH(k_dmma_peak, blocks, threads, 0, 0, out.p, iters);
      FB_CUDA(cudaEventRecord(e1, 0));
      FB_CUDA(cudaEventSynchronize(e1));
      float ms = 0;
      FB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
      const double fl = 512.0 * 6.0 * iters * (double)blocks * (threads / 32);
      if (rep >= 2) best = std::max(best, fl / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *tflops_out = best;
  });
}

int fb_tree_set_timing(fb_tree *t, int enabled) {
  if (!t) return FB_ERR_INVALID_ARGUMENT;
  t->timing = enabled != 0;
  return FB_OK;
}

int fb_tree_last_timing(fb_tree *t, double *ms_out8) {
  if (!t || !ms_out8) return FB_ERR_INVALID_ARGUMENT;
  for (int i = 0; i < 8; ++i) ms_out8[i] = t->last_ms[i];
  return FB_OK;
}

int fb_tree_source_points(const fb_tree *t, double *out, ptrdiff_t row_stride, ptrdiff_t col_stride) {
  if (!t || !out) return FB_ERR_INVALID_ARGUMENT;
  for (size_t i = 0; i < t->n; ++i)
    for (int d = 0; d < t->dim; ++d)
      out[(ptrdiff_t)i * row_stride + (ptrdiff_t)d * col_stride] = t->host_points[i * t->dim + d];
  return FB_OK;
}

int fb_tree_get_info(const fb_tree *t, fb_tree_info *info) {
  if (!t || !info) return FB_ERR_INVALID_ARGUMENT;
  std::memset(info, 0, sizeof(*info));
  info->n_points = t->n;
  info->n_cells = t->ht.ncells();
  info->n_leaves = t->ht.leaves.size();
  info->depth = (uint64_t)t->ht.depth;
  info->n_u = t->ht.u_idx.size();
  info->n_v = t->ht.v_idx.size();
  info->n_w = t->ht.w_idx.size();
  info->n_x = t->ht.x_idx.size();
  info->dim = t->dim;
  info->order = t->order;
  info->nrhs = t->nrhs;
  info->radius = t->ht.radius;
  for (int d = 0; d < 3; ++d) info->center[d] = t->ht.center[d];
  info->p2p_pairs = t->p2p_pairs;
  info->m2p_pairs = t->m2p_pairs;
  info->p2l_pairs = t->p2l_pairs;
  return FB_OK;
}

int fb_tree_dump_cells(const fb_tree *t, uint64_t *keys, uint8_t *leaf_flags, uint64_t *leaf_ptr,
                       uint64_t *leaf_idx) {
  if (!t) return FB_ERR_INVALID_ARGUMENT;
  return guarded([&] {
    const size_t nc = t->ht.ncells();
    std::vector<uint32_t> perm;
    if (leaf_idx) {
      perm.resize(t->n);
      FB_CUDA(cudaSetDevice(t->device));
      FB_CUDA(cudaMemcpy(perm.data(), t->d_perm.p, t->n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    }
    uint64_t off = 0;
    for (size_t c = 0; c < nc; ++c) {
      if (keys) keys[c] = t->ht.ref_key((int)c);
      if (leaf_flags) leaf_flags[c] = t->ht.is_leaf[c];
      if (leaf_ptr) leaf_ptr[c] = off;
      if (t->ht.is_leaf[c]) {
        const int b = t->ht.pt_begin[c], e = t->ht.pt_end[c];
        if (leaf_idx) {
          for (int i = b; i < e; ++i) leaf_idx[off + (i - b)] = perm[i];
          std::sort(leaf_idx + off, leaf_idx + off + (e - b));
        }
        off += (uint64_t)(e - b);
      }
    }
    if (leaf_ptr) leaf_ptr[nc] = off;
  });
}

int fb_tree_dump_list(const fb_tree *t, int which, uint64_t *ptr, uint64_t *idx) {
  if (!t || which < 0 || which > 3) return FB_ERR_INVALID_ARGUMENT;
  const std::vector<int64_t> *p[4] = {&t->ht.u_ptr, &t->ht.v_ptr, &t->ht.w_ptr, &t->ht.x_ptr};
  const std::vector<int32_t> *x[4] = {&t->ht.u_idx, &t->ht.v_idx, &t->ht.w_idx, &t->ht.x_idx};
  if (ptr)
    for (size_t i = 0; i < p[which]->size(); ++i) ptr[i] = (uint64_t)(*p[which])[i];
  if (idx)
    for (size_t i = 0; i < x[which]->size(); ++i) idx[i] = (uint64_t)(*x[which])[i];
  return FB_OK;
}

int fb_tree_m2l_rank(const fb_tree *t, int level, int ref) {
  if (!t || level < 2 || level > t->ht.depth || ref < 0 || ref >= t->ops.n_ref) return -1;
  return t->ops.m2l[level - 2][ref].rank;
}

int fb_m2l_stream_warps(int P, int compression) { return fb::m2l_stream_warps(P, compression); }

int fb_tree_m2l_stream_warps(const fb_tree *t) { return t ? fb::m2l_stream_plan_warps(t->m2l_plan) : 0; }

int fb_tree_m2l_operator(const fb_tree *t, int level, int ref, double *u_or_null, double *vt_or_null) {
  if (!t || level < 2 || level > t->ht.depth || ref < 0 || ref >= t->ops.n_ref) return FB_ERR_INVALID_ARGUMENT;
  const fb::M2LOperator &op = t->ops.m2l[level - 2][ref];
  if (u_or_null) std::copy(op.U.a.begin(), op.U.a.end(), u_or_null);
  if (vt_or_null) std::copy(op.Vt.a.begin(), op.Vt.a.end(), vt_or_null);
  return FB_OK;
}

struct fb_ops {
  fb::Operators ops;
};

int fb_ops_new(int interpolation_order, int dim, double radius, int depth, const fb_kernel_params *kernel,
               int compression_type, double epsilon, fb_ops **out) {
  if (!out || !kernel || dim < 1 || dim > 3 || interpolation_order < 1) return FB_ERR_INVALID_ARGUMENT;
  fb::KParams kp;
  if (!fb::make_kparams(*kernel, kp)) return FB_ERR_INVALID_ARGUMENT;
  fb_ops *o = new fb_ops();
  o->ops.build_cached(interpolation_order, dim, radius, depth, kp, compression_type, epsilon);
  *out = o;
  return FB_OK;
}
void fb_ops_free(fb_ops *o) { delete o; }
int fb_ops_rank(const fb_ops *o, int level, int ref) {
  if (!o || level < 2 || level - 2 >= (int)o->ops.m2l.size() || ref < 0 || ref >= o->ops.n_ref) return -1;
  return o->ops.m2l[level - 2][ref].rank;
}
int fb_ops_get(const fb_ops *o, int level, int ref, double *u_or_null, double *vt_or_null) {
  if (fb_ops_rank(o, level, ref) < 0) return FB_ERR_INVALID_ARGUMENT;
  const fb::M2LOperator &op = o->ops.m2l[level - 2][ref];
  if (u_or_null) std::copy(op.U.a.begin(), op.U.a.end(), u_or_null);
  if (vt_or_null) std::copy(op.Vt.a.begin(), op.Vt.a.end(), vt_or_null);
  return FB_OK;
}
int fb_ops_tables(const fb_ops *o, int32_t *n_perm, int32_t *n_ref, int32_t *perm, int32_t *inv_perm,
                  int32_t *perm_lookup, int32_t *ref_lookup, double *m2m_child_s) {
  if (!o) return FB_ERR_INVALID_ARGUMENT;
  if (n_perm) *n_perm = o->ops.n_perm;
  if (n_ref) *n_ref = o->ops.n_ref;
  if (perm) std::copy(o->ops.perm.begin(), o->ops.perm.end(), perm);
  if (inv_perm) std::copy(o->ops.inv_perm.begin(), o->ops.inv_perm.end(), inv_perm);
  if (perm_lookup) std::copy(o->ops.perm_lookup.begin(), o->ops.perm_lookup.end(), perm_lookup);
  if (ref_lookup) std::copy(o->ops.ref_lookup.begin(), o->ops.ref_lookup.end(), ref_lookup);
  if (m2m_child_s) std::copy(o->ops.child_s.begin(), o->ops.child_s.end(), m2m_child_s);
  return FB_OK;
}

}  // extern "C"
