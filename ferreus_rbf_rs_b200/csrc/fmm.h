// Internal declarations of the device-resident FMM evaluator (struct fb_tree) and its kernels.
#pragma once
#include <memory>

#include "common.h"
#include "host_ops.h"
#include "host_tree.h"
#include "kernel_functions.cuh"

namespace fb {

constexpr int kMaxOrder = 16;   // Chebyshev nodes per axis supported by the device kernels
constexpr int kTile = 128;      // targets per CTA in the direct-sum / L2P kernels
// Multipoles / locals are stored [cell][rhs][Ps]: P = p^d coefficients padded to an even count, so every column
// starts on a 16-byte boundary and its size is a multiple of 16 bytes (cp.async.bulk / cp.reduce.async.bulk in
// m2l.cu).  The pad element is zeroed with the array and never written.
__host__ __device__ __forceinline__ int coef_stride(int P) { return (P + 1) & ~1; }

// ---- a target set binned into the leaves of a tree (sorted by leaf, Morton order) -------------
struct TargetSet {
  size_t m = 0;              // number of targets
  const double *x = nullptr, *y = nullptr, *z = nullptr;  // sorted coordinates (unused dims are 0)
  const uint32_t *out_row = nullptr;                       // output row of each sorted target
  const int *leaf_begin = nullptr, *leaf_end = nullptr;    // per leaf slot: range in the sorted arrays
  const int *tile_leaf = nullptr, *tile_off = nullptr;     // CTA tiles of <= kTile targets
  const int *n_tiles_dev = nullptr;                        // device scalar: number of valid tiles
  int max_tiles = 0;                                       // launch bound for the tile grid
  bool all_sources = false;                                // the tree's own source set
  // targets = the sources at the sorted positions [own_lo, own_hi), in that order (target i = position own_lo + i): every
  // source, or the Morton-contiguous share of a rank (comm.cu: `out` then has a row for EVERY source and out_row /
  // row_of_pos name those global rows).  Enables the symmetric P2P (p2p_sym.cu); 0, 0 = neither
  int own_lo = 0, own_hi = 0;
  // targets that are source points (all of them, or a duplicate-free subset): enables the fused W/X pass
  const uint32_t *row_of_pos = nullptr;  // per sorted source position: output row, 0xFFFFFFFF when not a target
  const uint32_t *tgt_prefix = nullptr;  // n + 1 exclusive counts of targets over the sorted positions; null = all
  const uint8_t *cell_flag = nullptr;                      // per cell: subtree contains targets
  // symmetric P2P (p2p_sym.cu): the tiles in the order the kernel takes them, heaviest first; null = tile order
  const int *sym_tile_order = nullptr;
};

// device storage behind a TargetSet that is not the tree's own source set
struct TargetBuffers {
  DBuf<double> tx, ty, tz;
  DBuf<uint32_t> key, key2, val, val2;
  DBuf<int> tl_begin, tl_end, tile_leaf, tile_off, ntiles, tile_cnt;
  DBuf<uint8_t> flag;
  DBuf<uint32_t> row_of_pos, tgt_prefix;  // subset-of-sources sets only
  DBuf<unsigned long long> dup;
};

struct DirectArgs {  // leaf pass: P2P over U ranges + M2P over W cells (bbfmm.rs:1162-1355)
  TargetSet ts;
  const long long *u_ptr;
  const int *u_begin, *u_count;  // merged contiguous source ranges
  const long long *w_ptr;
  const int *w_cell;
  const double *sx, *sy, *sz, *w;  // sources (sorted) and weights [rhs][n]
  size_t n;
  const double *mult;  // multipoles [cell][rhs][P]
  const double *ccx, *ccy, *ccz, *chalf;
  const double *nodes;  // p Chebyshev nodes
  int p, dim, P, nrhs, rhs0;
  int nrhs_pass;   // symmetric P2P: right-hand sides [rhs0, rhs0 + nrhs_pass) of this call
  int atomic_out;  // 1: results are added with RED (the kernel runs concurrently with other writers of `out`)
  int has_w;       // 1: some leaf owns a W list that this call must apply (M2P)
  int skip_p2p;    // 1: the U ranges were served by another kernel (p2p_sym.cu / p2p_mma.cu)
  const uint32_t *sym_row;  // symmetric P2P: output row of EVERY sorted source position (null: kernel not applicable)
  double *out;    // [m][nrhs]
  double *gout;   // [m][nrhs*dim] or null
  KParams kp;
};

struct P2LArgs {  // bbfmm.rs:1001-1048
  const int *cells;  // cells that own a non-empty X list
  int n_cells;
  const long long *x_ptr;  // per entry of `cells`
  const int *x_begin, *x_count;
  const uint8_t *cell_flag;
  const double *sx, *sy, *sz, *w;
  size_t n;
  double *loc;  // locals [cell][rhs][P]
  const double *ccx, *ccy, *ccz, *chalf;
  const double *nodes;
  int p, dim, P, nrhs, rhs0;
  KParams kp;
  // fused M2P (non-null only when the targets are all sources): out[out_row[s]] += K(point s, nodes) . M_cell
  const double *mult;       // multipoles [cell][rhs][P]
  double *out;              // [n][nrhs]
  const uint32_t *out_row;  // output row of each sorted source position (0xFFFFFFFF: not a target)
  const uint32_t *tgt_prefix;  // n + 1 exclusive target counts over the sorted positions, or null (every source)
  // partitioned tree: the M2P half of a cell is applied by the rank that owns the cell's first point (sorted position
  // cell_ptb[c] in [own_lo, own_hi)), for all of the cell's X-list points — foreign rows travel in the result all-reduce
  const int *cell_ptb;
  int own_lo, own_hi;
};

// kernel family -> template argument
#define FB_FAM_SWITCH(fam, CALL)                         \
  switch (fam) {                                         \
    case KF_LINEAR: CALL(KF_LINEAR); break;              \
    case KF_TPS: CALL(KF_TPS); break;                    \
    case KF_CUBIC: CALL(KF_CUBIC); break;                \
    case KF_SPH: CALL(KF_SPH); break;                    \
    case KF_LAPLACE: CALL(KF_LAPLACE); break;            \
    case KF_R2: CALL(KF_R2); break;                      \
    default: CALL(KF_R4); break;                         \
  }

void launch_leaf_direct(const DirectArgs &a, cudaStream_t s);
bool p2p_sym_applicable(const DirectArgs &a);           // p2p_sym.cu
void launch_p2p_sym(const DirectArgs &a, cudaStream_t s);
bool p2p_mma_applicable(const DirectArgs &a);           // p2p_mma.cu (opt-in experiment)
void launch_p2p_mma(const DirectArgs &a, cudaStream_t s);
void launch_p2l(const P2LArgs &a, cudaStream_t s);
// transfers.cu: order / dimension templated P2M and L2P (values only); false = no instantiation, use the generic kernel
bool launch_p2m_fast(int n_leaves, const int *leaves, const int *ptb, const int *pte, const double *sx, const double *sy,
                     const double *sz, const double *w, size_t n, const double *ccx, const double *ccy,
                     const double *ccz, const double *chalf, const double *tnodes, int p, int dim, int nrhs,
                     double *mult, cudaStream_t s);
bool launch_l2p_fast(const TargetSet &ts, const int *leaf_cell, const double *loc, const double *ccx, const double *ccy,
                     const double *ccz, const double *chalf, const double *tnodes, int p, int dim, int nrhs,
                     double *out, cudaStream_t s);

// ---- device_io.cu: inputs and outputs in caller-owned device memory (the *_device entry points) -------------------
// FB_ERR_INVALID_ARGUMENT naming `what` unless the first and the last element of the rows x cols matrix at p (element
// strides rs, cs) lie in device memory of `device`
void require_device_matrix(const void *p, size_t rows, size_t cols, ptrdiff_t rs, ptrdiff_t cs, int device,
                           const char *what);
// Orders `own` (a handle's non-blocking stream) after the work queued so far on `caller`, and, in join() or when the
// object goes out of scope (a call that fails half way), `caller` after everything queued on `own` meanwhile.
struct StreamJoin {
  cudaStream_t caller, own;
  bool joined = false;
  StreamJoin(cudaStream_t caller_, cudaStream_t own_);
  void join();
  ~StreamJoin();
};
struct AffineMap {  // x' = [x 1] * a, a (dim+1) x (dim+1) row-major; on = 0: identity
  int on = 0;
  double a[16] = {0};
};
// rows x cols strided copy between device matrices, each row optionally mapped through `aff` (cols = dim)
void launch_copy_rows(const double *src, ptrdiff_t s_rs, ptrdiff_t s_cs, size_t rows, int cols, double *dst,
                      ptrdiff_t d_rs, ptrdiff_t d_cs, const AffineMap &aff, cudaStream_t s);
// [mins..., maxs...] over the rows of a strided m x dim device matrix; scratch is device memory for the partial
// results.  Blocks until the 2*dim values are on the host.
void device_extents(const double *x, size_t m, int dim, ptrdiff_t rs, ptrdiff_t cs, DBuf<double> &scratch,
                    cudaStream_t s, double *ext);
// finish of the interpolant (fr_model::eval_tree): one thread per (target, value column).  out / out_grads may be
// vals / grads (no pointer here is __restrict__)
struct RbfFinish {
  size_t m = 0;
  int dim = 0, n_cols = 0, basis = 0, degree = 0;
  const double *targets = nullptr;  // original coordinates
  ptrdiff_t t_rs = 0, t_cs = 0;
  const double *vals = nullptr, *grads = nullptr;  // leaf pass results [m][n_cols], [m][n_cols * dim] (null: none)
  const double *w = nullptr;                       // point coefficients [m][n_cols] when the nugget is added, else null
  double nugget = 0;
  const double *poly = nullptr;                    // basis x n_cols row-major
  double translation[3] = {0, 0, 0}, scale[3] = {1, 1, 1};
  AffineMap trend;                                 // gradients are mapped back through its linear part when on
  double *out = nullptr, *out_grads = nullptr;     // row-major, as fr_evaluate
};
void launch_rbf_finish(const RbfFinish &f, cudaStream_t s);

// ---- M2L work lists, one group per (level, reference vector) -----------------------------------
// m2l.cu: streaming M2L (TMA gathers / scatter-adds around register-resident operators); null plan = not applicable
struct M2LStreamPlan;
int m2l_stream_warps(int P, int compression);  // MMA warps of the streaming kernel for P, 0 = generic kernel
bool m2l_stream_supported(int P, int compression);  // the same, unless FB_M2L_STREAM=0 turns the stream off
int m2l_stream_plan_warps(const M2LStreamPlan *plan);  // MMA warps the plan launches with, 0 for no plan
M2LStreamPlan *m2l_stream_build(const HostTree &ht, const Operators &ops, int P, const int *d_inv_tab, cudaStream_t stream);
struct M2LItemTable;  // work items restricted to the cells [level_lo, level_hi) of every level (a rank's share)
M2LItemTable *m2l_stream_table_new(M2LStreamPlan *plan, int nrhs, const int *level_lo, const int *level_hi,
                                   cudaStream_t stream);
int m2l_stream_table_nrhs(const M2LItemTable *t);
void m2l_stream_table_free(M2LItemTable *t);
void m2l_stream_launch(M2LStreamPlan *plan, int nrhs, const uint8_t *flag_or_null, const M2LItemTable *table_or_null,
                       const double *mult, double *loc, cudaStream_t stream);
void m2l_stream_free(M2LStreamPlan *plan);

struct M2LGroup {
  int level, ref, rank, rank_pad;
  size_t n_entries;
  size_t entry_off;     // offset into the entry arrays
  size_t u_off, v_off;  // offsets (in doubles) into the operator pool
};

}  // namespace fb

struct fb_shard;  // comm.cu: partition of the tree across the ranks of an fb_comm
void fb_shard_free(fb_shard *s);

// The opaque C handle
struct fb_tree {
  int device = 0;
  cudaStream_t stream = nullptr;
  // low-priority side stream: the near field (P2P) of a rank's share of a partitioned tree, beside the upward pass,
  // the multipole all-reduce and the downward pass on `stream` (fb_tree_matvec_sharded)
  cudaStream_t stream2 = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  int dim = 3, order = 0, P = 0;
  size_t n = 0;
  int nrhs = 1;
  bool have_weights = false, have_locals = false;
  fb_kernel_params kparams_c{};
  fb::KParams kp{};
  fb_fmm_params fparams{};
  std::vector<double> host_points;  // n x dim row-major copy (source_points())
  fb::HostTree ht;
  fb::Operators ops;
  uint64_t p2p_pairs = 0, m2p_pairs = 0, p2l_pairs = 0;

  // --- device state
  fb::DBuf<double> d_sx, d_sy, d_sz;          // sorted source coordinates
  fb::DBuf<double> d_pts_user;                // source points as given (n x dim, row-major)
  fb::DBuf<uint32_t> d_perm, d_inv;           // sorted position -> source row, and inverse
  fb::DBuf<double> d_w;                       // weights, sorted, [rhs][n]
  fb::DBuf<double> d_w_user;                  // weights as uploaded [n][nrhs] row-major
  fb::PinnedBuf<double> h_w_last;             // pinned copy of the last contiguous upload (H2D source, duplicate test)
  size_t h_w_last_cnt = 0;
  bool w_cache_valid = false;                 // false once d_w_user was written on the device (solver)
  const double *last_w_ptr = nullptr;         // caller's pointer of the last contiguous upload (never dereferenced)
  const double *spec_targets = nullptr;       // caller's target pointer of the last evaluate confirmed to be the solver's call
  fb::DBuf<double> d_mult, d_loc;             // [cell][rhs][P]
  fb::DBuf<double> d_ccx, d_ccy, d_ccz, d_chalf;
  fb::DBuf<int> d_cell_parent, d_cell_slot, d_cell_ptb, d_cell_pte;
  fb::DBuf<int> d_child_ptr, d_child_idx;
  fb::DBuf<uint8_t> d_flag_all;               // per-cell "has targets" flags (all ones)
  fb::DBuf<int> d_leaf_cell;                  // leaf slot -> cell
  fb::DBuf<unsigned long long> d_leaf_lo, d_leaf_hi;  // level-16 code range of each leaf slot
  fb::DBuf<int> d_src_leaves;                 // cells of leaves that hold sources (P2M grid)
  std::vector<std::vector<int>> h_parents;    // per level: non-leaf cells
  fb::DBuf<int> d_parents;                    // concatenated, offsets in parents_off
  std::vector<int> parents_off;
  // lists
  fb::DBuf<long long> d_u_ptr, d_w_ptr, d_x_ptr, d_w_ptr_none;
  fb::DBuf<int> d_u_begin, d_u_count, d_w_cell, d_x_begin, d_x_count, d_x_cells;
  int n_x_cells = 0;
  long long n_w_entries = 0;
  int n_src_leaves = 0;
  // all-sources target set
  fb::DBuf<int> d_src_tl_begin, d_src_tl_end, d_src_tile_leaf, d_src_tile_off, d_src_ntiles;
  fb::DBuf<int> d_src_tile_order;  // the tiles by descending symmetric-P2P work (TargetSet::sym_tile_order)
  fb::DBuf<uint32_t> d_src_out_row;
  int src_tiles = 0;
  // general target set scratch
  fb::DBuf<double> d_t_user;
  fb::TargetBuffers tb_scratch;
  fb::TargetBuffers tb_subset;          // persistent subset for sharded matvecs
  fb::TargetSet ts_subset{};
  fb::DBuf<unsigned long long> d_subset_idx;
  bool have_subset = false;
  size_t last_out_rows = 0;
  fb::DBuf<unsigned long long> d_err;
  fb::DBuf<unsigned char> d_cub;
  fb::DBuf<unsigned long long> d_idx64;
  // outputs
  fb::DBuf<double> d_out, d_gout;
  fb::PinnedBuf<double> h_stage;
  // operators
  fb::DBuf<double> d_nodes, d_tnodes, d_child_s, d_oppool;
  fb::DBuf<int> d_perm_tab, d_inv_tab;
  // M2L
  std::vector<fb::M2LGroup> m2l_groups;
  fb::M2LStreamPlan *m2l_plan = nullptr;
  fb_shard *shard = nullptr;  // multi-GPU partition (fb_tree_shard), null = the whole tree on this device  // streaming kernel (m2l.cu) when applicable, else the grouped k_m2l below
  fb::DBuf<int> d_m2l_tgt, d_m2l_src, d_m2l_perm;
  int m2l_P4 = 0, m2l_Pp = 0;  // padded node counts of the M2L tiles
  size_t m2l_smem = 0;
  int m2l_nc = 32;  // (entry, rhs) columns per M2L CTA
  fb::DBuf<unsigned char> d_m2l_table;  // M2LGroupDev[] of the fused launch
  fb::DBuf<int> d_m2l_cta_group;        // group of every CTA of that launch
  int m2l_table_nrhs = -1;
  unsigned m2l_ctas = 0;
  // timing
  bool timing = false;
  double last_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  cudaEvent_t ev[12] = {};
  cudaEvent_t ev_mv[2] = {};
  double last_matvec_ms = 0;

  ~fb_tree();
  void build(const double *points, size_t n_, int dim_, ptrdiff_t rs, ptrdiff_t cs, int order_,
             const fb_kernel_params *k, int adaptive, int sparse, const double *extents,
             const fb_fmm_params *params);
  // returns false when `w` is byte-identical to the last upload (nothing sent)
  bool upload_weights(const double *w, size_t n_rows, size_t nrhs_, ptrdiff_t rs, ptrdiff_t cs);
  void sort_weights();
  // P2M over `leaves` (null = every leaf with sources) and M2M over the cells flagged in `cell_flag` (null = all)
  void upward(const int *leaves = nullptr, int n_leaves = 0, const uint8_t *cell_flag = nullptr);
  // fuse_m2p: the P2L kernel also applies the M2P transpose for that target set (ts.row_of_pos != null) into d_out
  // (zeroed here); leaf_pass(ts, false, m2p_done = true) must follow
  void downward(const uint8_t *flags, const fb::TargetSet *fuse_m2p = nullptr, bool out_zeroed = false,
                const fb::M2LItemTable *m2l_table = nullptr);
  void leaf_pass(const fb::TargetSet &ts, bool grads, bool m2p_done = false);
  void launch_l2p(const fb::TargetSet &ts, bool grads);
  // m2p_done: the W lists are (or will be) applied elsewhere; w_only: the U lists are
  void launch_p2p(const fb::TargetSet &ts, bool grads, bool m2p_done, cudaStream_t s, bool atomic_out,
                  bool w_only = false);
  void evaluate_sources_fused(const fb::TargetSet &ts);  // downward + leaf pass for targets that are source points
  fb::TargetSet source_target_set();
  fb::TargetSet bin_targets(const double *targets, size_t m, ptrdiff_t rs, ptrdiff_t cs, uint64_t *bad);
  // device_io.cu: targets in caller-owned device memory, mapped through the affine matrix `aff` ((dim+1) x (dim+1),
  // row-major, applied to homogeneous row vectors) when it is non-null
  fb::TargetSet bin_targets_dev(const double *d_targets, size_t m, ptrdiff_t rs, ptrdiff_t cs, const double *aff,
                                uint64_t *bad);
  // shared tail of bin_targets / bin_targets_dev: the m targets are in d_t_user (row-major); blocks the host until they
  // are binned (the outside-the-tree check reads d_err)
  fb::TargetSet bin_user_targets(size_t m, uint64_t *bad);
  // device_io.cu: weights in caller-owned device memory -> d_w_user, d_w (no upward pass)
  void upload_weights_dev(const double *d_w, size_t n_rows, size_t nrhs_, ptrdiff_t rs, ptrdiff_t cs);
  fb::TargetSet subset_target_set(const uint64_t *idx, size_t n_idx);
  // subset of the sources as targets, index list already on the device; storage owned by `tb`
  fb::TargetSet subset_target_set_dev(const unsigned long long *d_idx, size_t n_idx, fb::TargetBuffers &tb);
  fb::TargetSet finish_target_set(fb::TargetBuffers &tb, size_t m, int key_bits, bool keys_are_positions);
  // device-resident matvec pieces used by the solver (weights already in d_w_user, [n][nrhs])
  void matvec_dev(const fb::TargetSet &ts);
  void fetch_output(size_t m, bool grads, double *out_vals, double *out_grads, ptrdiff_t o_rs, ptrdiff_t o_cs);
};
