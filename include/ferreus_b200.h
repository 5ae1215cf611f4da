/*
 * ferreus_b200.h — C ABI of libferreus_b200.so (B200 / sm_100a implementation of the
 * ferreus_rbf_rs BBFMM matvec and the FGMRES + domain-decomposition RBF solve).
 *
 * Every entry point replaces one method of the reference's type-erased evaluator
 * `ferreus_rbf_utils::FmmTree` (ferreus_rbf_utils/src/utils.rs:383-493) or of
 * `ferreus_rbf::RBFInterpolator` (ferreus_rbf/src/rbf.rs:304-924).  Plain pointers and sizes
 * only; matrices are passed with element strides so faer column-major (`row_stride = 1,
 * col_stride = nrows`) and numpy row-major (`row_stride = ncols, col_stride = 1`) both pass
 * zero-copy.  All host pointers; the library owns all device memory.
 *
 * A handle is NOT thread-safe (same contract as `&mut self` in the reference); distinct
 * handles may be used concurrently.  No function aborts the process: errors are returned as
 * codes and `fb_last_error()` gives the message of the last failure on the calling thread.
 */
#ifndef FERREUS_B200_H
#define FERREUS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- error codes (reference: FmmError, ferreus_bbfmm/src/bbfmm.rs:20-45) ------------------ */
#define FB_OK 0
#define FB_ERR_POINT_OUTSIDE_TREE 1   /* FmmError::PointOutsideTree{point_index} -> *bad_index */
#define FB_ERR_NO_GRADIENTS 2         /* FmmError::KernelDoesNotSupportGradients (unreachable for built-ins) */
#define FB_ERR_INVALID_ARGUMENT 3     /* reference panics (bbfmm.rs:297, kernel_helpers.rs:72-73) */
#define FB_ERR_CUDA 4                 /* CUDA / NCCL failure, see fb_last_error() */

/* ---- kernel registry (ferreus_rbf_utils/src/utils.rs:558-571, same order) ------------------- */
enum fb_kernel_type {
  FB_KERNEL_LINEAR = 0,
  FB_KERNEL_THIN_PLATE_SPLINE = 1,
  FB_KERNEL_CUBIC = 2,
  FB_KERNEL_SPHEROIDAL3 = 3,
  FB_KERNEL_SPHEROIDAL5 = 4,
  FB_KERNEL_SPHEROIDAL7 = 5,
  FB_KERNEL_SPHEROIDAL9 = 6,
  FB_KERNEL_LAPLACIAN = 7,
  FB_KERNEL_ONE_OVER_R2 = 8,
  FB_KERNEL_ONE_OVER_R4 = 9
};

/* KernelParams (ferreus_rbf_utils/src/kernel_helpers.rs:17-36) */
typedef struct fb_kernel_params {
  int32_t kernel_type; /* enum fb_kernel_type */
  double base_range;   /* > 0 */
  double total_sill;   /* <= base_range */
} fb_kernel_params;

/* M2LCompressionType (ferreus_bbfmm/src/bbfmm.rs:62-73) */
enum fb_compression_type { FB_COMPRESSION_NONE = 0, FB_COMPRESSION_SVD = 1, FB_COMPRESSION_ACA = 2 };

/* FmmParams (ferreus_bbfmm/src/bbfmm.rs:77-104); NULL => new_defaults(order): 256, ACA, 10^-order, 1024 */
typedef struct fb_fmm_params {
  uint64_t max_points_per_cell;
  int32_t compression_type; /* enum fb_compression_type */
  double epsilon;
  uint64_t eval_chunk_size; /* accepted for API compatibility; affects memory only in the reference */
} fb_fmm_params;

typedef struct fb_tree fb_tree; /* opaque: replaces ferreus_rbf_utils::FmmTree */

const char *fb_last_error(void);
/* number of CUDA kernels launched by this library on the calling process so far (bench accounting) */
uint64_t fb_kernel_launch_count(void);
/* CUDA device used by handles created afterwards on this thread (default: current device) */
int fb_set_device(int device);
/* Page-locked host memory for result buffers (optional).  Every entry point accepts ordinary pageable memory; when an
 * output pointer lies in memory obtained here the device -> host copy lands in it directly (no staging copy, no page
 * faults of a freshly mapped buffer).  The reference returns freshly allocated matrices (bbfmm.rs:444-507); a binding
 * can back them with these blocks.  fb_host_alloc returns NULL on failure.                                         */
void *fb_host_alloc(size_t bytes);
void fb_host_free(void *p);
/* Square-root mode of the direct-sum hot loops (P2P, M2P, P2L) for trees and models built AFTER the call:
 * 1 = second-order refinement of the hardware seed (default): relative error <= 1.3e-12 per kernel value (measured,
 *     tools/fp64_ubench.cu), two FP64 operations fewer per pair; 0 = third-order refinement, ~1 ulp.  Both keep the
 *     parity gates (matvec <= 1e-10, interpolant <= 1e-8).  The environment variable FB_SQRT=exact|fast sets the
 *     initial value.  3 = mode 1 plus an experiment: squared distances of the P2P sums (linear, cubic, spheroidal
 *     kernels) from the FP64 tensor cores (csrc/p2p_mma.cu; measured 4 % faster only, not the default).            */
int fb_set_sqrt_mode(int fast);
int fb_get_sqrt_mode(void);
/* Device memory released by trees / models is cached for the next allocation of a similar size (repeated fits do not
 * pay cudaMalloc / cudaFree again); fb_trim_memory hands the cache back to the driver and returns the bytes released.
 * FB_NO_MEMORY_CACHE=1 in the environment disables the cache.                                                        */
uint64_t fb_trim_memory(void);

/* FmmTree::new  (ferreus_rbf_utils/src/utils.rs:392-421 -> ferreus_bbfmm/src/bbfmm.rs:272-353).
 * points: n x dim (dim 1..3).  extents: NULL or [mins..., maxs...] (2*dim doubles).            */
int fb_tree_new(const double *points, size_t n, int dim, ptrdiff_t row_stride, ptrdiff_t col_stride,
                int interpolation_order, const fb_kernel_params *kernel, int adaptive_tree, int sparse,
                const double *extents_or_null, const fb_fmm_params *params_or_null, fb_tree **out);
void fb_tree_free(fb_tree *t);

/* FmmTree::set_weights (bbfmm.rs:383-401): upward pass P2M + M2M; only the first n rows are read.  The weights are
 * copied before the call returns; the transfer and the upward pass are only enqueued (they overlap the host-side work
 * of the next call), so a device failure in them is reported by the next call on this handle.                    */
int fb_tree_set_weights(fb_tree *t, const double *w, size_t n_rows, size_t nrhs, ptrdiff_t row_stride,
                        ptrdiff_t col_stride);
/* FmmTree::set_local_coefficients (bbfmm.rs:518-524): full downward pass. */
int fb_tree_set_local_coefficients(fb_tree *t, const double *w, size_t n_rows, size_t nrhs,
                                   ptrdiff_t row_stride, ptrdiff_t col_stride);

/* FmmTree::evaluate / evaluate_with_gradients (bbfmm.rs:411-507).
 * out_vals: m x nrhs, out_grads (NULL => values only): m x (nrhs*dim), columns
 * [rhs0_dx, rhs0_dy, rhs0_dz, rhs1_dx, ...]; both with the given output strides.
 * On FB_ERR_POINT_OUTSIDE_TREE *bad_index is the first offending target row.                  */
int fb_tree_evaluate(fb_tree *t, const double *w, size_t n_rows, size_t nrhs, ptrdiff_t w_rs, ptrdiff_t w_cs,
                     const double *targets, size_t m, ptrdiff_t t_rs, ptrdiff_t t_cs, double *out_vals,
                     double *out_grads_or_null, ptrdiff_t o_rs, ptrdiff_t o_cs, uint64_t *bad_index);
/* FmmTree::evaluate_leaves / evaluate_leaves_with_gradients (bbfmm.rs:537-616): leaf pass only. */
int fb_tree_evaluate_leaves(fb_tree *t, const double *w, size_t n_rows, size_t nrhs, ptrdiff_t w_rs,
                            ptrdiff_t w_cs, const double *targets, size_t m, ptrdiff_t t_rs, ptrdiff_t t_cs,
                            double *out_vals, double *out_grads_or_null, ptrdiff_t o_rs, ptrdiff_t o_cs,
                            uint64_t *bad_index);
/* Extension used by the solver: identical to evaluate(w, source_points[idx]) (the call made by
 * fast_matrix_vector_product, ferreus_rbf/src/rbf.rs:1357-1364) but skips re-binning targets that
 * are source points.  idx NULL => all sources in order.  out: n_idx x nrhs.                   */
int fb_tree_evaluate_at_sources(fb_tree *t, const double *w, size_t n_rows, size_t nrhs, ptrdiff_t w_rs,
                                ptrdiff_t w_cs, const uint64_t *idx_or_null, size_t n_idx, double *out_vals,
                                ptrdiff_t o_rs, ptrdiff_t o_cs);
/* One matvec = set_weights + evaluate at all sources with w and the result kept resident in HBM
 * (the timed region of the headline metric without host<->device copies).  Inputs must have been
 * uploaded with fb_tree_upload_weights; result fetched with fb_tree_download_result.           */
int fb_tree_upload_weights(fb_tree *t, const double *w, size_t n_rows, size_t nrhs, ptrdiff_t rs, ptrdiff_t cs);
int fb_tree_matvec_resident(fb_tree *t);
int fb_tree_download_result(fb_tree *t, double *out_vals, ptrdiff_t o_rs, ptrdiff_t o_cs);
/* per-pass device time (ms, CUDA events) of the last fb_tree_matvec_resident call when timing is
 * enabled with fb_tree_set_timing(t, 1).  names: p2m m2m m2l p2l l2l l2p p2p_m2p total          */
int fb_tree_set_timing(fb_tree *t, int enabled);
/* algorithmic FLOPs of one M2L pass per right-hand side: sum over V-list entries of 4 r P (2 P^2 uncompressed) */
int fb_tree_m2l_flops(const fb_tree *t, double *flops_out);
/* FP64 peak of the tensor instruction (mma.sync m8n8k4) next to fb_measure_fp64_tflops (DFMA): same datapath on B200 */
int fb_measure_fp64_dmma_tflops(double *tflops_out);
/* device time (ms, CUDA events on the handle's stream) of the last fb_tree_matvec_resident call */
int fb_tree_last_matvec_ms(fb_tree *t, double *ms_out);
/* FP64 FMA-pipe peak of the current device (TFLOP/s): in-run DFMA micro-benchmark, CUDA-event timed */
int fb_measure_fp64_tflops(double *tflops_out);
int fb_tree_last_timing(fb_tree *t, double *ms_out8);

/* FmmTree::source_points (utils.rs:486-492): n x dim copy with the given strides. */
int fb_tree_source_points(const fb_tree *t, double *out, ptrdiff_t row_stride, ptrdiff_t col_stride);

/* ---- introspection for the bit-exact tree gate (not in the reference API) ------------------- */
typedef struct fb_tree_info {
  uint64_t n_points, n_cells, n_leaves, depth;
  uint64_t n_u, n_v, n_w, n_x; /* total entries of each interaction list */
  int32_t dim, order, nrhs;
  double radius;
  double center[3];
  uint64_t p2p_pairs, m2p_pairs, p2l_pairs; /* sum n_t*n_s over U / n_t over (leaf,W) / n_s over (cell,X) */
} fb_tree_info;
int fb_tree_get_info(const fb_tree *t, fb_tree_info *info);
/* keys: n_cells reference-format Morton keys ((interleave<<15)|level, morton.rs:58-119), level-major;
 * leaf_flags: n_cells (1 = leaf); leaf_ptr: n_cells+1, leaf_idx: n_points (source rows of each cell in
 * ascending order, non-leaf cells have empty ranges).  Any pointer may be NULL.                 */
int fb_tree_dump_cells(const fb_tree *t, uint64_t *keys, uint8_t *leaf_flags, uint64_t *leaf_ptr,
                       uint64_t *leaf_idx);
/* which: 0=U 1=V 2=W 3=X.  ptr: n_cells+1, idx: total entries (cell indices into keys[]). */
int fb_tree_dump_list(const fb_tree *t, int which, uint64_t *ptr, uint64_t *idx);
/* rank of the compressed M2L operator for (level 2..depth, reference vector 0..n_ref-1); -1 if absent */
int fb_tree_m2l_rank(const fb_tree *t, int level, int ref);
/* dense copy of U (P x rank, column-major) / Vt (rank x P, column-major) */
int fb_tree_m2l_operator(const fb_tree *t, int level, int ref, double *u_or_null, double *vt_or_null);
/* which M2L kernel serves P = order^dim nodes per cell (host only): the number of MMA warps of the streaming kernel
 * (csrc/m2l.cu), or 0 when the generic kernel does (uncompressed operators, or P outside the streaming windows).
 * The environment variable FB_M2L_STREAM=0, read when a tree is built, is not consulted here.                    */
int fb_m2l_stream_warps(int P, int compression_type);
/* the same for a built tree: the MMA warps of the streaming plan it holds, 0 when it runs the generic kernel (its P
 * is not served, FB_M2L_STREAM=0 at build time, depth < 2, or no V-list entries)                                  */
int fb_tree_m2l_stream_warps(const fb_tree *t);


/* ---- multi-GPU sharding by Morton-contiguous leaf ranges (SURVEY.md §8e) ---------------------------------
 * The tree is replicated on every rank; a rank evaluates only the targets of its own contiguous range of
 * leaves.  fb_tree_leaf_work returns the leaves in Morton order with an estimate of their evaluation work
 * (direct pairs + M2L entries of the leaf and its ancestors), fb_tree_morton_order the source rows in that
 * order; fb_tree_set_target_subset makes fb_tree_matvec_resident evaluate at that subset only (n_idx = 0
 * restores all sources) and fb_tree_result_device exposes the device result buffer (rows in subset order) so it
 * can be handed to NCCL without a host round trip.                                                          */
int fb_tree_leaf_work(const fb_tree *t, uint64_t *leaf_ptr /* n_leaves+1 */, double *work /* n_leaves */);
int fb_tree_morton_order(const fb_tree *t, uint64_t *order /* n_points */);
int fb_tree_set_target_subset(fb_tree *t, const uint64_t *idx, size_t n_idx);
int fb_tree_result_device(fb_tree *t, const double **dev_ptr, uint64_t *n_rows, uint64_t *n_cols);

/* ---- NCCL partition (csrc/comm.cu): one process per GPU, the reference's rayon loops (bbfmm.rs:669, 682, 788, 841,
 * 1122) split across devices.  Every rank builds the same tree from the same points and calls fb_tree_shard with its
 * communicator: the Morton leaf sequence is cut into world_size contiguous ranges of nearly equal estimated work, a rank
 * owns the points of its range.  fb_tree_matvec_sharded then runs P2M / M2M over the owned part, completes the
 * multipoles with ncclAllReduce (under the near-field pass), runs M2L / L2L / L2P for the owned cells / targets, the
 * symmetric P2P for the owned chunks and the fused P2L + M2P pass for the owned cells (every kernel evaluation of the
 * unpartitioned matvec is made by exactly one rank; symmetric halves that belong to foreign rows are added into the
 * rank's full-length partial result) and ncclAllReduce's that result: the full A w, in the caller's row order,
 * replicated, stays in device memory (fb_tree_sharded_result_device) or is copied out (fb_tree_sharded_download).
 * Weights: all N rows, uploaded with fb_tree_upload_weights on every rank (before fb_tree_shard: the work model of the
 * cut depends on the number of right-hand sides).  NCCL is dlopen'ed on first use.                                    */
typedef struct fb_comm fb_comm;
int fb_comm_unique_id(uint8_t *id_out128);                       /* rank 0; broadcast the 128 bytes out of band   */
int fb_comm_init(const uint8_t *id128, int rank, int world_size, fb_comm **out);  /* on the current device        */
void fb_comm_free(fb_comm *c);
int fb_comm_rank(const fb_comm *c);
int fb_comm_world_size(const fb_comm *c);
int fb_tree_shard(fb_tree *t, fb_comm *comm_or_null);            /* NULL drops the partition                      */
/* profiling / test aid: with a world-1 communicator, take the share rank `rank` of `world` ranks would own — the per-rank
 * kernel times of an N-GPU partition on one GPU.  The collectives degenerate to copies: exact = 0 forms the owned
 * multipoles only (faithful times, partial sums in the result), exact = 1 forms all of them (owned rows exact)       */
int fb_tree_shard_as(fb_tree *t, fb_comm *comm, int rank, int world, int exact);
/* where the near-field pass forks off: 0 = after the weight sort (beside the upward pass, exchange 1 and the downward
 * pass), 1 = after the upward pass (beside exchange 1 and the downward pass).  fb_tree_shard picks one from the      *
 * estimated length of the near field; this call overrides it                                                      */
int fb_tree_shard_fork_mode(fb_tree *t, int mode);
int fb_tree_shard_rows(const fb_tree *t, int rank, uint64_t *begin_pos, uint64_t *end_pos);  /* Morton positions  */
int fb_tree_matvec_sharded(fb_tree *t);
int fb_tree_sharded_timing(const fb_tree *t, double *ms_out4);   /* upward pass + multipole all-reduce, downward pass (near field beside both), rest of the near field + L2P, result all-reduce */
int fb_tree_sharded_result_device(const fb_tree *t, const double **dev_ptr);
int fb_tree_sharded_download(fb_tree *t, double *out_vals /* n x nrhs row-major */);
/* the cut itself (host only): n_parts + 1 boundaries into the leaf sequence */
int fb_partition_by_work(const double *work, size_t n_leaves, int parts, uint64_t *bounds_out);

/* ---- host-only tree + interaction lists (no GPU needed): the HostTree the device path builds (morton.rs:29-373,
 * linear_tree.rs:20-485), from level-16 codes computed and sorted on the host instead of by the device radix sort; used
 * by the CPU test-suite to compare keys, leaf membership and the U / V / W / X lists with the oracle bit for bit.
 * dump_* have the layouts of fb_tree_dump_cells / fb_tree_dump_list.                                            ---- */
typedef struct fb_host_tree fb_host_tree;
int fb_host_tree_new(const double *points, size_t n, int dim, ptrdiff_t row_stride, ptrdiff_t col_stride,
                     const double *extents_or_null, uint64_t max_points_per_cell, int adaptive_tree, int sparse,
                     fb_host_tree **out);
void fb_host_tree_free(fb_host_tree *t);
int fb_host_tree_counts(const fb_host_tree *t, uint64_t *n_cells, uint64_t *n_leaves, int32_t *depth,
                        uint64_t *n_list4 /* U, V, W, X entries */);
int fb_host_tree_dump_cells(const fb_host_tree *t, uint64_t *keys, uint8_t *leaf_flags, uint64_t *leaf_ptr,
                            uint64_t *leaf_idx);
int fb_host_tree_dump_list(const fb_host_tree *t, int which, uint64_t *ptr, uint64_t *idx);

/* ---- host-only operator precompute (no GPU needed): used by the CPU test-suite to check the
 * Chebyshev / ACA / SVD restatement (chebyshev.rs:650-814, aca.rs:23-247) against the oracle. ---- */
typedef struct fb_ops fb_ops;
int fb_ops_new(int interpolation_order, int dim, double radius, int depth, const fb_kernel_params *kernel,
               int compression_type, double epsilon, fb_ops **out);
void fb_ops_free(fb_ops *o);
int fb_ops_rank(const fb_ops *o, int level, int ref);
/* u: P x rank column-major, vt: rank x P column-major (vt untouched when uncompressed) */
int fb_ops_get(const fb_ops *o, int level, int ref, double *u_or_null, double *vt_or_null);
/* tables: perm / inv_perm are n_perm x P (row-major), lookups have 7^dim entries; any pointer may be NULL */
int fb_ops_tables(const fb_ops *o, int32_t *n_perm, int32_t *n_ref, int32_t *perm, int32_t *inv_perm,
                  int32_t *perm_lookup, int32_t *ref_lookup, double *m2m_child_s);

#ifdef __cplusplus
}
#endif
#endif /* FERREUS_B200_H */
