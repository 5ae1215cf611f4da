// Evaluation with inputs and outputs in caller-owned device memory: the *_device entry points of
// include/ferreus_b200.h (FmmTree) and the kernels behind them and behind every interpolant evaluation
// (fr_model::eval_tree, solver.cu).  Targets and weights are gathered from the caller's strides on the device,
// then the host path takes over unchanged from the binning (fb_tree::bin_user_targets) or the weight sort on; results
// go back to the caller's memory with one more kernel or a device-to-device copy.  Nothing crosses the PCIe bus but the
// outside-the-tree flag (and, for the one-shot interpolant, the 2 * dim extents).
#include "fmm.h"
#include "monomials.h"

#include <algorithm>

namespace fb {

static inline unsigned nblocks(size_t n, int bs) { return (unsigned)((n + bs - 1) / bs); }

void require_device_matrix(const void *p, size_t rows, size_t cols, ptrdiff_t rs, ptrdiff_t cs, int device,
                           const char *what) {
  FB_REQUIRE(p != nullptr && rows > 0 && cols > 0, std::string(what) + " must be a non-empty device matrix");
  // the elements at the smallest and the largest offset the strides reach
  ptrdiff_t lo = 0, hi = 0;
  const ptrdiff_t span[2] = {(ptrdiff_t)(rows - 1) * rs, (ptrdiff_t)(cols - 1) * cs};
  for (ptrdiff_t s : span) (s < 0 ? lo : hi) += s;
  for (ptrdiff_t off : {lo, hi}) {
    cudaPointerAttributes at{};
    const cudaError_t e = cudaPointerGetAttributes(&at, static_cast<const double *>(p) + off);
    if (e != cudaSuccess) cudaGetLastError();
    FB_REQUIRE(e == cudaSuccess && at.type == cudaMemoryTypeDevice && at.device == device,
               std::string(what) + " must be device memory of CUDA device " + std::to_string(device));
  }
}

StreamJoin::StreamJoin(cudaStream_t caller_, cudaStream_t own_) : caller(caller_), own(own_) {
  cudaEvent_t ev;
  FB_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  const cudaError_t e1 = cudaEventRecord(ev, caller);
  const cudaError_t e2 = e1 == cudaSuccess ? cudaStreamWaitEvent(own, ev, 0) : e1;
  cudaEventDestroy(ev);  // released once the wait has been satisfied
  if (e2 != cudaSuccess) {
    joined = true;  // nothing was queued on `own` for the caller to wait for
    FB_CUDA(e2);
  }
}

void StreamJoin::join() {
  if (joined) return;
  joined = true;
  cudaEvent_t ev;
  FB_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  const cudaError_t e1 = cudaEventRecord(ev, own);
  const cudaError_t e2 = e1 == cudaSuccess ? cudaStreamWaitEvent(caller, ev, 0) : e1;
  cudaEventDestroy(ev);
  FB_CUDA(e2);
}

StreamJoin::~StreamJoin() {
  try {
    join();
  } catch (...) {  // the error that unwound the call is the one reported
  }
}

// ------------------------------------------------------------------------------------------ kernels
// Row i of src (strides s_rs, s_cs) -> row i of dst (d_rs, d_cs); with aff.on the row is the homogeneous vector
// [x 1] times aff.a, bit for bit as fr_model::apply_affine (solver.cu) computes it on the host (same order, every
// product and sum rounded on its own; the host compiles with -ffp-contract=off).  With a global trend,
// evaluate_at_source relies on it: the mapped source points must equal the tree's kernel-space points for
// bin_user_targets to recognise them.
__global__ void k_copy_rows(const double *__restrict__ src, ptrdiff_t s_rs, ptrdiff_t s_cs, size_t rows, int cols,
                            double *__restrict__ dst, ptrdiff_t d_rs, ptrdiff_t d_cs, AffineMap aff) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= rows) return;
  const double *s = src + (ptrdiff_t)i * s_rs;
  double *d = dst + (ptrdiff_t)i * d_rs;
  if (!aff.on) {
    for (int c = 0; c < cols; ++c) d[(ptrdiff_t)c * d_cs] = s[(ptrdiff_t)c * s_cs];
    return;
  }
  const int h = cols + 1;
  double x[4] = {0, 0, 0, 1.0};
  for (int k = 0; k < cols; ++k) x[k] = s[(ptrdiff_t)k * s_cs];
  x[cols] = 1.0;
  for (int j = 0; j < cols; ++j) {
    double v = 0.0;
    for (int k = 0; k < h; ++k) v = __dadd_rn(v, __dmul_rn(x[k], aff.a[k * h + j]));
    d[(ptrdiff_t)j * d_cs] = v;
  }
}

constexpr int kExtBlocks = 256, kExtThreads = 256;

// per block: [mins..., maxs...] of its grid-stride share of the rows (min / max as std::min / std::max compare)
__global__ void __launch_bounds__(kExtThreads) k_extents_partial(const double *__restrict__ x, size_t m, int dim,
                                                                 ptrdiff_t rs, ptrdiff_t cs, double *part) {
  __shared__ double s_lo[kExtThreads], s_hi[kExtThreads];
  for (int d = 0; d < dim; ++d) {
    double lo = x[(ptrdiff_t)d * cs], hi = lo;  // row 0: a valid start for every thread
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < m; i += (size_t)gridDim.x * blockDim.x) {
      const double v = x[(ptrdiff_t)i * rs + (ptrdiff_t)d * cs];
      lo = v < lo ? v : lo;
      hi = hi < v ? v : hi;
    }
    s_lo[threadIdx.x] = lo;
    s_hi[threadIdx.x] = hi;
    __syncthreads();
    for (int w = blockDim.x / 2; w > 0; w >>= 1) {
      if ((int)threadIdx.x < w) {
        const double a = s_lo[threadIdx.x + w], b = s_hi[threadIdx.x + w];
        s_lo[threadIdx.x] = a < s_lo[threadIdx.x] ? a : s_lo[threadIdx.x];
        s_hi[threadIdx.x] = s_hi[threadIdx.x] < b ? b : s_hi[threadIdx.x];
      }
      __syncthreads();
    }
    if (threadIdx.x == 0) {
      part[(size_t)blockIdx.x * 2 * dim + d] = s_lo[0];
      part[(size_t)blockIdx.x * 2 * dim + dim + d] = s_hi[0];
    }
    __syncthreads();
  }
}

__global__ void k_extents_final(const double *part, int n_parts, int dim, double *ext) {
  const int j = threadIdx.x;  // 0 .. 2*dim-1: mins, then maxs
  if (j >= 2 * dim) return;
  double v = part[j];
  for (int b = 1; b < n_parts; ++b) {
    const double u = part[(size_t)b * 2 * dim + j];
    v = j < dim ? (u < v ? u : v) : (v < u ? u : v);
  }
  ext[j] = v;
}

// The per-target finish of fr_model::eval_tree (solver.cu), one thread per (target, value column), every product and
// sum rounded on its own:
//   1. kernel gradient mapped back through the trend, g <- g B^T;
//   2. + nugget * w[i][c] when w is given (evaluate_at_source(add_nugget)), before the drift;
//   3. + sum_k mono_k(x) poly[k][c] on the original coordinates (monomial_row, monomials.h);
//   4. + the drift gradient (degree 1 and 2, evaluate_monomial_gradients);
//   5. stored row-major.
// Each thread reads and writes only its own (target, column) elements, so out may be vals and out_grads grads.
__global__ void k_rbf_finish(RbfFinish f) {
  const size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (t >= f.m * (size_t)f.n_cols) return;
  const size_t i = t / f.n_cols;
  const int c = (int)(t % f.n_cols), dim = f.dim, nc = f.n_cols;
  double val = f.vals[t];
  double g[3] = {0, 0, 0};
  const bool grads = f.out_grads != nullptr;
  if (grads) {
    for (int d = 0; d < dim; ++d) g[d] = f.grads[i * (size_t)(nc * dim) + (size_t)c * dim + d];
    if (f.trend.on) {  // grad_x f = grad_x' f * B^T (B^T[j][k] = B[k][j])
      const int h = dim + 1;
      const double tmp[3] = {g[0], g[1], g[2]};
      for (int k = 0; k < dim; ++k) {
        double acc = 0.0;
        for (int j = 0; j < dim; ++j) acc = __dadd_rn(acc, __dmul_rn(tmp[j], f.trend.a[k * h + j]));
        g[k] = acc;
      }
    }
  }
  if (f.w) val = __dadd_rn(val, __dmul_rn(f.nugget, f.w[t]));
  if (f.basis > 0) {
    double sp[3] = {0, 0, 0};
    for (int d = 0; d < dim; ++d)
      sp[d] = (f.targets[(ptrdiff_t)i * f.t_rs + (ptrdiff_t)d * f.t_cs] - f.translation[d]) / f.scale[d];
    double mono[10];
    monomial_row(sp, dim, f.degree, mono);
    double v = 0;
    for (int k = 0; k < f.basis; ++k) v = __dadd_rn(v, __dmul_rn(mono[k], f.poly[(size_t)k * nc + c]));
    val = __dadd_rn(val, v);
    if (grads && f.degree >= 1) {
      for (int d = 0; d < dim; ++d) g[d] = __dadd_rn(g[d], f.poly[(size_t)(1 + d) * nc + c] / f.scale[d]);
      if (f.degree == 2) {
        int k = 1 + dim;
        for (int a = 0; a < dim; ++a)
          for (int b = a; b < dim; ++b) {
            const double cf = f.poly[(size_t)k * nc + c];
            if (a == b) {
              g[a] = __dadd_rn(g[a], __dmul_rn(cf, 2.0 * sp[a] / f.scale[a]));
            } else {
              g[a] = __dadd_rn(g[a], __dmul_rn(cf, sp[b] / f.scale[a]));
              g[b] = __dadd_rn(g[b], __dmul_rn(cf, sp[a] / f.scale[b]));
            }
            ++k;
          }
      }
    }
  }
  f.out[t] = val;
  if (grads)
    for (int d = 0; d < dim; ++d) f.out_grads[i * (size_t)(nc * dim) + (size_t)c * dim + d] = g[d];
}

// ----------------------------------------------------------------------------------------- launches
void launch_copy_rows(const double *src, ptrdiff_t s_rs, ptrdiff_t s_cs, size_t rows, int cols, double *dst,
                      ptrdiff_t d_rs, ptrdiff_t d_cs, const AffineMap &aff, cudaStream_t s) {
  FB_LAUNCH(k_copy_rows, nblocks(rows, 256), 256, 0, s, src, s_rs, s_cs, rows, cols, dst, d_rs, d_cs, aff);
}

void device_extents(const double *x, size_t m, int dim, ptrdiff_t rs, ptrdiff_t cs, DBuf<double> &scratch,
                    cudaStream_t s, double *ext) {
  const int parts = (int)std::min<size_t>(kExtBlocks, nblocks(m, kExtThreads));
  scratch.reserve((size_t)(parts + 1) * 2 * dim);
  double *fin = scratch.p + (size_t)parts * 2 * dim;
  FB_LAUNCH(k_extents_partial, parts, kExtThreads, 0, s, x, m, dim, rs, cs, scratch.p);
  FB_LAUNCH(k_extents_final, 1, 32, 0, s, scratch.p, parts, dim, fin);
  FB_CUDA(cudaMemcpyAsync(ext, fin, 2 * dim * sizeof(double), cudaMemcpyDeviceToHost, s));
  FB_CUDA(cudaStreamSynchronize(s));
}

void launch_rbf_finish(const RbfFinish &f, cudaStream_t s) {
  FB_LAUNCH(k_rbf_finish, nblocks(f.m * (size_t)f.n_cols, 128), 128, 0, s, f);
}

}  // namespace fb

using namespace fb;

// ------------------------------------------------------------------------------------ fb_tree pieces
TargetSet fb_tree::bin_targets_dev(const double *d_targets, size_t m, ptrdiff_t rs, ptrdiff_t cs, const double *aff,
                                   uint64_t *bad) {
  FB_REQUIRE(m < (1ull << 31), "at most 2^31-1 targets per call");
  AffineMap map;
  if (aff) {
    map.on = 1;
    std::copy(aff, aff + (dim + 1) * (dim + 1), map.a);
  }
  d_t_user.reserve(m * dim);
  launch_copy_rows(d_targets, rs, cs, m, dim, d_t_user.p, dim, 1, map, stream);
  return bin_user_targets(m, bad);
}

void fb_tree::upload_weights_dev(const double *d_w_in, size_t n_rows, size_t nrhs_, ptrdiff_t rs, ptrdiff_t cs) {
  FB_REQUIRE(n_rows >= n, "weights must have at least one row per source point");
  d_w_user.reserve(n * nrhs_);
  launch_copy_rows(d_w_in, rs, cs, n, (int)nrhs_, d_w_user.p, (ptrdiff_t)nrhs_, 1, AffineMap{}, stream);
  // d_w_user no longer holds h_w_last: a later host upload of those bytes must not be skipped as a repeat, and no
  // evaluate may take the solver's speculative path on the strength of an earlier host upload
  w_cache_valid = false;
  last_w_ptr = nullptr;
  spec_targets = nullptr;
  nrhs = (int)nrhs_;
  sort_weights();
}

// ------------------------------------------------------------------------------------------ C ABI
extern "C" {

int fb_tree_set_weights_device(fb_tree *t, const double *d_w, size_t n_rows, size_t nrhs, ptrdiff_t rs, ptrdiff_t cs,
                               void *stream) {
  return guarded([&] {
    FB_REQUIRE(t, "null tree");
    FB_REQUIRE(d_w != nullptr && nrhs >= 1, "weights must be a non-empty device matrix");
    FB_REQUIRE(n_rows >= t->n, "weights must have at least one row per source point");
    FB_CUDA(cudaSetDevice(t->device));
    require_device_matrix(d_w, t->n, nrhs, rs, cs, t->device, "weights");
    StreamJoin sj((cudaStream_t)stream, t->stream);
    t->upload_weights_dev(d_w, n_rows, nrhs, rs, cs);
    t->upward();
    sj.join();
  });
}

int fb_tree_evaluate_device(fb_tree *t, const double *d_w, size_t n_rows, size_t nrhs, ptrdiff_t w_rs, ptrdiff_t w_cs,
                            const double *d_targets, size_t m, ptrdiff_t t_rs, ptrdiff_t t_cs, double *d_out,
                            double *d_grads_or_null, ptrdiff_t o_rs, ptrdiff_t o_cs, void *stream,
                            uint64_t *bad_index) {
  return guarded(
      [&] {
        FB_REQUIRE(t, "null tree");
        FB_REQUIRE(d_w != nullptr, "weights must be a non-empty device matrix");
        FB_REQUIRE(n_rows >= t->n, "weights must have at least one row per source point");
        FB_REQUIRE(d_targets != nullptr && m > 0, "target_points must be a non-empty m x dim device matrix");
        FB_REQUIRE(d_out, "output buffer required");
        FB_REQUIRE(t->have_weights, "set_weights must be called before evaluate");
        FB_REQUIRE((int)nrhs == t->nrhs, "weights must have the column count given to set_weights");
        FB_CUDA(cudaSetDevice(t->device));
        const bool grads = d_grads_or_null != nullptr;
        const size_t gcols = nrhs * (size_t)t->dim;
        // gradients: row-major when the values are (o_cs == 1), column-major otherwise, as fb_tree_evaluate
        const ptrdiff_t g_rs = o_cs == 1 ? (ptrdiff_t)gcols : 1, g_cs = o_cs == 1 ? 1 : (ptrdiff_t)m;
        require_device_matrix(d_w, t->n, nrhs, w_rs, w_cs, t->device, "weights");
        require_device_matrix(d_targets, m, t->dim, t_rs, t_cs, t->device, "target_points");
        require_device_matrix(d_out, m, nrhs, o_rs, o_cs, t->device, "output");
        if (grads) require_device_matrix(d_grads_or_null, m, gcols, g_rs, g_cs, t->device, "gradient output");
        StreamJoin sj((cudaStream_t)stream, t->stream);
        // targets before weights: a target outside the tree leaves the tree's state intact
        TargetSet ts = t->bin_targets_dev(d_targets, m, t_rs, t_cs, nullptr, bad_index);
        t->upload_weights_dev(d_w, n_rows, nrhs, w_rs, w_cs);
        if (ts.all_sources && !grads) {
          t->evaluate_sources_fused(ts);
        } else {
          t->downward(ts.cell_flag);
          t->leaf_pass(ts, grads);
        }
        auto store = [&](const double *src, size_t cols, double *dst, ptrdiff_t rs, ptrdiff_t cs) {
          if (cs == 1 && rs == (ptrdiff_t)cols)
            FB_CUDA(cudaMemcpyAsync(dst, src, m * cols * sizeof(double), cudaMemcpyDeviceToDevice, t->stream));
          else
            launch_copy_rows(src, (ptrdiff_t)cols, 1, m, (int)cols, dst, rs, cs, AffineMap{}, t->stream);
        };
        store(t->d_out.p, nrhs, d_out, o_rs, o_cs);
        if (grads) store(t->d_gout.p, gcols, d_grads_or_null, g_rs, g_cs);
        sj.join();
      },
      bad_index);
}

}  // extern "C"
