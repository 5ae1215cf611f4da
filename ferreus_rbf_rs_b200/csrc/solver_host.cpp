// Host-side setup of the RBF solve.  See solver_host.h for the reference mapping.
#include "solver_host.h"

#include <algorithm>
#include <parallel/algorithm>
#include <chrono>
#include <cmath>
#include <deque>
#include <memory>
#include <numeric>
#include <string>

#include "monomials.h"

namespace fb {

bool resolve_settings(const fr_settings &in, int dim, Settings &out, std::string &err) {
  out = Settings{};
  out.kernel_type = in.kernel_type;
  if (in.kernel_type < 0 || in.kernel_type > 3) {
    err = "unknown RBF kernel type";
    return false;
  }
  static const int min_drift[4] = {FR_DRIFT_CONSTANT, FR_DRIFT_LINEAR, FR_DRIFT_LINEAR, FR_DRIFT_NONE};
  out.drift = in.drift == FR_DRIFT_DEFAULT ? min_drift[in.kernel_type] : in.drift;
  out.spheroidal_order = in.spheroidal_order ? in.spheroidal_order : 3;
  out.nugget = in.nugget;
  out.base_range = in.base_range;
  out.total_sill = in.total_sill;
  out.tolerance = in.tolerance;
  out.tolerance_type = in.tolerance_type;
  // set_basis_size, interpolant_config.rs:229-264
  if (out.drift < 0 || out.drift > 3) {
    err = "unknown drift";
    return false;
  }
  const int deg = out.drift - 1;
  static const int min_degree[4] = {0, 1, 1, -1};
  if (deg < min_degree[in.kernel_type]) {
    err = "Min degree for kernel: " + std::to_string(min_degree[in.kernel_type]);
    return false;
  }
  const int k = deg + 1;
  out.basis_size = deg < 0 ? 0 : (dim == 1 ? k : (dim == 2 ? k * (k + 1) / 2 : k * (k + 1) * (k + 2) / 6));
  out.polynomial_degree = deg;
  // From<InterpolantSettings> for KernelParams, interpolant_config.rs:267-291
  int kt = FB_KERNEL_LINEAR;
  if (in.kernel_type == FR_KERNEL_THIN_PLATE_SPLINE) kt = FB_KERNEL_THIN_PLATE_SPLINE;
  if (in.kernel_type == FR_KERNEL_CUBIC) kt = FB_KERNEL_CUBIC;
  if (in.kernel_type == FR_KERNEL_SPHEROIDAL) {
    switch (out.spheroidal_order) {
      case 3: kt = FB_KERNEL_SPHEROIDAL3; break;
      case 5: kt = FB_KERNEL_SPHEROIDAL5; break;
      case 7: kt = FB_KERNEL_SPHEROIDAL7; break;
      case 9: kt = FB_KERNEL_SPHEROIDAL9; break;
      default: err = "spheroidal order must be 3, 5, 7 or 9"; return false;
    }
  }
  out.kparams.kernel_type = kt;
  out.kparams.base_range = in.base_range;
  out.kparams.total_sill = in.total_sill;
  // (the builder asserts of kernel_helpers.rs:72-73 are not on this path: From<InterpolantSettings> builds the
  //  struct directly, interpolant_config.rs:267-291)
  return true;
}

void cheb_cube_scaling(const double *pts, const int64_t *idx, size_t n, int dim, double *translation, double *scale) {
  for (int d = 0; d < dim; ++d) {
    double lo = pts[(size_t)(idx ? idx[0] : 0) * dim + d], hi = lo;
    for (size_t i = 0; i < n; ++i) {
      const double v = pts[(size_t)(idx ? idx[i] : (int64_t)i) * dim + d];
      if (v < lo) lo = v;
      if (v > hi) hi = v;
    }
    translation[d] = (hi + lo) / 2.0;
    scale[d] = (hi - lo) / 2.0;
    if (scale[d] == 0.0) scale[d] = 1.0;
  }
}

void evaluate_monomials(const double *pts, const int64_t *idx, size_t n, int dim, int degree, int basis,
                        const double *translation, const double *scale, double *out) {
  if (basis == 0) return;
  for (size_t i = 0; i < n; ++i) {
    const double *p = pts + (size_t)(idx ? idx[i] : (int64_t)i) * dim;
    double s[3] = {0, 0, 0};
    for (int d = 0; d < dim; ++d) s[d] = (p[d] - translation[d]) / scale[d];
    monomial_row(s, dim, degree, out + i * basis);
  }
}

double duplicate_cutoff_distance(double h_ref, const KParams &kp) {
  auto phi = [&](double r) { return kernel_value_rt(r * r, kp); };
  const double eps = 2.220446049250313e-16;
  const double phi0 = phi(0.0), phih = phi(h_ref);
  const double target = eps * std::fabs(phih - phi0);
  auto resid = [&](double r) { return std::fabs(phi(r) - phi0) - target; };
  if (resid(h_ref) <= 0.0) return h_ref;
  double lo = 0.0, hi = h_ref;  // bisection (roots::find_root_inverse_quadratic in the reference, rtol 1e-12)
  for (int it = 0; it < 200; ++it) {
    const double mid = 0.5 * (lo + hi);
    if (resid(mid) > 0.0)
      hi = mid;
    else
      lo = mid;
    if (hi - lo <= 1e-13 * hi) break;
  }
  return 0.5 * (lo + hi);
}

std::vector<int64_t> remove_duplicates(const double *pts, size_t n, int dim, const KParams &kp) {
  double max_len = -INFINITY;
  for (int d = 0; d < dim; ++d) {
    double lo = pts[d], hi = pts[d];
    for (size_t i = 0; i < n; ++i) {
      lo = std::min(lo, pts[i * dim + d]);
      hi = std::max(hi, pts[i * dim + d]);
    }
    max_len = std::max(max_len, std::fabs(hi - lo));
  }
  const double tol = duplicate_cutoff_distance(max_len, kp);
  std::vector<int64_t> order(n);
  std::iota(order.begin(), order.end(), 0);
  __gnu_parallel::stable_sort(order.begin(), order.end(),
                              [&](int64_t a, int64_t b) { return pts[a * dim] < pts[b * dim]; });
  std::vector<double> xs(n);
#pragma omp parallel for schedule(static)
  for (long i = 0; i < (long)n; ++i) xs[i] = pts[order[i] * dim];
  // fast path: no two points within the cutoff of each other => the greedy pass below keeps every point
  bool any_near = false;
#pragma omp parallel for schedule(static) reduction(|| : any_near)
  for (long k = 0; k < (long)n; ++k) {
    const int64_t i = order[k];
    for (size_t q = (size_t)k + 1; q < n && xs[q] - xs[k] <= tol; ++q) {
      const int64_t j = order[q];
      bool near = true;
      for (int d = 0; d < dim && near; ++d)
        if (!(std::fabs(pts[j * dim + d] - pts[i * dim + d]) <= tol)) near = false;
      if (near) any_near = true;
    }
  }
  if (!any_near) {
    std::vector<int64_t> all(n);
    std::iota(all.begin(), all.end(), 0);
    return all;
  }
  std::vector<uint8_t> visited(n, 0);
  std::vector<int64_t> keep;
  for (size_t i = 0; i < n; ++i) {
    if (visited[i]) continue;
    keep.push_back((int64_t)i);
    const double x = pts[i * dim];
    const size_t a = std::lower_bound(xs.begin(), xs.end(), x - tol) - xs.begin();
    const size_t b = std::upper_bound(xs.begin(), xs.end(), x + tol) - xs.begin();
    for (size_t k = a; k < b; ++k) {
      const int64_t j = order[k];
      bool near = true;
      for (int d = 0; d < dim && near; ++d)
        if (!(std::fabs(pts[j * dim + d] - pts[i * dim + d]) <= tol)) near = false;  // infinity norm, inclusive
      if (near) visited[j] = 1;
    }
  }
  return keep;
}

std::vector<int> farthest_point_sampling(const double *pts, const int64_t *idx, size_t n, int dim, size_t wanted,
                                         size_t seed) {
  std::vector<int> selected;
  if (wanted == 0) {  // the reference always pushes the seed (common.rs:256)
    selected.push_back((int)seed);
    return selected;
  }
  selected.reserve(wanted);
  std::vector<uint8_t> is_sel(n, 0);
  std::vector<double> min_d(n, INFINITY);
  selected.push_back((int)seed);
  is_sel[seed] = 1;
  for (size_t it = 1; it < wanted; ++it) {
    const double *last = pts + (size_t)idx[selected.back()] * dim;
    for (size_t i = 0; i < n; ++i) {
      if (is_sel[i]) continue;
      const double *p = pts + (size_t)idx[i] * dim;
      double r2 = 0;
      for (int d = 0; d < dim; ++d) {
        const double df = last[d] - p[d];
        r2 += df * df;
      }
      const double dist = std::sqrt(r2);
      if (dist < min_d[i]) min_d[i] = dist;
    }
    int far = 0;
    double max_dist = -1.0;
    for (size_t i = 0; i < n; ++i)
      if (!is_sel[i] && min_d[i] > max_dist) {
        max_dist = min_d[i];
        far = (int)i;
      }
    selected.push_back(far);
    is_sel[far] = 1;
  }
  return selected;
}

// Householder QR with column pivoting on a column-major rows x cols matrix (overwritten); performs `steps`
// steps, returns the pivot order and |R_kk|.  Pivot = largest remaining column norm, first on ties.
static void qrcp(std::vector<double> &a, int rows, int cols, int steps, std::vector<int> &piv, std::vector<double> &rdiag) {
  piv.resize(cols);
  std::iota(piv.begin(), piv.end(), 0);
  rdiag.assign(steps, 0.0);
  std::vector<double> norms(cols);
  for (int j = 0; j < cols; ++j) {
    double s = 0;
    for (int i = 0; i < rows; ++i) s += a[(size_t)j * rows + i] * a[(size_t)j * rows + i];
    norms[j] = s;
  }
  for (int k = 0; k < steps && k < rows; ++k) {
    int best = k;
    for (int j = k + 1; j < cols; ++j)
      if (norms[j] > norms[best]) best = j;
    if (best != k) {
      for (int i = 0; i < rows; ++i) std::swap(a[(size_t)k * rows + i], a[(size_t)best * rows + i]);
      std::swap(norms[k], norms[best]);
      std::swap(piv[k], piv[best]);
    }
    double nrm = 0;
    for (int i = k; i < rows; ++i) nrm += a[(size_t)k * rows + i] * a[(size_t)k * rows + i];
    nrm = std::sqrt(nrm);
    rdiag[k] = nrm;
    if (nrm == 0.0) continue;
    const double alpha = a[(size_t)k * rows + k] > 0 ? -nrm : nrm;
    const double v0 = a[(size_t)k * rows + k] - alpha;
    std::vector<double> v(rows - k);
    v[0] = 1.0;
    for (int i = k + 1; i < rows; ++i) v[i - k] = a[(size_t)k * rows + i] / v0;
    const double tau = -v0 / alpha;
    a[(size_t)k * rows + k] = alpha;
    for (int i = k + 1; i < rows; ++i) a[(size_t)k * rows + i] = 0.0;
    for (int j = k + 1; j < cols; ++j) {
      double s = 0;
      for (int i = k; i < rows; ++i) s += v[i - k] * a[(size_t)j * rows + i];
      s *= tau;
      for (int i = k; i < rows; ++i) a[(size_t)j * rows + i] -= s * v[i - k];
      // recompute the remaining norm exactly (columns are short; avoids downdating cancellation)
      double r = 0;
      for (int i = k + 1; i < rows; ++i) r += a[(size_t)j * rows + i] * a[(size_t)j * rows + i];
      norms[j] = r;
    }
  }
}

static bool invert_small(std::vector<double> &a, int n, std::vector<double> &inv) {  // row-major, partial pivoting
  inv.assign((size_t)n * n, 0.0);
  for (int i = 0; i < n; ++i) inv[(size_t)i * n + i] = 1.0;
  for (int c = 0; c < n; ++c) {
    int p = c;
    for (int r = c + 1; r < n; ++r)
      if (std::fabs(a[(size_t)r * n + c]) > std::fabs(a[(size_t)p * n + c])) p = r;
    if (a[(size_t)p * n + c] == 0.0) return false;
    if (p != c)
      for (int k = 0; k < n; ++k) {
        std::swap(a[(size_t)p * n + k], a[(size_t)c * n + k]);
        std::swap(inv[(size_t)p * n + k], inv[(size_t)c * n + k]);
      }
    const double d = 1.0 / a[(size_t)c * n + c];
    for (int k = 0; k < n; ++k) {
      a[(size_t)c * n + k] *= d;
      inv[(size_t)c * n + k] *= d;
    }
    for (int r = 0; r < n; ++r) {
      if (r == c) continue;
      const double f = a[(size_t)r * n + c];
      if (f == 0.0) continue;
      for (int k = 0; k < n; ++k) {
        a[(size_t)r * n + k] -= f * a[(size_t)c * n + k];
        inv[(size_t)r * n + k] -= f * inv[(size_t)c * n + k];
      }
    }
  }
  return true;
}

void DomainHost::prepare(const double *pts, int dim, const Settings &s, bool solve_for_poly_, const double *mono_pts) {
  const int n = (int)idx.size();
  if (mask.size() > (size_t)n) mask.resize(n);  // overlap padding beyond the point list (domain_decomposition.rs:303-308)
  rank = 0;
  qtop.clear();
  sp_inv.clear();
  solve_for_poly = false;
  if (s.basis_size == 0) return;
  const int m = s.basis_size;
  double tr[3], sc[3];
  cheb_cube_scaling(pts, idx.data(), n, dim, tr, sc);  // domain.rs:168-169
  std::vector<double> mono((size_t)n * m);
  evaluate_monomials(mono_pts ? mono_pts : pts, idx.data(), n, dim, s.polynomial_degree, m, tr, sc, mono.data());
  // column-pivoted QR of the monomials: unisolvent columns (domain.rs:187-204)
  std::vector<double> a((size_t)n * m);
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < m; ++j) a[(size_t)j * n + i] = mono[(size_t)i * m + j];
  std::vector<int> piv;
  std::vector<double> rd;
  qrcp(a, n, m, std::min(n, m), piv, rd);
  const double thresh = 1e-10 * std::fabs(rd[0]);
  int rk = 0;
  for (double v : rd)
    if (std::fabs(v) > thresh) ++rk;
  std::vector<int> cols(piv.begin(), piv.begin() + rk);
  std::sort(cols.begin(), cols.end());
  // column-pivoted QR of the transpose: special points (domain.rs:219-222)
  std::vector<double> at((size_t)rk * n);
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < rk; ++j) at[(size_t)i * rk + j] = mono[(size_t)i * m + cols[j]];
  std::vector<int> piv2;
  std::vector<double> rd2;
  qrcp(at, rk, n, rk, piv2, rd2);
  std::vector<int> special(piv2.begin(), piv2.begin() + rk);
  std::sort(special.begin(), special.end());
  std::vector<uint8_t> is_special(n, 0);
  for (int sp : special) is_special[sp] = 1;
  std::vector<int> order(special);
  for (int i = 0; i < n; ++i)
    if (!is_special[i]) order.push_back(i);
  std::vector<int64_t> nidx(n);
  std::vector<uint8_t> nmask(n);
  for (int i = 0; i < n; ++i) {
    nidx[i] = idx[order[i]];
    nmask[i] = mask.empty() ? 1 : mask[order[i]];
  }
  idx.swap(nidx);
  mask.swap(nmask);
  rank = rk;
  // Lagrange coefficients on the special points and Q_top = -(ns_mono * lag)^T (domain.rs:300-312)
  std::vector<double> spm((size_t)rk * rk);
  for (int a2 = 0; a2 < rk; ++a2)
    for (int b = 0; b < rk; ++b) spm[(size_t)a2 * rk + b] = mono[(size_t)order[a2] * m + cols[b]];
  std::vector<double> lag;
  invert_small(spm, rk, lag);
  const int mm = n - rk;
  qtop.assign((size_t)rk * mm, 0.0);
  for (int j = 0; j < mm; ++j) {
    const double *row = &mono[(size_t)order[rk + j] * m];
    for (int a2 = 0; a2 < rk; ++a2) {
      double v = 0;
      for (int b = 0; b < rk; ++b) v += row[cols[b]] * lag[(size_t)b * rk + a2];
      qtop[(size_t)a2 * mm + j] = -v;
    }
  }
  if (solve_for_poly_) {
    solve_for_poly = true;
    sp_inv = lag;
  }
}

static int argmax_first_positive(const double *v, int n) {  // ferreus_rbf_utils argmax: strict >, default 0
  int best = 0;
  double bv = 0.0;
  for (int i = 0; i < n; ++i)
    if (v[i] > bv) {
      bv = v[i];
      best = i;
    }
  return best;
}

std::vector<LevelHost> build_ddm(const double *pts, size_t n, int dim, const Settings &s, const fr_params &p,
                                 const double *mono_pts, const LevelCallback *on_level) {
  std::vector<LevelHost> levels;
  static const bool verbose = std::getenv("FB_TIMING") != nullptr;
  auto t_lap = std::chrono::steady_clock::now();
  auto lap = [&](const char *what) {
    if (verbose)
      fprintf(stderr, "[fr_fit]     ddm %-24s %8.3f s\n", what,
              std::chrono::duration<double>(std::chrono::steady_clock::now() - t_lap).count());
    t_lap = std::chrono::steady_clock::now();
  };
  // host part of the factorisations (special points, Q_top), parallel over domains (domain_decomposition.rs:314), as soon
  // as a level is complete; the caller may then queue that level's device factorisation while the next level is built
  auto finish = [&](LevelHost &level, bool is_coarse) {
    std::vector<DomainHost> &doms = level.domains;
#pragma omp parallel for schedule(dynamic, 4)
    for (long i = 0; i < (long)doms.size(); ++i) doms[i].prepare(pts, dim, s, is_coarse && s.basis_size != 0, mono_pts);
    lap("prepare (special points, Q)");
    if (on_level) (*on_level)(levels.size(), level, is_coarse);
    lap("queue level on the device");
  };
  std::vector<int64_t> active(n);
  std::iota(active.begin(), active.end(), 0);
  while (active.size() > p.coarse_threshold) {
    LevelHost level;
    level.point_indices = active;
    DomainHost root;
    root.idx = active;
    root.extents.assign(2 * dim, 0.0);
    for (int d = 0; d < dim; ++d) {
      double lo = pts[active[0] * dim + d], hi = lo;
      for (int64_t i : active) {
        lo = std::min(lo, pts[i * dim + d]);
        hi = std::max(hi, pts[i * dim + d]);
      }
      root.extents[d] = lo;
      root.extents[dim + d] = hi;
    }
    // Bisection, generation by generation: the reference pops a FIFO deque (domain_decomposition.rs:93-162), so a
    // generation is processed completely, in order, before the next one; children and leaves are appended in
    // that same order here, while the domains of one generation are split in parallel.
    std::vector<DomainHost> gen;
    gen.push_back(std::move(root));
    while (!gen.empty()) {
      const size_t ng = gen.size();
      std::vector<DomainHost> lefts(ng), rights(ng);
      std::vector<uint8_t> split_more(ng, 0);
      const bool outer_par = ng >= 8;  // few large domains: parallelise inside a domain instead
#pragma omp parallel for schedule(dynamic, 1) if (outer_par)
      for (long gi = 0; gi < (long)ng; ++gi) {
        DomainHost &cur = gen[gi];
        const size_t nd = cur.idx.size();
        double len[3] = {0, 0, 0};
        for (int d = 0; d < dim; ++d) {
          double lo = pts[cur.idx[0] * dim + d], hi = lo;
#pragma omp parallel for schedule(static) reduction(min : lo) reduction(max : hi) if (!outer_par && nd > 50000)
          for (long k = 0; k < (long)nd; ++k) {
            const double v = pts[cur.idx[k] * dim + d];
            lo = std::min(lo, v);
            hi = std::max(hi, v);
          }
          len[d] = hi - lo;
        }
        const int axis = argmax_first_positive(len, dim);
        // The reference takes a stable argsort by the axis coordinate and cuts it at nd / 2
        // (domain_decomposition.rs:118-131).  The first half of that order is the set of the nd / 2 smallest
        // (coordinate, position) pairs, and both halves are re-sorted by index afterwards, so a selection
        // (nth_element) yields the same two index sets and the same cut coordinate without the full sort.
        std::vector<std::pair<double, int>> ord(nd);
#pragma omp parallel for schedule(static) if (!outer_par && nd > 50000)
        for (long k = 0; k < (long)nd; ++k) ord[k] = {pts[cur.idx[k] * dim + axis], (int)k};
        const size_t mid = nd / 2;
        if (!outer_par && nd > 100000)  // the first generations: few, large domains
          __gnu_parallel::nth_element(ord.begin(), ord.begin() + mid, ord.end());
        else
          std::nth_element(ord.begin(), ord.begin() + mid, ord.end());
        const double mid_coord = ord[mid].first;
        std::vector<uint8_t> in_left(nd, 0);
        DomainHost &left = lefts[gi], &right = rights[gi];
        if (!outer_par && nd > 100000) {
          // the first generations are a handful of huge domains: mark and split with all threads (a stable partition by
          // per-chunk counts), cur.idx is ascending, so both children come out ascending
#pragma omp parallel for schedule(static)
          for (long k = 0; k < (long)mid; ++k) in_left[ord[k].second] = 1;
          left.idx.resize(mid);
          right.idx.resize(nd - mid);
          const int nchunk = 64;
          std::vector<size_t> cnt_l(nchunk + 1, 0);
          const size_t per = (nd + nchunk - 1) / nchunk;
#pragma omp parallel for schedule(static)
          for (int c = 0; c < nchunk; ++c) {
            size_t cl = 0;
            for (size_t k = c * per; k < std::min(nd, (c + 1) * per); ++k) cl += in_left[k];
            cnt_l[c + 1] = cl;
          }
          for (int c = 0; c < nchunk; ++c) cnt_l[c + 1] += cnt_l[c];
#pragma omp parallel for schedule(static)
          for (int c = 0; c < nchunk; ++c) {
            size_t wl = cnt_l[c], wr = std::min(nd, c * per) - cnt_l[c];
            for (size_t k = c * per; k < std::min(nd, (c + 1) * per); ++k) {
              if (in_left[k]) left.idx[wl++] = cur.idx[k];
              else right.idx[wr++] = cur.idx[k];
            }
          }
        } else {
          for (size_t k = 0; k < mid; ++k) in_left[ord[k].second] = 1;
          left.idx.reserve(mid);
          right.idx.reserve(nd - mid);
          for (size_t k = 0; k < nd; ++k)  // cur.idx is ascending, so both children come out ascending
            (in_left[k] ? left.idx : right.idx).push_back(cur.idx[k]);
        }
        left.extents = cur.extents;
        left.extents[axis + dim] = mid_coord;
        right.extents = cur.extents;
        right.extents[axis] = mid_coord;
        split_more[gi] = ((double)nd + (double)nd * p.overlap_quota >= 2.0 * (double)p.leaf_threshold) ? 1 : 0;
        if (!split_more[gi]) {
          left.mask.assign(left.idx.size(), 1);
          right.mask.assign(right.idx.size(), 1);
        }
      }
      std::vector<DomainHost> next_gen;
      for (size_t gi = 0; gi < ng; ++gi) {
        if (split_more[gi]) {
          next_gen.push_back(std::move(lefts[gi]));
          next_gen.push_back(std::move(rights[gi]));
        } else {
          level.domains.push_back(std::move(lefts[gi]));
          level.domains.push_back(std::move(rights[gi]));
        }
      }
      gen.swap(next_gen);
    }
    lap("bisection");
    const size_t nl = level.domains.size();
    const size_t num_coarse =
        (size_t)std::ceil(std::ceil((double)active.size() * p.coarse_ratio) / (double)nl);
    std::vector<std::vector<int64_t>> internal(nl);
    for (size_t i = 0; i < nl; ++i) internal[i] = level.domains[i].idx;
    std::vector<std::vector<int64_t>> coarse_sel(nl), overlap(nl);
#pragma omp parallel for schedule(dynamic, 4)
    for (long ii = 0; ii < (long)nl; ++ii) {
      const size_t i = (size_t)ii;
      const std::vector<int64_t> &in = internal[i];
      const size_t ni = in.size();
      const size_t sample = std::min(ni, num_coarse);
      double centroid[3] = {0, 0, 0};
      for (int d = 0; d < dim; ++d) {
        double sum = 0;
        for (int64_t g : in) sum += pts[g * dim + d];
        centroid[d] = sum / (double)ni;
      }
      size_t centre = 0;
      double best = 0;
      for (size_t k = 0; k < ni; ++k) {
        double r2 = 0;
        for (int d = 0; d < dim; ++d) {
          const double df = centroid[d] - pts[in[k] * dim + d];
          r2 += df * df;
        }
        const double dist = std::sqrt(r2);
        if (k == 0 || dist < best) {
          best = dist;
          centre = k;
        }
      }
      std::vector<int> sel = farthest_point_sampling(pts, in.data(), ni, dim, sample, centre);
      for (int sidx : sel) coarse_sel[i].push_back(in[sidx]);
      std::sort(coarse_sel[i].begin(), coarse_sel[i].end());
      // neighbours: leaf boxes that intersect this one (touching counts, self excluded; rtree.rs:76-89), ascending
      const std::vector<double> &ext = level.domains[i].extents;
      const size_t num_overlap = (size_t)std::ceil((double)(level.domains[i].idx.size() * 2) * p.overlap_quota);
      std::vector<int64_t> nidx;
      for (size_t j = 0; j < nl; ++j) {
        if (j == i) continue;
        const std::vector<double> &o = level.domains[j].extents;
        bool hit = true;
        for (int d = 0; d < dim && hit; ++d)
          if (!(o[d] <= ext[dim + d] && o[dim + d] >= ext[d])) hit = false;
        if (hit) nidx.insert(nidx.end(), internal[j].begin(), internal[j].end());
      }
      std::vector<double> dist(nidx.size());
      for (size_t k = 0; k < nidx.size(); ++k) {
        double r2 = 0;
        for (int d = 0; d < dim; ++d) {
          const double v = pts[nidx[k] * dim + d];
          const double c = std::max(std::min(v, ext[dim + d]), ext[d]);
          const double df = v - c;
          r2 += df * df;
        }
        dist[k] = std::sqrt(r2);
      }
      // the reference takes a stable argsort of the distances and keeps the first `take` (domain_decomposition.rs:289-298):
      // the same prefix, in the same order, comes from selecting the `take` smallest (distance, position) pairs and
      // sorting only those
      std::vector<int> ord(nidx.size());
      std::iota(ord.begin(), ord.end(), 0);
      const size_t take = std::min(num_overlap, nidx.size());
      auto before = [&](int a, int b) { return dist[a] < dist[b] || (dist[a] == dist[b] && a < b); };
      if (take < ord.size()) std::nth_element(ord.begin(), ord.begin() + take, ord.end(), before);
      std::sort(ord.begin(), ord.begin() + take, before);
      for (size_t k = 0; k < take; ++k) overlap[i].push_back(nidx[ord[k]]);
    }
    std::vector<int64_t> next;
    for (size_t i = 0; i < nl; ++i) {
      next.insert(next.end(), coarse_sel[i].begin(), coarse_sel[i].end());
      DomainHost &dm = level.domains[i];
      dm.idx.insert(dm.idx.end(), overlap[i].begin(), overlap[i].end());
      dm.mask.insert(dm.mask.end(), overlap[i].size(), 0);
    }
    std::sort(next.begin(), next.end());
    lap("coarse points + overlap");
    finish(level, false);
    levels.push_back(std::move(level));
    active.swap(next);
  }
  LevelHost coarse;
  coarse.point_indices = active;
  DomainHost cd;
  cd.idx = active;
  cd.mask.assign(active.size(), 1);
  coarse.domains.push_back(std::move(cd));
  finish(coarse, true);
  levels.push_back(std::move(coarse));
  return levels;
}

void thin_q_rowmajor(const double *a, size_t n, int m, double *q) {
  // modified Gram-Schmidt with reorthogonalisation: spans the same column space as Householder thin Q;
  // the Schwarz projection I - Q Q^T only depends on that space (schwarz.rs:122-126)
  std::vector<double> col((size_t)m * n);
  for (size_t i = 0; i < n; ++i)
    for (int j = 0; j < m; ++j) col[(size_t)j * n + i] = a[i * m + j];
  for (int j = 0; j < m; ++j) {
    double *v = &col[(size_t)j * n];
    for (int pass = 0; pass < 2; ++pass)
      for (int k = 0; k < j; ++k) {
        const double *u = &col[(size_t)k * n];
        double dot = 0;
        for (size_t i = 0; i < n; ++i) dot += u[i] * v[i];
        for (size_t i = 0; i < n; ++i) v[i] -= dot * u[i];
      }
    double nrm = 0;
    for (size_t i = 0; i < n; ++i) nrm += v[i] * v[i];
    nrm = std::sqrt(nrm);
    const double inv = nrm > 0 ? 1.0 / nrm : 0.0;
    for (size_t i = 0; i < n; ++i) v[i] *= inv;
  }
  for (size_t i = 0; i < n; ++i)
    for (int j = 0; j < m; ++j) q[i * m + j] = col[(size_t)j * n + i];
}

}  // namespace fb

// ---- host-only duplicate removal + DDM hierarchy (no GPU) --------------------------------------------------------------
// What fr_fit does on the host before anything reaches the device (rbf.rs:341-359, domain_decomposition.rs:67-346), behind
// plain entry points so that the CPU test-suite can compare the kept rows, the levels, the domains, their point order
// (special points first) and the internal masks with the oracle.
struct fr_host_ddm {
  std::vector<int64_t> keep;
  std::vector<fb::LevelHost> levels;
};

extern "C" {

int fr_host_ddm_new(const double *points, size_t n, int dim, ptrdiff_t p_rs, ptrdiff_t p_cs, const fr_settings *settings,
                    const fr_params *params_or_null, fr_host_ddm **out) {
  if (!out) return FB_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  if (!points || !settings || n == 0 || dim < 1 || dim > 3) return FB_ERR_INVALID_ARGUMENT;
  try {
    fb::Settings st;
    std::string err;
    if (!fb::resolve_settings(*settings, dim, st, err)) return FB_ERR_INVALID_ARGUMENT;
    fb::KParams kp;
    if (!fb::make_kparams(st.kparams, kp)) return FB_ERR_INVALID_ARGUMENT;
    fr_params params;
    if (params_or_null) params = *params_or_null;
    else fr_params_default(settings->kernel_type, &params);
    std::vector<double> pts(n * dim);
    for (size_t i = 0; i < n; ++i)
      for (int d = 0; d < dim; ++d) pts[i * dim + d] = points[(ptrdiff_t)i * p_rs + (ptrdiff_t)d * p_cs];
    std::unique_ptr<fr_host_ddm> h(new fr_host_ddm());
    if (params.test_unique) {
      h->keep = fb::remove_duplicates(pts.data(), n, dim, kp);
    } else {
      h->keep.resize(n);
      for (size_t i = 0; i < n; ++i) h->keep[i] = (int64_t)i;
    }
    const size_t m = h->keep.size();
    std::vector<double> kept(m * dim);
    for (size_t k = 0; k < m; ++k) std::copy(&pts[h->keep[k] * dim], &pts[h->keep[k] * dim] + dim, &kept[k * dim]);
    if (m > (size_t)params.naive_solve_threshold) h->levels = fb::build_ddm(kept.data(), m, dim, st, params);
    *out = h.release();
    return FB_OK;
  } catch (...) {
    return FB_ERR_INVALID_ARGUMENT;
  }
}

void fr_host_ddm_free(fr_host_ddm *h) { delete h; }

int fr_host_ddm_counts(const fr_host_ddm *h, uint64_t *n_kept, uint64_t *n_levels) {
  if (!h) return FB_ERR_INVALID_ARGUMENT;
  if (n_kept) *n_kept = h->keep.size();
  if (n_levels) *n_levels = h->levels.size();
  return FB_OK;
}

int fr_host_ddm_kept(const fr_host_ddm *h, uint64_t *rows) {
  if (!h || !rows) return FB_ERR_INVALID_ARGUMENT;
  for (size_t i = 0; i < h->keep.size(); ++i) rows[i] = (uint64_t)h->keep[i];
  return FB_OK;
}

// same layout as fr_ddm_level
int fr_host_ddm_level(const fr_host_ddm *h, int level, uint64_t *n_domains, uint64_t *n_level_points,
                      uint64_t *level_points, uint64_t *dom_ptr, uint64_t *dom_idx, uint8_t *dom_internal) {
  if (!h || level < 0 || level >= (int)h->levels.size()) return FB_ERR_INVALID_ARGUMENT;
  const fb::LevelHost &lh = h->levels[level];
  if (n_domains) *n_domains = lh.domains.size();
  if (n_level_points) *n_level_points = lh.point_indices.size();
  if (level_points)
    for (size_t i = 0; i < lh.point_indices.size(); ++i) level_points[i] = (uint64_t)lh.point_indices[i];
  uint64_t off = 0;
  for (size_t d = 0; d < lh.domains.size(); ++d) {
    if (dom_ptr) dom_ptr[d] = off;
    const fb::DomainHost &dh = lh.domains[d];
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
