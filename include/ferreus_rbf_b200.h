/*
 * ferreus_rbf_b200.h — C ABI of the RBF interpolator (fit + evaluate) in libferreus_b200.so.
 *
 * Replaces `ferreus_rbf::RBFInterpolator` (ferreus_rbf/src/rbf.rs:267-924): builder/new -> fr_fit,
 * coefficients -> fr_coefficients, evaluate* -> fr_evaluate, evaluate_at_source -> fr_evaluate_at_source,
 * build_evaluator -> fr_build_evaluator, evaluate_targets* -> fr_evaluate_targets.  The solve runs on the
 * GPU: device-resident FGMRES (iterative_solvers.rs:38-173), Schwarz DDM preconditioner with batched
 * dense subdomain factorisations / triangular solves (schwarz.rs:32-155, domain.rs:153-467) and the
 * BBFMM matvec of ferreus_b200.h.  Same conventions as ferreus_b200.h: host pointers, element strides,
 * error codes, fb_last_error().
 */
#ifndef FERREUS_RBF_B200_H
#define FERREUS_RBF_B200_H

#include "ferreus_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* RBFKernelType, Drift, SpheroidalOrder, FittingAccuracyType (ferreus_rbf/src/interpolant_config.rs:20-92) */
enum fr_kernel_type { FR_KERNEL_LINEAR = 0, FR_KERNEL_THIN_PLATE_SPLINE = 1, FR_KERNEL_CUBIC = 2, FR_KERNEL_SPHEROIDAL = 3 };
enum fr_drift { FR_DRIFT_NONE = 0, FR_DRIFT_CONSTANT = 1, FR_DRIFT_LINEAR = 2, FR_DRIFT_QUADRATIC = 3, FR_DRIFT_DEFAULT = -1 };
enum fr_tolerance_type { FR_TOL_RELATIVE = 0, FR_TOL_ABSOLUTE = 1 };
enum fr_solver_type { FR_SOLVER_DDM = 0, FR_SOLVER_FGMRES = 1 };

/* InterpolantSettings (interpolant_config.rs:179-264); defaults via fr_settings_default */
typedef struct fr_settings {
  int32_t kernel_type;      /* enum fr_kernel_type */
  int32_t drift;            /* enum fr_drift; FR_DRIFT_DEFAULT = minimum drift for the kernel */
  int32_t spheroidal_order; /* 3, 5, 7 or 9 */
  double nugget;
  double base_range;
  double total_sill;
  double tolerance;         /* FittingAccuracy.tolerance (default 1e-6) */
  int32_t tolerance_type;   /* enum fr_tolerance_type (default relative) */
} fr_settings;

/* Params = solver + DDMParams + FmmParams (ferreus_rbf/src/config.rs:43-253); defaults via fr_params_default */
typedef struct fr_params {
  int32_t solver_type;          /* enum fr_solver_type (default FGMRES) */
  uint64_t leaf_threshold;      /* DDMParams: 1024 */
  double overlap_quota;         /*            0.5  */
  double coarse_ratio;          /*            0.125 */
  uint64_t coarse_threshold;    /*            4096 */
  uint64_t interpolation_order; /* FmmParams: 7 / 9 / 11 for linear(+spheroidal) / TPS / cubic */
  uint64_t max_points_per_cell; /*            256 */
  int32_t compression_type;     /*            ACA */
  double epsilon;               /*            10^-order */
  uint64_t eval_chunk_size;     /*            1024 */
  uint64_t naive_solve_threshold; /* 4096 */
  int32_t test_unique;          /* 1 */
} fr_params;

void fr_settings_default(int32_t kernel_type, fr_settings *out);
void fr_params_default(int32_t kernel_type, fr_params *out);

/* progress events (ferreus_rbf/src/progress.rs:21-41): invoked on the calling host thread */
enum fr_event_kind { FR_EVENT_DUPLICATES_REMOVED = 0, FR_EVENT_SOLVER_ITERATION = 1, FR_EVENT_MESSAGE = 2 };
typedef struct fr_event {
  int32_t kind;
  uint64_t iter;            /* SolverIteration.iter / DuplicatesRemoved.num_duplicates */
  double residual;
  double progress;
  const char *message;
} fr_event;
typedef void (*fr_progress_cb)(const fr_event *ev, void *user);

typedef struct fr_model fr_model; /* opaque: replaces ferreus_rbf::RBFInterpolator */

/* GlobalTrend (ferreus_rbf/src/global_trend.rs:36-126): anisotropy by rotation + axis ratios about the centroid of the
 * (unique) points; angles in degrees.  dim 1: ratios[0] = major.  dim 2: angles[0] = rotation_angle, ratios = {major,
 * minor}.  dim 3: angles = {dip, dip_direction, pitch}, ratios = {major, semi_major, minor}.                        */
typedef struct fr_global_trend {
  int32_t dim;
  double angles[3];
  double ratios[3];
} fr_global_trend;

/* RBFInterpolator::builder(points, values, settings).params(..).progress_callback(..).build()  (rbf.rs:304-412).
 * points: n x dim, values: n x n_cols.  params NULL => defaults.                                      */
int fr_fit(const double *points, size_t n, int dim, ptrdiff_t p_rs, ptrdiff_t p_cs, const double *values,
           size_t n_cols, ptrdiff_t v_rs, ptrdiff_t v_cs, const fr_settings *settings,
           const fr_params *params_or_null, fr_progress_cb cb_or_null, void *user, fr_model **out);
/* ...builder(..).global_trend(trend).build() (rbf.rs:239-242, 361-371); trend NULL == fr_fit */
int fr_fit_trend(const double *points, size_t n, int dim, ptrdiff_t p_rs, ptrdiff_t p_cs, const double *values,
                 size_t n_cols, ptrdiff_t v_rs, ptrdiff_t v_cs, const fr_settings *settings,
                 const fr_params *params_or_null, const fr_global_trend *trend_or_null, fr_progress_cb cb_or_null,
                 void *user, fr_model **out);
void fr_free(fr_model *m);

typedef struct fr_model_info {
  uint64_t n_points;      /* after duplicate removal */
  uint64_t n_duplicates;
  uint64_t n_cols, basis_size, dim;
  uint64_t iterations;    /* total inner iterations over all value columns */
  double last_residual;
  uint64_t ddm_levels;
  uint64_t ddm_domains[8];
  double fit_seconds, setup_seconds, solve_seconds;
  uint64_t matvecs;       /* FMM matvecs executed by the solve */
} fr_model_info;
int fr_get_info(const fr_model *m, fr_model_info *info);

/* fields points / point_values / coefficients (rbf.rs:267-302); any pointer may be NULL; row-major outputs */
int fr_source_points(const fr_model *m, double *points_out /* n x dim */, double *values_out /* n x n_cols */);
int fr_coefficients(const fr_model *m, double *point_out /* n x n_cols */, double *poly_out /* basis x n_cols */);

/* ---- model state for save_model / load_model (rbf.rs:1087-1171: serde JSON envelope of the public + private fields;
 * the JSON itself is written by the host language binding).  fr_model_state describes a fitted model: resolved
 * settings (basis_size / polynomial_degree included), params, monomial scaling and the global-trend matrices.      */
typedef struct fr_model_state {
  fr_settings settings;
  fr_params params;
  int32_t basis_size, polynomial_degree;
  double translation_factor[3], scale_factor[3];
  int32_t has_trend;
  double affine_transform[16], inverse_transform[16]; /* (dim+1) x (dim+1) row-major (global_trend.rs:128-132) */
} fr_model_state;
int fr_get_state(const fr_model *m, fr_model_state *out);
/* rebuilds a fitted model from its parts WITHOUT solving (load_model): points n x dim (original coordinates), values
 * n x n_cols, point coefficients n x n_cols, poly coefficients basis_size x n_cols (or NULL), all row-major.        */
int fr_model_restore(const double *points, size_t n, int dim, const double *values, size_t n_cols,
                     const double *point_coefficients, const double *poly_coefficients_or_null,
                     const fr_model_state *state, fr_progress_cb cb_or_null, void *user, fr_model **out);

/* Host-array evaluation: fr_evaluate, fr_evaluate_at_source and fr_evaluate_targets run the device path of
 * fr_evaluate_device / fr_evaluate_targets_device below, behind one host-to-device copy of the targets and one
 * device-to-host copy of the results.
 * evaluate / evaluate_with_gradients (rbf.rs:676-752): one-shot non-sparse adaptive tree on the union extents.
 * out_vals m x n_cols row-major; out_grads (or NULL) m x (n_cols*dim).                                  */
int fr_evaluate(fr_model *m, const double *targets, size_t n_targets, ptrdiff_t t_rs, ptrdiff_t t_cs,
                double *out_vals, double *out_grads_or_null);
/* evaluate_at_source (rbf.rs:777-828): values at the source points, optionally + nugget * coefficient */
int fr_evaluate_at_source(fr_model *m, int add_nugget, double *out_vals);
/* build_evaluator(extents) (rbf.rs:830-858) + evaluate_targets(_with_gradients) (rbf.rs:860-924) */
int fr_build_evaluator(fr_model *m, const double *extents_or_null);
int fr_evaluate_targets(fr_model *m, const double *targets, size_t n_targets, ptrdiff_t t_rs, ptrdiff_t t_cs,
                        double *out_vals, double *out_grads_or_null);

/* ---- device-memory variants (not in the reference API): targets (n_targets x dim, element strides) and outputs
 * (row-major, the layouts of fr_evaluate) are device memory of the current CUDA device; `stream` is the caller's
 * cudaStream_t.  Pointer checks, stream order, input lifetime and errors as fb_tree_evaluate_device
 * (ferreus_b200.h); the handle stays usable after any error.
 *  - fr_evaluate_device: fr_evaluate, the one-shot tree over the union of source and target extents.  The extents
 *    are reduced on `stream` and read back (2 * dim doubles), and the temporary tree is freed at the end, so this call
 *    blocks until its results are complete.
 *  - fr_evaluate_targets_device: fr_evaluate_targets, through the tree of fr_build_evaluator.  Blocks until the
 *    targets are binned, not until the results are complete.  With d_grads it returns the evaluator's gradients
 *    (unlike the reference's evaluate_targets_with_gradients, which takes the one-shot path).                    */
int fr_evaluate_device(fr_model *m, const double *d_targets, size_t n_targets, ptrdiff_t t_rs, ptrdiff_t t_cs,
                       double *d_out, double *d_grads_or_null, void *stream);
int fr_evaluate_targets_device(fr_model *m, const double *d_targets, size_t n_targets, ptrdiff_t t_rs, ptrdiff_t t_cs,
                               double *d_out, double *d_grads_or_null, void *stream);

/* ---- isosurfaces of 3-D interpolants (not in the reference API) ------------------------------------------------
 * Lattice: extents = {x0, y0, z0, x1, y1, z1} with lo < hi, resolution = {nx, ny, nz} >= 2, at most 2^28 nodes; node
 * idx on an axis is idx * step + lo, step = (hi - lo) / (n - 1), the last node exactly hi (np.linspace); node
 * p = i + nx * (j + ny * k).  A node is below when its value is < iso.  Every cube is split into the 6 Kuhn
 * tetrahedra, so the mesh has no cracks: one vertex per crossing lattice edge (numbered by edge id), triangles ordered
 * by (cube, tetrahedron, triangle) and oriented so that (B-A) x (C-A) points along increasing value.  Every mesh edge
 * is used by two triangles in opposite directions except on the lattice's boundary faces.  DESIGN.md has the full
 * specification.
 *  - fr_isosurface_extract: one transient tree over the union of the lattice and the source points (the rule of
 *    fr_evaluate_device; fr_build_evaluator's tree is not touched) evaluates column `column` on the lattice; one
 *    surface per isovalue.  refine != 0 moves every vertex along its edge onto the interpolant (Illinois regula falsi
 *    from the lattice bracket: stops at a bracket of 2^-40 of the edge, f == iso, or 60 evaluations); normals are the
 *    normalised interpolant gradient at the final vertices.  Blocks until complete.
 *  - fr_lattice_isosurface: the mesh of caller-owned lattice values (device memory, nz x ny x nx contiguous) on the
 *    caller's cudaStream_t; vertices stay on the lattice edges' linear interpolation and there are no normals.
 *    Blocks until complete.
 *  - results stay in the handle's device memory: fr_isosurface_counts, then fr_isosurface_copy to host or device
 *    memory (vertices V x 3, faces F x 3 of int64 vertex indices, normals V x 3 or NULL; `which` = isovalue index).
 *  - fr_isosurface_timing: milliseconds of {lattice evaluation with the tree, extraction, refinement, normals}.
 *  - fr_isosurface_refine_stats: trial points evaluated by the refinement and its iteration count (the slowest
 *    vertex's evaluations).
 * Solids: fr_isosurface_extract_solid and fr_lattice_solid take the arguments above plus side (0: the region
 * {f < iso}, 1: {f >= iso}) and close each isosurface at the lattice box into the boundary of that region.  The
 * isosurface's vertices and faces come first, unchanged except that side 1 exchanges every face's last two vertices;
 * then the boundary nodes on the solid's side (ascending node index) and the cap faces on the six box faces.  Every
 * face points out of the solid; normals (model path) are outward too.  fr_isosurface_counts / _copy include the cap.
 *  - fr_isosurface_solid_info: the number of isosurface vertices and faces at the front, the enclosed volume and the
 *    area of the isosurface faces, computed on the device from the final vertices by fixed-order reductions (the same
 *    bits from call to call).  FB_ERR_INVALID_ARGUMENT on a handle of open isosurfaces.
 *  - for solids the refinement time of fr_isosurface_timing includes the volume and area reductions.
 * Invalid arguments (a model that is not 3-D, a bad lattice, n_iso < 1, a non-finite isovalue or lattice value, a
 * column out of range, a side other than 0 or 1) return FB_ERR_INVALID_ARGUMENT and leave the model usable.       */
typedef struct fr_isosurface fr_isosurface;
int fr_isosurface_extract(fr_model *m, const double *extents, const uint64_t *resolution, const double *isovalues,
                          int n_iso, int column, int refine, fr_isosurface **out);
int fr_lattice_isosurface(const double *d_values, const uint64_t *resolution, const double *extents, double isovalue,
                          void *stream, fr_isosurface **out);
int fr_isosurface_counts(const fr_isosurface *s, int which, uint64_t *n_vertices, uint64_t *n_faces);
int fr_isosurface_copy(const fr_isosurface *s, int which, double *vertices, int64_t *faces, double *normals_or_null);
int fr_isosurface_timing(const fr_isosurface *s, double *ms_out4);
int fr_isosurface_refine_stats(const fr_isosurface *s, int which, uint64_t *evaluations, uint64_t *iterations);
void fr_isosurface_free(fr_isosurface *s);
int fr_isosurface_extract_solid(fr_model *m, const double *extents, const uint64_t *resolution,
                                const double *isovalues, int n_iso, int column, int refine, int side,
                                fr_isosurface **out);
int fr_lattice_solid(const double *d_values, const uint64_t *resolution, const double *extents, double isovalue,
                     int side, void *stream, fr_isosurface **out);
int fr_isosurface_solid_info(const fr_isosurface *s, int which, uint64_t *surface_vertices, uint64_t *surface_faces,
                             double *volume, double *surface_area);

/* ---- introspection for the parity gates ------------------------------------------------------------- */
/* DDM hierarchy: level l (0 = finest ... levels-1 = coarse): number of domains, and per domain the point
 * indices (CSR) with the internal mask.  Any pointer may be NULL (call once for sizes, once for data).     */
int fr_ddm_level(const fr_model *m, int level, uint64_t *n_domains, uint64_t *n_level_points,
                 uint64_t *level_points, uint64_t *dom_ptr, uint64_t *dom_idx, uint8_t *dom_internal);

/* ---- host-only duplicate removal + DDM hierarchy (no GPU needed): what fr_fit does on the host before anything reaches
 * the device (rbf.rs:341-359, 1391-1467; domain_decomposition.rs:67-346; the host part of domain.rs:153-330), for the CPU
 * test-suite.  No levels are built when the kept points do not exceed naive_solve_threshold (single dense domain).
 * fr_host_ddm_level has the layout of fr_ddm_level.                                                             ---- */
typedef struct fr_host_ddm fr_host_ddm;
int fr_host_ddm_new(const double *points, size_t n, int dim, ptrdiff_t p_rs, ptrdiff_t p_cs, const fr_settings *settings,
                    const fr_params *params_or_null, fr_host_ddm **out);
void fr_host_ddm_free(fr_host_ddm *h);
int fr_host_ddm_counts(const fr_host_ddm *h, uint64_t *n_kept, uint64_t *n_levels);
int fr_host_ddm_kept(const fr_host_ddm *h, uint64_t *rows /* n_kept input rows that survive duplicate removal */);
int fr_host_ddm_level(const fr_host_ddm *h, int level, uint64_t *n_domains, uint64_t *n_level_points,
                      uint64_t *level_points, uint64_t *dom_ptr, uint64_t *dom_idx, uint8_t *dom_internal);

/* ---- entry points of the reference's reproducible known-answer tests --------------------------------------------
 * fr_dense_spd_solve: x = A^-1 b for a dense symmetric n x n matrix (row-major) through the batched subdomain kernels
 * (blocked Cholesky with the DMMA trailing update, forward / backward substitution; an indefinite matrix takes the
 * fallback of domain.rs:63-68) -- linalg.rs:638-764 (make_spd) runs against it.  b, x: n x nrhs row-major.
 * fr_evaluate_monomials: polynomials.rs:15-62 / its tests :163-239 (column order [1, x, y, z, x^2, xy, xz, y^2, yz, z^2]);
 * host only, translation / scale may be NULL (0 / 1).
 * fr_ddm_level_solve: the subdomain solves of one DDM level, for tests against dense references.  The points (n x dim,
 * row-major) go through fr_fit's set-up without the FMM tree: duplicate removal, monomial scaling, the hierarchy (or the
 * single dense domain below naive_solve_threshold; fr_host_ddm_level shows its domains) and every level's
 * factorisation.  Then each of the nvec residuals res (n_kept + basis_size rows each, one after the other) is solved on
 * `level`: fine levels write the point rows of every domain's internal points, the coarse level those of all its points
 * and, with add_poly, the recovered polynomial into the last `rank` rows; out (same layout) is zeroed first, so rows
 * nothing writes stay 0.  n_fallback_or_null: domains of the level that took the indefinite fallback;
 * domain_ranks_or_null: special points per domain (one entry per domain of the level).                            */
int fr_dense_spd_solve(const double *a, int n, const double *b, int nrhs, double *x, int *used_fallback_or_null);
int fr_ddm_level_solve(const double *points, size_t n, int dim, const fr_settings *settings, const fr_params *params_or_null,
                       int level, int add_poly, const double *res, int nvec, double *out, uint64_t *n_fallback_or_null,
                       uint64_t *domain_ranks_or_null);
int fr_evaluate_monomials(const double *points, size_t n, int dim, int degree, const double *translation_or_null,
                          const double *scale_or_null, double *out, int *basis_out);

#ifdef __cplusplus
}
#endif
#endif /* FERREUS_RBF_B200_H */
