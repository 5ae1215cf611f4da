"""GPU parity tests of the RBF solve path (FGMRES + Schwarz DDM + batched subdomain solves) through the C ABI.

Bars (BASELINE.json north_star): interpolant values <= 1e-8 relative to the reference's solve at equal FGMRES
tolerance — run at a tight tolerance where both solves reach the same fixed point (SURVEY.md §7 hard part 2);
DDM hierarchy (index construction) bit-exact against the oracle restatement.
"""
import numpy as np
import pytest

from tests import helpers as H

pytestmark = pytest.mark.gpu

INTERP_TOL = 1e-8


def _settings(kernel, tol=1e-6, **kw):
    import ferreus_rbf_rs_b200 as fb
    ic = fb.interpolant_config
    return ic.InterpolantSettings(ic.RBFKernelType(kernel),
                                  fitting_accuracy=ic.FittingAccuracy(tol, ic.FittingAccuracyType.Relative), **kw)


def _params(kernel, leaf=128, coarse=300, naive=100, order=8, max_pts=40, eps=1e-10, solver=None):
    import ferreus_rbf_rs_b200 as fb
    cfg = fb.config
    return cfg.Params(fb.interpolant_config.RBFKernelType(kernel),
                      solver_type=solver,
                      ddm_params=cfg.DDMParams(leaf, 0.5, 0.125, coarse),
                      fmm_params=cfg.FmmParams(order, max_pts, cfg.FmmCompressionType.ACA, eps, 1024),
                      naive_solve_threshold=naive)


def _oracle(kernel, pts, vals, tol, leaf=128, coarse=300, naive=100, order=8, max_pts=40, eps=1e-10, solver=1, **kw):
    from oracle import rbf as orbf
    s = orbf.InterpolantSettings(kernel, tolerance=tol, **kw)
    p = orbf.Params(kernel, solver_type=solver, leaf_threshold=leaf, coarse_threshold=coarse,
                    naive_solve_threshold=naive, interpolation_order=order, max_points_per_cell=max_pts, epsilon=eps)
    return orbf.RBFInterpolator(pts, vals, s, p)


def _values(pts):
    if pts.shape[1] == 1:
        return np.sin(3 * pts[:, 0]) + pts[:, 0] ** 2
    v = np.sin(3 * pts[:, 0]) + pts[:, 1] ** 2
    return v - pts[:, 2] if pts.shape[1] == 3 else v


def _dense_solution(pts, vals, oracle_model):
    from oracle import rbf as orbf
    s = oracle_model.settings
    n, m = pts.shape[0], s.basis_size
    A = s.kernel().matrix(pts, pts) + s.nugget * np.eye(n)
    if m == 0:
        return np.linalg.solve(A, vals), None
    P = orbf.evaluate_monomials(pts, s.polynomial_degree, m, oracle_model.translation, oracle_model.scale)
    K = np.block([[A, P], [P.T, np.zeros((m, m))]])
    sol = np.linalg.solve(K, np.concatenate([vals, np.zeros((m, vals.shape[1]))]))
    return sol[:n], sol[n:]


@pytest.mark.parametrize("kernel,dim,n", [(0, 3, 900), (1, 2, 800), (2, 3, 700), (3, 3, 600)])
def test_direct_domain_solve_matches_dense(kernel, dim, n):
    """N < naive_solve_threshold: single dense domain (rbf.rs:423-454); reference tests domain.rs:683-762."""
    import ferreus_rbf_rs_b200 as fb
    pts = H.make_points(n, dim, "uniform", seed=7)
    vals = np.stack([_values(pts), np.cos(2 * pts[:, 0])], axis=1)
    kw = {"base_range": 0.4} if kernel == 3 else {}
    model = fb.RBFInterpolator(pts, vals, _settings(kernel, **kw))
    om = _oracle(kernel, pts, vals, 1e-6, naive=4096, **kw)
    lam, c = _dense_solution(pts, vals, om)
    co = model.coefficients
    assert H.rel_l2(co.point_coefficients, lam) <= 1e-7
    if c is not None:
        assert H.rel_l2(co.poly_coefficients, c) <= 1e-7
    # interpolation reproduces the data (atol 1e-12 + rtol 1e-10 in domain.rs:683-729; FMM evaluation adds ~1e-7)
    at_src = model.evaluate_at_source()
    assert H.rel_l2(at_src, vals) <= 1e-5


@pytest.mark.parametrize("kernel,dim,n", [(0, 3, 2600), (1, 2, 2600)])
def test_ddm_hierarchy_bit_exact(kernel, dim, n):
    import ferreus_rbf_rs_b200 as fb
    from oracle import rbf as orbf
    pts = H.make_points(n, dim, "clustered", seed=17)
    vals = _values(pts)
    model = fb.RBFInterpolator(pts, vals, _settings(kernel, tol=1e-2), params=_params(kernel, order=5, eps=1e-5))
    s = orbf.InterpolantSettings(kernel)
    s.set_basis_size(dim)
    keep = orbf.remove_duplicates(pts, s.kernel())
    ddm = orbf.DDMTree(pts[keep], s, 128, 0.5, 0.125, 300, factorise=False)
    info = model.info()
    assert info["ddm_levels"] == len(ddm.levels)
    assert info["ddm_domains"] == [len(l.leaf_domains) for l in ddm.levels]
    for li, lvl in enumerate(ddm.levels):
        lp, ptr, idx, internal = model.ddm_level(li)
        assert np.array_equal(lp.astype(np.int64), lvl.point_indices)
        for d, dom in enumerate(lvl.leaf_domains):
            a, b = int(ptr[d]), int(ptr[d + 1])
            mine_all = idx[a:b].astype(np.int64)
            mine_int = mine_all[internal[a:b] == 1]
            k = min(len(dom.mask), len(dom.idx))
            assert sorted(mine_all.tolist()) == sorted(dom.idx.tolist())
            assert sorted(mine_int.tolist()) == sorted(dom.idx[:k][dom.mask[:k]].tolist())


@pytest.mark.parametrize("kernel,dim,n,kind", [(0, 3, 2400, "uniform"), (2, 3, 2000, "clustered"), (1, 2, 2400, "uniform")])
def test_fgmres_ddm_fit_matches_oracle_and_dense(kernel, dim, n, kind):
    import ferreus_rbf_rs_b200 as fb
    pts = H.make_points(n, dim, kind, seed=23)
    vals = _values(pts)
    tol = 1e-10
    model = fb.RBFInterpolator(pts, vals, _settings(kernel, tol=tol), params=_params(kernel))
    om = _oracle(kernel, pts, vals, tol)
    info = model.info()
    assert info["ddm_levels"] >= 2 and info["iterations"] > 0
    targets = np.random.default_rng(1).random((400, dim)) * (pts.max(0) - pts.min(0)) + pts.min(0)
    got = np.asarray(model.evaluate(targets)).reshape(-1, 1)
    ref = om.evaluate(targets)
    assert H.rel_l2(got, ref) <= INTERP_TOL
    # against the exact solution of the bordered dense system, evaluated densely
    lam, c = _dense_solution(om.points, om.values, om)
    from oracle import rbf as orbf
    s = om.settings
    exact = s.kernel().matrix(targets, om.points) @ lam
    if c is not None:
        exact = exact + orbf.evaluate_monomials(targets, s.polynomial_degree, s.basis_size, om.translation, om.scale) @ c
    assert H.rel_l2(got, exact) <= 2e-5   # accuracy of the FMM-approximated solve itself (the oracle has the same error)
    # iteration counts of the two solves agree (same algorithm, same stopping rule)
    assert abs(info["iterations"] - om.iterations) <= 1


def test_default_tolerance_fit_and_evaluators():
    """tol 1e-6 (reference default): the comparison the north star quotes, reported at its natural accuracy."""
    import ferreus_rbf_rs_b200 as fb
    kernel, dim, n = 0, 3, 3000
    pts = H.make_points(n, dim, "uniform", seed=29)
    vals = np.stack([_values(pts), np.cos(2 * pts[:, 0])], axis=1)
    events = []
    prog = fb.progress.Progress(lambda ev: events.append(ev))
    model = fb.RBFInterpolator(pts, vals, _settings(kernel), params=_params(kernel), progress_callback=prog)
    its = [e for e in events if isinstance(e, fb.progress.SolverIteration)]
    assert its and its[-1].residual < 1e-6 and 0.0 <= its[0].progress <= 1.0
    assert any(isinstance(e, fb.progress.Message) for e in events)
    at_src = model.evaluate_at_source()
    assert H.rel_l2(at_src, vals) <= 1e-4
    targets = np.random.default_rng(2).random((500, dim))
    v1 = model.evaluate(targets)
    v2, g2 = model.evaluate_with_gradients(targets)
    assert v1.shape == (500, 2) and g2.shape == (500, 6)
    assert H.rel_l2(v2, v1) <= 1e-12
    model.build_evaluator()
    with pytest.raises(ValueError):
        model.evaluate_targets(np.array([[5.0, 5.0, 5.0]]))     # outside the evaluator extents
    inside = pts[:300] * 0.999 + 0.0005
    v3 = model.evaluate_targets(inside)
    v4 = model.evaluate(inside)
    assert H.rel_l2(v3, v4) <= 1e-6
    # central differences of the interpolant agree with the analytic gradients
    h = 1e-5
    x = targets[:50]
    _, g = model.evaluate_with_gradients(x)
    for d in range(3):
        e = np.zeros(3)
        e[d] = h
        fd = (model.evaluate(x + e) - model.evaluate(x - e)) / (2 * h)
        assert np.allclose(fd[:, 0], g[:, d], rtol=2e-3, atol=2e-3)
        assert np.allclose(fd[:, 1], g[:, 3 + d], rtol=2e-3, atol=2e-3)


def test_stationary_ddm_solver_and_duplicates():
    import ferreus_rbf_rs_b200 as fb
    kernel, dim, n = 0, 3, 2200
    pts = H.make_points(n, dim, "uniform", seed=31)
    pts = np.concatenate([pts, pts[:25]])                      # exact duplicates are dropped (rbf.rs:1418-1467)
    vals = _values(pts)
    events = []
    model = fb.RBFInterpolator(pts, vals, _settings(kernel, tol=1e-8),
                               params=_params(kernel, solver=fb.config.Solvers.DDM),
                               progress_callback=fb.progress.Progress(lambda ev: events.append(ev)))
    info = model.info()
    assert info["n_points"] == n and info["n_duplicates"] == 25
    assert any(isinstance(e, fb.progress.DuplicatesRemoved) and e.num_duplicates == 25 for e in events)
    assert info["last_residual"] <= 1e-8
    om = _oracle(kernel, pts, vals, 1e-8, solver=0)
    t = np.random.default_rng(3).random((200, dim))
    assert H.rel_l2(np.asarray(model.evaluate(t)).reshape(-1, 1), om.evaluate(t)) <= 1e-7


@pytest.mark.parametrize("kernel,dim,n,naive", [(0, 3, 2400, 100), (2, 3, 600, 4096), (1, 2, 2400, 100), (0, 1, 300, 4096)])
def test_global_trend_matches_oracle(kernel, dim, n, naive):
    """GlobalTrend (global_trend.rs:128-287; rbf.rs:361-371, 477-484, 579-615, 1181-1229, 1272-1298): the kernel
    works in the rotated / scaled space, the polynomial in the original one, gradients are transformed back."""
    import ferreus_rbf_rs_b200 as fb
    from oracle import rbf as orbf
    pts = H.make_points(n, dim, "uniform", seed=61)
    vals = _values(pts)
    tol = 1e-10
    if dim == 3:
        gt, ogt = fb.GlobalTrend.three(25.0, 70.0, 15.0, 3.0, 2.0, 1.0), orbf.GlobalTrend.three(25.0, 70.0, 15.0, 3.0, 2.0, 1.0)
    elif dim == 2:
        gt, ogt = fb.GlobalTrend.two(35.0, 2.5, 1.0), orbf.GlobalTrend.two(35.0, 2.5, 1.0)
    else:
        gt, ogt = fb.GlobalTrend.one(2.0), orbf.GlobalTrend.one(2.0)
    model = fb.RBFInterpolator(pts, vals, _settings(kernel, tol=tol), params=_params(kernel, naive=naive), global_trend=gt)
    s = orbf.InterpolantSettings(kernel, tolerance=tol)
    p = orbf.Params(kernel, solver_type=1, leaf_threshold=128, coarse_threshold=300, naive_solve_threshold=naive,
                    interpolation_order=8, max_points_per_cell=40, epsilon=1e-10)
    om = orbf.RBFInterpolator(pts, vals, s, p, global_trend=ogt)
    # public points are the inverse transform of the transformed points (rbf.rs:579-581): equal up to round-off
    assert np.allclose(model.source_points, om.points, rtol=0, atol=1e-12)
    co = model.coefficients
    assert H.rel_l2(co.point_coefficients, om.point_coefficients) <= 1e-6
    targets = np.random.default_rng(2).random((300, dim)) * (pts.max(0) - pts.min(0)) + pts.min(0)
    got, gg = model.evaluate_with_gradients(targets)
    ref, rg = om.evaluate(targets, True)
    assert H.rel_l2(np.asarray(got).reshape(-1, 1), ref) <= INTERP_TOL
    assert H.rel_l2(gg, rg) <= 1e-6
    # exact (dense) evaluation of the oracle's interpolant: same function
    assert H.rel_l2(np.asarray(got).reshape(-1, 1), om.evaluate_dense(targets)) <= 1e-5
    # persistent evaluator with user extents given in the ORIGINAL space (corner-transformed, rbf.rs:603-615)
    ext = list(np.minimum(pts.min(0), targets.min(0)) - 0.1) + list(np.maximum(pts.max(0), targets.max(0)) + 0.1)
    model.build_evaluator(ext)
    got2 = np.asarray(model.evaluate_targets(targets)).reshape(-1, 1)
    assert H.rel_l2(got2, ref) <= 1e-7
    # the interpolant reproduces the data
    at_src = np.asarray(model.evaluate_at_source()).reshape(-1)
    assert H.rel_l2(at_src, vals) <= 1e-6
    # a trivial trend changes nothing
    if dim == 3 and n <= 1000:
        m0 = fb.RBFInterpolator(pts, vals, _settings(kernel, tol=tol), params=_params(kernel, naive=naive))
        m1 = fb.RBFInterpolator(pts, vals, _settings(kernel, tol=tol), params=_params(kernel, naive=naive),
                                global_trend=fb.GlobalTrend.three(0.0, 0.0, 0.0, 1.0, 1.0, 1.0))
        assert H.rel_l2(np.asarray(m1.evaluate(targets)), np.asarray(m0.evaluate(targets))) <= 1e-10


@pytest.mark.parametrize("trend", [False, True])
def test_save_and_load_model_round_trip(tmp_path, trend):
    """save_model / load_model (rbf.rs:1087-1171): the JSON envelope restores a model that evaluates identically."""
    import json
    import ferreus_rbf_rs_b200 as fb
    pts = H.make_points(1500, 3, "clustered", seed=71)
    vals = np.stack([_values(pts), np.cos(2 * pts[:, 0])], axis=1)
    gt = fb.GlobalTrend.three(10.0, 120.0, 30.0, 2.0, 1.0, 0.5) if trend else None
    model = fb.RBFInterpolator(pts, vals, _settings(2, tol=1e-9), params=_params(2), global_trend=gt)
    path = str(tmp_path / "model.json")
    model.save_model(path)
    doc = json.load(open(path))
    assert doc["format"] == "ferreus_rbf.json" and doc["version"] == 1
    assert doc["points"]["nrows"] == model.info()["n_points"] and doc["points"]["ncols"] == 3
    assert doc["interpolant_settings"]["kernel_type"] == "Cubic" and doc["params"]["solver_type"] == "FGMRES"
    assert (doc["global_trend"] is not None) == trend
    loaded = fb.RBFInterpolator.load_model(path)
    targets = np.random.default_rng(3).random((200, 3)) * (pts.max(0) - pts.min(0)) + pts.min(0)
    a, ga = model.evaluate_with_gradients(targets)
    b, gb = loaded.evaluate_with_gradients(targets)
    assert H.rel_l2(b, a) <= 1e-12 and H.rel_l2(gb, ga) <= 1e-12   # same state; M2L REDs reorder round-off
    assert np.array_equal(loaded.coefficients.point_coefficients, model.coefficients.point_coefficients)
    loaded.build_evaluator()
    assert H.rel_l2(loaded.evaluate_targets(targets), a) <= 1e-5   # another tree (own extents): FMM accuracy at order 8
    doc["version"] = 2
    json.dump(doc, open(path, "w"))
    with pytest.raises(ValueError):
        fb.RBFInterpolator.load_model(path)


@pytest.mark.parametrize("kernel,dim,n", [(0, 3, 2400), (1, 2, 2400)])
def test_absolute_tolerance_fit_matches_oracle(kernel, dim, n):
    """FittingAccuracyType.Absolute (iterative_solvers.rs:57, 137-163): beta and the restart test use the max-norm of the
    residual, the in-loop test the 2-norm estimate |g[j + 1]| un-normalised.  Same stopping iteration as the oracle
    at a loose tolerance (the mixed norms decide where it stops), same interpolant at a tight one."""
    import ferreus_rbf_rs_b200 as fb
    from oracle import rbf as orbf
    ic = fb.interpolant_config
    pts = H.make_points(n, dim, "uniform", seed=131)
    vals = 50.0 * _values(pts)          # |values| well above 1: absolute and relative tolerances differ by that factor
    for tol, interp_tol in ((1e-3, 1e-5), (1e-9, INTERP_TOL)):
        st = ic.InterpolantSettings(ic.RBFKernelType(kernel),
                                    fitting_accuracy=ic.FittingAccuracy(tol, ic.FittingAccuracyType.Absolute))
        model = fb.RBFInterpolator(pts, vals, st, params=_params(kernel))
        s = orbf.InterpolantSettings(kernel, tolerance=tol, tolerance_type=orbf.ABSOLUTE)
        p = orbf.Params(kernel, solver_type=1, leaf_threshold=128, coarse_threshold=300, naive_solve_threshold=100,
                        interpolation_order=8, max_points_per_cell=40, epsilon=1e-10)
        om = orbf.RBFInterpolator(pts, vals, s, p)
        info = model.info()
        assert info["last_residual"] < tol
        assert abs(info["iterations"] - om.iterations) <= 1
        targets = np.random.default_rng(1).random((300, dim)) * (pts.max(0) - pts.min(0)) + pts.min(0)
        got = np.asarray(model.evaluate(targets)).reshape(-1, 1)
        assert H.rel_l2(got, om.evaluate(targets)) <= interp_tol
    # the absolute test is un-normalised: the same tolerance read as Relative stops (much) earlier
    st_rel = ic.InterpolantSettings(ic.RBFKernelType(kernel),
                                    fitting_accuracy=ic.FittingAccuracy(1e-3, ic.FittingAccuracyType.Relative))
    rel_its = fb.RBFInterpolator(pts, vals, st_rel, params=_params(kernel)).info()["iterations"]
    st_abs = ic.InterpolantSettings(ic.RBFKernelType(kernel),
                                    fitting_accuracy=ic.FittingAccuracy(1e-3, ic.FittingAccuracyType.Absolute))
    abs_its = fb.RBFInterpolator(pts, vals, st_abs, params=_params(kernel)).info()["iterations"]
    assert abs_its >= rel_its


@pytest.mark.parametrize("kernel,dim,n", [(0, 3, 2600), (2, 3, 2600), (1, 2, 2600)])
def test_ddm_overlap_order_matches_oracle(kernel, dim, n):
    """domain_decomposition.rs:236-311: the overlap points of a leaf are the nearest internal points of its neighbour
    leaves in ascending point-to-box distance, appended after the internal points.  Domain::factorise then moves the
    special points to the front (domain.rs:219-260); everything else keeps the order, which is compared here
    element by element (test_ddm_hierarchy_bit_exact compares the sets)."""
    import ferreus_rbf_rs_b200 as fb
    from oracle import rbf as orbf
    pts = H.make_points(n, dim, "clustered", seed=141)
    vals = _values(pts)
    model = fb.RBFInterpolator(pts, vals, _settings(kernel, tol=1e-2), params=_params(kernel, order=5, eps=1e-5))
    s = orbf.InterpolantSettings(kernel)
    s.set_basis_size(dim)
    keep = orbf.remove_duplicates(pts, s.kernel())
    ddm = orbf.DDMTree(pts[keep], s, 128, 0.5, 0.125, 300, factorise=False)
    checked = 0
    for li, lvl in enumerate(ddm.levels):
        _, ptr, idx, internal = model.ddm_level(li)
        for d, dom in enumerate(lvl.leaf_domains):
            mine = idx[int(ptr[d]):int(ptr[d + 1])].astype(np.int64).tolist()
            ref = [int(v) for v in dom.idx]
            ok = False
            for rk in range(0, s.basis_size + 1):      # rk special points were moved to the front
                front = set(mine[:rk])
                if len(front) == rk and mine[rk:] == [v for v in ref if v not in front]:
                    ok = True
                    break
            assert ok, f"level {li} domain {d}: point order differs from the oracle's"
            # internal flags follow their points
            k = min(len(dom.mask), len(dom.idx))
            ref_int = {int(v) for v, mk in zip(dom.idx[:k], dom.mask[:k]) if mk}
            assert {v for v, f in zip(mine, internal[int(ptr[d]):int(ptr[d + 1])]) if f} == ref_int
            checked += 1
    assert checked >= 10


def test_indefinite_subdomain_falls_back_like_the_reference():
    """domain.rs:63-68: when the Cholesky factorisation of Q^T A Q fails the reference silently switches to its
    Bunch-Kaufman LBL^T; here the domain is inverted by a pivoted elimination instead.  A negative nugget makes the
    spheroidal kernel matrix indefinite; the fit must solve (K + nugget I) lambda = f all the same."""
    import ferreus_rbf_rs_b200 as fb
    from oracle import kernels as okern
    ic = fb.interpolant_config
    n = 700
    pts = H.make_points(n, 3, "uniform", seed=151)
    vals = _values(pts).reshape(-1, 1)
    st = ic.InterpolantSettings(ic.RBFKernelType.Spheroidal, nugget=-0.4, base_range=0.5, total_sill=0.5)
    model = fb.RBFInterpolator(pts, vals, st)          # n < naive_solve_threshold: one dense domain
    k = okern.Kernel(3, 0.5, 0.5).matrix(pts, pts) - 0.4 * np.eye(n)
    ev = np.linalg.eigvalsh(k)
    assert ev[0] < -1e-3 and ev[-1] > 1e-3             # indefinite: the Cholesky path cannot have been taken
    lam = np.linalg.solve(k, vals)
    assert H.rel_l2(model.coefficients.point_coefficients, lam) <= 1e-8


def test_strided_host_targets_match_a_contiguous_copy():
    """The host-array evaluators gather the caller's rows at any strides: a Fortran-order array and a row-sliced view give
    the results of a contiguous copy (the persistent evaluator bit for bit; the one-shot calls build a tree each, and
    its M2L reductions reorder round-off, which reaches the gradients as up to ~2e-14, see test_gpu_device_eval)."""
    import ferreus_rbf_rs_b200 as fb
    pts = H.make_points(2000, 3, "uniform", seed=161)
    vals = np.stack([_values(pts), np.cos(2 * pts[:, 0])], axis=1)
    gt = fb.GlobalTrend.three(25.0, 70.0, 15.0, 3.0, 2.0, 1.0)
    model = fb.RBFInterpolator(pts, vals, _settings(2, tol=1e-8), params=_params(2), global_trend=gt)
    model.build_evaluator()
    wide = np.random.default_rng(162).random((800, 3)) * 0.98 + 0.01
    for x in (np.asfortranarray(wide), wide[::2]):
        c = np.ascontiguousarray(x)
        assert np.array_equal(model.evaluate_targets(x), model.evaluate_targets(c))
        assert H.rel_l2(model.evaluate(x), model.evaluate(c)) <= 1e-14
        v, g = model.evaluate_with_gradients(x)
        vc, gc = model.evaluate_with_gradients(c)
        assert H.rel_l2(v, vc) <= 1e-14 and H.rel_l2(g, gc) <= 1e-13


@pytest.mark.parametrize("n,naive", [(600, 4096), (2400, 100)])
def test_evaluate_at_source_adds_the_nugget(n, naive):
    """evaluate_at_source(add_nugget=True) (rbf.rs:777-828) adds nugget * lambda to the interpolant at the source points,
    which then reproduces the data: (K + nugget I) lambda + P c = f.  One dense domain, then the DDM solve."""
    import ferreus_rbf_rs_b200 as fb
    nugget, tol = 0.05, 1e-8
    pts = H.make_points(n, 3, "uniform", seed=171)
    vals = np.stack([_values(pts), np.cos(2 * pts[:, 0])], axis=1)
    st = _settings(0, tol=tol, nugget=nugget, drift=fb.interpolant_config.Drift.Linear)
    model = fb.RBFInterpolator(pts, vals, st, params=_params(0, naive=naive))
    lam = model.coefficients.point_coefficients
    plain = model.evaluate_at_source()
    with_nugget = model.evaluate_at_source(add_nugget=True)
    assert H.rel_l2(with_nugget - plain, nugget * lam) <= 1e-12
    assert H.rel_l2(with_nugget, vals) <= 1e-6
