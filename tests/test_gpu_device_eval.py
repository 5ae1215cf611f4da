"""Evaluation from and into torch CUDA tensors (FmmTree.set_weights_cuda / evaluate_cuda,
RBFInterpolator.evaluate_cuda / evaluate_targets_cuda over the fb_tree_*_device / fr_evaluate*_device entry points)
against the host methods on the same tree or model, the oracle, strided views, the caller's stream and a profiler
trace of the copies."""
import ctypes as C
import json

import numpy as np
import pytest

from tests import helpers as H

pytestmark = pytest.mark.gpu

SAME = 1e-14   # host and device run the same kernels; the M2L reductions reorder round-off (~3e-16) run to run
# Gradients after a downward pass differ run to run on the host path alone by up to 2.3e-14 (FmmTree, linear kernel,
# measured on a B200 against a second host call), so the device path is held to 1e-13 there; each value column's
# gradient is compared as one m x dim block, because a component that is nearly zero (d/dy of a function of x and z)
# has a relative error of its own ~1e-13 on either path.  The evaluator's leaf pass is deterministic: SAME.
GRAD_SAME = 1e-13
MATVEC_TOL = 1e-10
INTERP_TOL = 1e-8


def _torch():
    import torch
    return torch


def _cuda(a):
    torch = _torch()
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda")


def _np(t):
    return t.detach().cpu().numpy()


def _per_column(got, ref, tol, block=1):
    """relative L2 of every value column, or of every gradient block of `block` (= dim) columns"""
    got = np.asarray(got).reshape(ref.shape[0], -1)
    ref = np.asarray(ref).reshape(ref.shape[0], -1)
    assert got.shape == ref.shape
    for c in range(0, ref.shape[1], block):
        err = H.rel_l2(got[:, c:c + block], ref[:, c:c + block])
        assert err <= tol, (c // block, err)


def _cloud(n, m, dim, seed):
    pts = H.make_points(n, dim, "uniform", seed=seed)
    rng = np.random.default_rng(seed + 1)
    targets = np.ascontiguousarray(rng.random((m, dim)) * 1.1 - 0.05)
    ext = np.concatenate([np.minimum(pts.min(0), targets.min(0)), np.maximum(pts.max(0), targets.max(0))])
    return pts, targets, ext


# ---------------------------------------------------------------------------------------------- FmmTree
@pytest.mark.parametrize("dim", [1, 2, 3])
@pytest.mark.parametrize("kernel", [0, 1, 2, 3, 7])
def test_fmm_tree_device_matches_host(kernel, dim):
    n, m = {1: (600, 300), 2: (2000, 700), 3: (3000, 900)}[dim]
    pts, targets, ext = _cloud(n, m, dim, seed=10 * kernel + dim)
    tree = H.product_tree(pts, 5, kernel, True, False, 40, 2, 1e-5, extents=ext)
    x = _cuda(targets)
    for nrhs in (1, 3, 8):
        w = np.random.default_rng(nrhs).random((n, nrhs)) - 0.5
        tree.set_weights(w)
        hv, hg = tree.evaluate_with_gradients(w, targets)
        hv2 = tree.evaluate(w, targets)
        wd = _cuda(w)
        tree.set_weights_cuda(wd)
        dv = tree.evaluate_cuda(wd, x)
        dv2, dg = tree.evaluate_cuda(wd, x, gradients=True)
        assert tuple(dv.shape) == hv2.shape and tuple(dg.shape) == hg.shape and dv.device == x.device
        _per_column(_np(dv), hv2, SAME)
        _per_column(_np(dv2), hv, SAME)
        _per_column(_np(dg), hg, GRAD_SAME, dim)


@pytest.mark.parametrize("dim", [1, 2, 3])
def test_fmm_tree_device_matches_oracle(dim):
    n, m = {1: (500, 200), 2: (1500, 400), 3: (2000, 400)}[dim]
    pts, targets, ext = _cloud(n, m, dim, seed=70 + dim)
    w = np.random.default_rng(5).random((n, 2)) - 0.5
    ot = H.oracle_tree(pts, 5, 0, True, False, 40, 2, 1e-5, extents=list(ext))
    ot.set_weights(w)
    rv, rg = ot.evaluate(w, targets, with_gradients=True)
    tree = H.product_tree(pts, 5, 0, True, False, 40, 2, 1e-5, extents=ext)
    tree.set_weights_cuda(_cuda(w))
    dv, dg = tree.evaluate_cuda(_cuda(w), _cuda(targets), gradients=True)
    assert H.rel_l2(_np(dv), rv) <= MATVEC_TOL
    assert H.rel_l2(_np(dg), rg) <= 1e-9


def test_strided_targets_and_weights():
    torch = _torch()
    n, m, dim = 3000, 800, 3
    pts, targets, ext = _cloud(n, m, dim, seed=91)
    w = np.random.default_rng(92).random((n, 3)) - 0.5
    tree = H.product_tree(pts, 5, 2, True, False, 40, 2, 1e-5, extents=ext)
    x = _cuda(targets)
    wd = _cuda(w)
    tree.set_weights_cuda(wd)
    ref_v, ref_g = tree.evaluate_cuda(wd, x, gradients=True)
    wide = torch.zeros((m, dim + 3), dtype=torch.float64, device="cuda")
    wide[:, 2:2 + dim] = x
    views = {"transposed": x.t().contiguous().t(), "column slice": wide[:, 2:2 + dim]}
    for name, xv in views.items():
        assert not xv.is_contiguous(), name
        v, g = tree.evaluate_cuda(wd, xv, gradients=True)
        _per_column(_np(v), _np(ref_v), SAME)
        _per_column(_np(g), _np(ref_g), GRAD_SAME, dim)
    v, g = tree.evaluate_cuda(wd, x[::2], gradients=True)
    rv, rg = tree.evaluate_cuda(wd, x[::2].contiguous(), gradients=True)
    _per_column(_np(v), _np(rv), SAME)
    _per_column(_np(g), _np(rg), GRAD_SAME, dim)
    # non-contiguous weights: column-major, and every other column of a wider matrix
    w_cm = wd.t().contiguous().t()
    w_wide = torch.zeros((n, 6), dtype=torch.float64, device="cuda")
    w_wide[:, ::2] = wd
    tree.set_weights_cuda(wd)
    ref_v0 = tree.evaluate_cuda(wd, x)  # values only: the L2P kernel differs from the one that also forms gradients
    for wv in (w_cm, w_wide[:, ::2]):
        assert not wv.is_contiguous()
        tree.set_weights_cuda(wv)
        v = tree.evaluate_cuda(wv, x)
        _per_column(_np(v), _np(ref_v0), SAME)


def test_targets_equal_to_the_sources_match_evaluate_at_sources():
    n = 4000
    pts = H.make_points(n, 3, "clustered", seed=101)
    w = np.random.default_rng(102).random((n, 2))
    tree = H.product_tree(pts, 5, 0, True, True, 30, 2, 1e-5)
    tree.set_weights(w)
    ref = np.asarray(tree.evaluate_at_sources(w))
    tree.set_weights_cuda(_cuda(w))
    got = tree.evaluate_cuda(_cuda(w), _cuda(pts))
    _per_column(_np(got), ref, SAME)


def test_target_outside_the_tree_is_reported_and_the_tree_stays_usable():
    pts, targets, ext = _cloud(1500, 300, 3, seed=111)
    w = np.random.default_rng(112).random((1500, 1))
    tree = H.product_tree(pts, 5, 0, True, False, 40, 2, 1e-5, extents=ext)
    tree.set_weights(w)
    ref = tree.evaluate(w, targets)
    bad = targets.copy()
    bad[17] = [5.0, 5.0, 5.0]
    with pytest.raises(ValueError) as host_err:
        tree.evaluate(w, bad)
    wd = _cuda(w)
    tree.set_weights_cuda(wd)
    with pytest.raises(ValueError) as dev_err:
        tree.evaluate_cuda(wd, _cuda(bad))
    assert str(dev_err.value) == str(host_err.value)
    assert str(dev_err.value) == "FMM evaluation failed: target point at row 17 lies outside the tree extents"
    _per_column(_np(tree.evaluate_cuda(wd, _cuda(targets))), ref, SAME)


def test_host_and_device_weight_uploads_interleave():
    """host w1, device w2, host w1 on one tree: the host upload after the device one is not mistaken for a repeat"""
    pts, targets, ext = _cloud(3000, 600, 3, seed=121)
    rng = np.random.default_rng(122)
    w1, w2 = rng.random((3000, 2)), rng.random((3000, 2)) - 0.5

    def fresh(w):
        t = H.product_tree(pts, 5, 0, True, False, 40, 2, 1e-5, extents=ext)
        t.set_weights(w)
        return t.evaluate(w, targets)

    f1, f2 = fresh(w1), fresh(w2)
    tree = H.product_tree(pts, 5, 0, True, False, 40, 2, 1e-5, extents=ext)
    tree.set_weights(w1)
    _per_column(tree.evaluate(w1, targets), f1, SAME)
    tree.set_weights_cuda(_cuda(w2))
    _per_column(_np(tree.evaluate_cuda(_cuda(w2), _cuda(targets))), f2, SAME)
    tree.set_weights(w1)
    _per_column(tree.evaluate(w1, targets), f1, SAME)
    # the solver's call shape (targets = sources, same weights twice) after a device upload
    tree.set_weights_cuda(_cuda(w2))
    tree.set_weights(w1)
    _per_column(np.asarray(tree.evaluate(w1, pts)), np.asarray(tree.evaluate_at_sources(w1)), SAME)


# --------------------------------------------------------------------------------------- RBFInterpolator
def _settings(kernel, drift, tol=1e-9, **kw):
    import ferreus_rbf_rs_b200 as fb
    ic = fb.interpolant_config
    return ic.InterpolantSettings(ic.RBFKernelType(kernel), drift=None if drift is None else ic.Drift(drift),
                                  fitting_accuracy=ic.FittingAccuracy(tol, ic.FittingAccuracyType.Relative), **kw)


def _params(kernel, naive=4096):
    import ferreus_rbf_rs_b200 as fb
    cfg = fb.config
    return cfg.Params(fb.interpolant_config.RBFKernelType(kernel), ddm_params=cfg.DDMParams(128, 0.5, 0.125, 300),
                      fmm_params=cfg.FmmParams(8, 40, cfg.FmmCompressionType.ACA, 1e-10, 1024),
                      naive_solve_threshold=naive)


def _values(pts, cols):
    v = np.sin(3 * pts[:, 0]) + pts[:, -1] ** 2
    return v if cols == 1 else np.stack([v, np.cos(2 * pts[:, 0]) - pts[:, 0] * pts[:, -1]], axis=1)


def _host_evaluator(model, targets, gradients):
    """fr_evaluate_targets with a gradient buffer: the evaluator's own gradients"""
    from ferreus_rbf_rs_b200 import _lib
    m = targets.shape[0]
    out = np.zeros((m, model._cols))
    g = np.zeros((m, model._cols * model._dim))
    xr, xc = _lib.strides_of(targets)
    model._check(model._L.fr_evaluate_targets(model._h, _lib.dptr(targets), m, xr, xc, _lib.dptr(out),
                                              _lib.dptr(g) if gradients else None))
    return out, g


def _check_model(model, targets, tol):
    x = _cuda(targets)
    dim = targets.shape[1]
    hv, hg = model.evaluate_with_gradients(targets)
    dv, dg = model.evaluate_cuda(x, gradients=True)
    assert tuple(dv.shape) == np.asarray(hv).shape and tuple(dg.shape) == hg.shape
    _per_column(_np(dv), np.asarray(hv), tol)
    _per_column(_np(dg), hg, max(tol, GRAD_SAME), dim)
    _per_column(_np(model.evaluate_cuda(x)), np.asarray(model.evaluate(targets)), tol)
    model.build_evaluator()
    ev, eg = _host_evaluator(model, targets, True)
    tv, tg = model.evaluate_targets_cuda(x, gradients=True)
    _per_column(_np(tv), ev, tol)
    _per_column(_np(tg), eg, tol, dim)
    _per_column(_np(model.evaluate_targets_cuda(x)), np.asarray(model.evaluate_targets(targets)), tol)


# drift None needs a kernel without a minimum degree (spheroidal); constant / linear / quadratic on the linear kernel
DRIFTS = [(3, 0, {"base_range": 0.6}), (0, 1, {}), (0, 2, {}), (0, 3, {})]


@pytest.mark.parametrize("cols", [1, 2])
@pytest.mark.parametrize("kernel,drift,kw", DRIFTS)
def test_interpolator_device_matches_host(kernel, drift, kw, cols):
    import ferreus_rbf_rs_b200 as fb
    pts = H.make_points(1500, 3, "uniform", seed=131)
    model = fb.RBFInterpolator(pts, _values(pts, cols), _settings(kernel, drift, **kw), params=_params(kernel))
    targets = np.random.default_rng(132).random((700, 3)) * 0.98 + 0.01
    _check_model(model, targets, SAME)


@pytest.mark.parametrize("dim", [2, 3])
def test_interpolator_with_global_trend(dim):
    import ferreus_rbf_rs_b200 as fb
    pts = H.make_points(1800, dim, "uniform", seed=141)
    gt = fb.GlobalTrend.three(25.0, 70.0, 15.0, 3.0, 2.0, 1.0) if dim == 3 else fb.GlobalTrend.two(35.0, 2.5, 1.0)
    for kernel, drift in ((0, 3), (2, 2)):
        model = fb.RBFInterpolator(pts, _values(pts, 2), _settings(kernel, drift), params=_params(kernel),
                                   global_trend=gt)
        targets = np.random.default_rng(142).random((600, dim)) * 0.98 + 0.01
        _check_model(model, targets, 1e-13)


def test_interpolator_device_matches_oracle():
    import ferreus_rbf_rs_b200 as fb
    from oracle import rbf as orbf
    pts = H.make_points(800, 3, "uniform", seed=151)
    vals = _values(pts, 1)
    tol = 1e-10
    model = fb.RBFInterpolator(pts, vals, _settings(0, None, tol=tol), params=_params(0))
    s = orbf.InterpolantSettings(0, tolerance=tol)
    p = orbf.Params(0, solver_type=1, leaf_threshold=128, coarse_threshold=300, naive_solve_threshold=4096,
                    interpolation_order=8, max_points_per_cell=40, epsilon=1e-10)
    om = orbf.RBFInterpolator(pts, vals, s, p)
    targets = np.random.default_rng(152).random((400, 3))
    ref = om.evaluate(targets)
    assert H.rel_l2(_np(model.evaluate_cuda(_cuda(targets))).reshape(-1, 1), ref) <= INTERP_TOL
    model.build_evaluator()
    inside = pts[:300] * 0.999 + 0.0005
    assert H.rel_l2(_np(model.evaluate_targets_cuda(_cuda(inside))).reshape(-1, 1), om.evaluate(inside)) <= 1e-7


def test_loaded_model_through_both_device_methods(tmp_path):
    import ferreus_rbf_rs_b200 as fb
    pts = H.make_points(1200, 3, "clustered", seed=161)
    gt = fb.GlobalTrend.three(10.0, 120.0, 30.0, 2.0, 1.0, 0.5)
    model = fb.RBFInterpolator(pts, _values(pts, 2), _settings(2, 2), params=_params(2), global_trend=gt)
    path = str(tmp_path / "model.json")
    model.save_model(path)
    loaded = fb.RBFInterpolator.load_model(path)
    targets = np.random.default_rng(162).random((500, 3)) * (pts.max(0) - pts.min(0)) + pts.min(0)
    _check_model(loaded, targets, 1e-13)


# ------------------------------------------------------------------------------------------ stream order
def test_stream_order_with_torch_streams():
    torch = _torch()
    import ferreus_rbf_rs_b200 as fb
    pts = H.make_points(2000, 3, "uniform", seed=171)
    model = fb.RBFInterpolator(pts, _values(pts, 1), _settings(0, 2), params=_params(0))
    model.build_evaluator()
    targets = np.random.default_rng(172).random((50_000, 3)) * 0.98 + 0.01
    ref = np.asarray(model.evaluate_targets(targets))
    w = np.random.default_rng(173).random((2000, 2))
    tree = H.product_tree(pts, 5, 0, True, False, 40, 2, 1e-5, extents=np.array([0, 0, 0, 1, 1, 1.0]))
    tree.set_weights(w)
    tref = tree.evaluate(w, targets)
    base = _cuda(targets)
    wd = _cuda(w)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    # targets written by a torch kernel on s, the calls made inside the stream context, results consumed on s
    with torch.cuda.stream(s):
        x = base * 2.0 - base
        out = model.evaluate_targets_cuda(x)
        res = out * 1.0
        tree.set_weights_cuda(wd)
        tres = tree.evaluate_cuda(wd, x) + 0.0
    s.synchronize()
    _per_column(_np(res), ref, SAME)
    _per_column(_np(tres), tref, SAME)
    # the same with long work queued on s ahead of the producer: the library must wait for it
    with torch.cuda.stream(s):
        x2 = torch.empty_like(base)
        torch.cuda._sleep(200_000_000)
        x2.copy_(base)
        out2 = model.evaluate_targets_cuda(x2)
        torch.cuda._sleep(50_000_000)
        res2 = out2 * 1.0
        w2 = torch.empty_like(wd)
        torch.cuda._sleep(50_000_000)
        w2.copy_(wd)
        tree.set_weights_cuda(w2)
        tres2 = tree.evaluate_cuda(w2, x2) + 0.0
    s.synchronize()
    _per_column(_np(res2), ref, SAME)
    _per_column(_np(tres2), tref, SAME)


# --------------------------------------------------------------------------------------------- transfers
def _memcpy_sizes(trace_path):
    """(kind, bytes) of every host <-> device copy in a chrome trace written by torch.profiler"""
    with open(trace_path) as f:
        events = json.load(f)["traceEvents"]
    sizes = []
    for ev in events:
        if ev.get("cat") != "gpu_memcpy":
            continue
        name = ev.get("name", "")
        if "HtoD" in name or "DtoH" in name:
            sizes.append((name, int(ev.get("args", {}).get("bytes", -1))))
    return sizes


def test_device_evaluator_moves_no_bulk_data_between_host_and_device(tmp_path):
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile
    import ferreus_rbf_rs_b200 as fb
    pts = H.make_points(3000, 3, "uniform", seed=181)
    model = fb.RBFInterpolator(pts, _values(pts, 1), _settings(0, 2), params=_params(0))
    model.build_evaluator()
    m = 200_000
    targets = np.random.default_rng(182).random((m, 3)) * 0.98 + 0.01
    x = _cuda(targets)
    model.evaluate_targets_cuda(x)   # warm-up: the first call uploads the polynomial coefficients
    model.evaluate_targets(targets)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        model.evaluate_targets_cuda(x)
        torch.cuda.synchronize()
    dev_trace = str(tmp_path / "device.json")
    prof.export_chrome_trace(dev_trace)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        model.evaluate_targets(targets)
        torch.cuda.synchronize()
    host_trace = str(tmp_path / "host.json")
    prof.export_chrome_trace(host_trace)
    host = _memcpy_sizes(host_trace)
    assert any(b >= m * 3 * 8 for _, b in host), host   # the trace sees the host method's bulk copies
    dev = _memcpy_sizes(dev_trace)
    assert all(0 <= b < 64 * 1024 for _, b in dev), dev


# --------------------------------------------------------------------------------------------- rejections
def test_rejected_tensors_leave_the_model_usable():
    torch = _torch()
    import ferreus_rbf_rs_b200 as fb
    pts = H.make_points(1500, 3, "uniform", seed=191)
    model = fb.RBFInterpolator(pts, _values(pts, 1), _settings(0, 2), params=_params(0))
    model.build_evaluator()
    targets = np.random.default_rng(192).random((300, 3)) * 0.98 + 0.01
    ref = np.asarray(model.evaluate_targets(targets))
    x = _cuda(targets)
    for fn in (model.evaluate_cuda, model.evaluate_targets_cuda):
        with pytest.raises(TypeError):
            fn(x.float())
        with pytest.raises(TypeError):
            fn(x.cpu())
        with pytest.raises(TypeError):
            fn(targets)
        with pytest.raises(ValueError):
            fn(x[:, :2])
    w = np.random.default_rng(193).random((1500, 2))
    tree = H.product_tree(pts, 5, 0, True, False, 40, 2, 1e-5, extents=np.array([0, 0, 0, 1, 1, 1.0]))
    tree.set_weights_cuda(_cuda(w))
    with pytest.raises(ValueError):
        tree.evaluate_cuda(_cuda(w[:, :1]), x)     # not the column count given to set_weights
    with pytest.raises(ValueError):
        tree.set_weights_cuda(_cuda(w[:100]))      # fewer rows than source points
    with pytest.raises(TypeError):
        tree.set_weights_cuda(_cuda(w).float())
    if torch.cuda.device_count() >= 2:
        other = x.to("cuda:1")
        for fn in (model.evaluate_cuda, model.evaluate_targets_cuda):
            with pytest.raises(ValueError):
                fn(other)
        with pytest.raises(ValueError):
            tree.evaluate_cuda(_cuda(w), other)
    _per_column(_np(model.evaluate_targets_cuda(x)), ref, SAME)
    _per_column(_np(model.evaluate_cuda(x)), np.asarray(model.evaluate(targets)), SAME)
    t2 = H.product_tree(pts, 5, 0, True, False, 40, 2, 1e-5, extents=np.array([0, 0, 0, 1, 1, 1.0]))
    t2.set_weights(w)
    _per_column(_np(tree.evaluate_cuda(_cuda(w), x)), t2.evaluate(w, targets), SAME)
