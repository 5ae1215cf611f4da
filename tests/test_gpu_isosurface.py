"""Isosurfaces on the GPU: ferreus_rbf_rs_b200.lattice_isosurface against the numpy restatement of the mesh
specification (tests/isosurface_oracle.py), and RBFInterpolator.extract_isosurfaces(_cuda) against evaluate_cuda on
the lattice, on its own vertices and on the evaluator."""
import numpy as np
import pytest

from tests import helpers as H
from tests import isosurface_oracle as oi

pytestmark = pytest.mark.gpu


def _torch():
    import torch
    return torch


def _cuda(a):
    torch = _torch()
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda")


def _np(t):
    return t.detach().cpu().numpy()


def _gaussians(ext, res, seed):
    rng = np.random.default_rng(seed)
    x = oi.lattice_points(ext, res)
    v = np.zeros(x.shape[0])
    for _ in range(4):
        c = rng.uniform(ext[:3], ext[3:])
        w = rng.uniform(0.2, 0.6)
        v += rng.uniform(-1, 1) * np.exp(-((x - c) ** 2).sum(1) / (w * w))
    return v.reshape(res[2], res[1], res[0])


def _settings(kernel=0, drift=2):
    import ferreus_rbf_rs_b200 as fb
    ic = fb.interpolant_config
    return ic.InterpolantSettings(ic.RBFKernelType(kernel), drift=ic.Drift(drift))


def _sd_model(n, seed, radius=0.5, cols=1, trend=None):
    """signed distance to a sphere (column 1: to a smaller one) from n points in [-1, 1]^3"""
    import ferreus_rbf_rs_b200 as fb
    pts = np.random.default_rng(seed).uniform(-1, 1, (n, 3))
    r = np.linalg.norm(pts, axis=1)
    vals = r - radius if cols == 1 else np.stack([r - radius, r - 0.6 * radius], axis=1)
    return fb.RBFInterpolator(pts, vals, _settings(), global_trend=trend), pts


def _col(v, column):
    v = _np(v)
    return v if v.ndim == 1 else v[:, column]


EXT_IN = [-0.85, -0.8, -0.75, 0.8, 0.85, 0.9]   # inside the points' box: the same tree as evaluate_cuda's


# ------------------------------------------------------------------------------------------------- lattice level
@pytest.mark.parametrize("res,seed", [((2, 2, 2), 1), ((17, 23, 31), 2), ((64, 64, 64), 3)])
def test_lattice_isosurface_matches_the_oracle(res, seed):
    import ferreus_rbf_rs_b200 as fb
    ext = np.array([-1.1, -0.9, -1.0, 1.2, 0.8, 1.05])
    v = _gaussians(ext, res, seed)
    flat = np.sort(v.ravel())
    isos = [0.0, float(np.median(flat)), float(flat[len(flat) // 3]), float(flat[-1]), float(flat[0]),
            float(flat[0]) - 1.0]   # exact ties with lattice values, and a value below them all
    span = float(np.max(ext[3:] - ext[:3]))
    d = _cuda(v)
    for iso in isos:
        rv, rf = oi.extract(v, ext, iso)
        gv, gf = fb.lattice_isosurface(d, ext, iso)
        assert gv.is_cuda and gf.is_cuda and gf.dtype == _torch().int64
        assert np.array_equal(_np(gf), rf), iso
        assert _np(gv).shape == rv.shape
        assert np.abs(_np(gv) - rv).max(initial=0.0) <= 1e-15 * span, iso


def test_lattice_isosurface_of_a_tie_lattice_is_closed():
    import ferreus_rbf_rs_b200 as fb
    ext = [-1.0, -1.0, -1.0, 1.0, 1.0, 1.0]
    res = (24, 24, 24)
    x = oi.lattice_points(ext, res)
    v = np.round(4.0 * np.linalg.norm(x, axis=1)).reshape(24, 24, 24)
    gv, gf = fb.lattice_isosurface(_cuda(v), ext, 2.0)
    rv, rf = oi.extract(v, ext, 2.0)
    assert np.array_equal(_np(gf), rf)
    once, open_edges = oi.edge_use(_np(gf))
    assert once and not open_edges and oi.euler_characteristic(_np(gv), _np(gf)) == 2


def test_lattice_isosurface_rejects_bad_values():
    import ferreus_rbf_rs_b200 as fb
    ext = [0, 0, 0, 1, 1, 1]
    v = _gaussians(np.array(ext, float), (6, 7, 8), 4)
    v[3, 2, 1] = np.nan
    with pytest.raises(ValueError, match="not finite"):
        fb.lattice_isosurface(_cuda(v), ext, 0.0)
    v[3, 2, 1] = 0.0
    with pytest.raises(ValueError):
        fb.lattice_isosurface(_cuda(v), ext, float("inf"))
    with pytest.raises(ValueError):
        fb.lattice_isosurface(_cuda(v), [0, 0, 0, 1, 0, 1], 0.0)
    with pytest.raises(ValueError):
        fb.lattice_isosurface(_cuda(v[:, :, :1]), ext, 0.0)
    fb.lattice_isosurface(_cuda(v), ext, 0.0)


# --------------------------------------------------------------------------------------------------- model level
def test_unrefined_mesh_is_the_lattice_mesh_of_evaluate_cuda():
    model, _ = _sd_model(3000, 11)
    res = (21, 26, 23)
    lat = oi.lattice_points(EXT_IN, res)
    vals = _np(model.evaluate_cuda(_cuda(lat)))
    # isovalues at least 1e-8 away from every lattice value: both evaluations classify every node alike
    isos = []
    for iso in (-0.1, 0.0, 0.15):
        while np.abs(vals - iso).min() < 1e-8:
            iso += 3e-8
        isos.append(iso)
    import ferreus_rbf_rs_b200 as fb
    cell = float(np.max((np.array(EXT_IN[3:]) - EXT_IN[:3]) / (np.array(res) - 1)))
    meshes = model.extract_isosurfaces(isos, EXT_IN, res, refine=False)
    for iso, (v, f, n) in zip(isos, meshes):
        lv, lf = fb.lattice_isosurface(_cuda(vals.reshape(res[2], res[1], res[0])), EXT_IN, iso)
        assert np.array_equal(f, _np(lf))
        assert np.abs(v - _np(lv)).max() <= 1e-9 * cell
        assert n.shape == v.shape


def _check_sphere(model, ext, res, iso, column=0):
    v0, f0, _ = model.extract_isosurfaces(iso, ext, res, column=column, refine=False)[0]
    v, f, n = model.extract_isosurfaces(iso, ext, res, column=column, refine=True)[0]
    assert np.array_equal(f, f0)
    once, open_edges = oi.edge_use(f)
    assert once and not open_edges
    assert oi.euler_characteristic(v, f) == 2
    vmax = np.abs(model.source_values).max()
    err0 = np.abs(_col(model.evaluate_cuda(_cuda(v0)), column) - iso).max()
    err = np.abs(_col(model.evaluate_cuda(_cuda(v)), column) - iso).max()
    assert err <= 1e-8 * vmax, (err, err0)
    assert err < err0
    assert np.allclose(np.linalg.norm(n, axis=1), 1.0, rtol=0, atol=1e-12)
    fn = oi.face_normals(v, f)
    big = np.linalg.norm(fn, axis=1) > 1e-6 * np.median(np.linalg.norm(fn, axis=1))
    assert (np.einsum("ij,ij->i", fn, n[f].sum(axis=1))[big] > 0).all()
    return v, f, n


def test_signed_distance_sphere_through_the_fmm():
    model, _ = _sd_model(6000, 12)          # more points than naive_solve_threshold: DDM fit, FMM evaluation
    v, f, n = _check_sphere(model, EXT_IN, 40, 0.0)
    assert np.abs(np.linalg.norm(v, axis=1) - 0.5).max() < 0.02
    assert (np.einsum("ij,ij->i", n, v) > 0).all()   # outward, along increasing distance
    torch = _torch()
    cv, cf, cn = model.extract_isosurfaces_cuda(0.0, EXT_IN, 40)[0]
    assert cv.is_cuda and cf.dtype == torch.int64 and cn.is_cuda
    assert np.array_equal(_np(cf), f)
    assert np.abs(_np(cv) - v).max() < 1e-12


def test_several_isovalues_in_one_call():
    model, _ = _sd_model(3000, 13)
    isos = [-0.2, 0.0, 0.15]
    together = model.extract_isosurfaces(isos, EXT_IN, (30, 31, 32))
    areas = []
    for iso, (v, f, n) in zip(isos, together):
        v1, f1, n1 = model.extract_isosurfaces([iso], EXT_IN, (30, 31, 32))[0]
        assert np.array_equal(f, f1)
        assert np.abs(v - v1).max() < 1e-12 and np.abs(n - n1).max() < 1e-10
        areas.append(oi.area(v, f))
    assert areas[0] < areas[1] < areas[2]


def test_second_value_column():
    model, _ = _sd_model(3000, 14, cols=2)
    v, f, _ = _check_sphere(model, EXT_IN, 36, 0.0, column=1)
    assert np.abs(np.linalg.norm(v, axis=1) - 0.3).max() < 0.02


def test_global_trend_model_in_user_coordinates():
    import ferreus_rbf_rs_b200 as fb
    gt = fb.GlobalTrend.three(25.0, 70.0, 15.0, 2.0, 1.5, 1.0)
    model, _ = _sd_model(3000, 15, trend=gt)
    res = (27, 25, 29)
    lat = oi.lattice_points(EXT_IN, res)
    vals = _np(model.evaluate_cuda(_cuda(lat)))
    iso = 0.0
    while np.abs(vals - iso).min() < 1e-8:
        iso += 3e-8
    v0, f0, _ = model.extract_isosurfaces(iso, EXT_IN, res, refine=False)[0]
    lv, lf = fb.lattice_isosurface(_cuda(vals.reshape(res[2], res[1], res[0])), EXT_IN, iso)
    assert np.array_equal(f0, _np(lf))
    _check_sphere(model, EXT_IN, res, iso)


def test_extraction_leaves_the_evaluator_unchanged():
    model, _ = _sd_model(3000, 16)
    model.build_evaluator()
    targets = np.random.default_rng(17).uniform(-0.9, 0.9, (500, 3))
    before = np.asarray(model.evaluate_targets(targets)).copy()
    before_cuda = _np(model.evaluate_targets_cuda(_cuda(targets)))
    model.extract_isosurfaces([0.0, 0.1], [-2, -2, -2, 2, 2, 2], 24)
    assert np.array_equal(np.asarray(model.evaluate_targets(targets)), before)
    assert np.array_equal(_np(model.evaluate_targets_cuda(_cuda(targets))), before_cuda)


def test_rejected_arguments_leave_the_model_usable():
    import ferreus_rbf_rs_b200 as fb
    model, pts = _sd_model(1500, 18)
    ref = np.asarray(model.evaluate(pts[:50]))
    ext = [-1, -1, -1, 1, 1, 1]
    bad = [((0.0, ext, 1), {}), ((0.0, ext, (8, 8, 0)), {}), ((0.0, [-1, -1, -1, 1, -1, 1], 8), {}),
           ((0.0, [-1, -1, -1, 1, 1, np.nan], 8), {}), (([], ext, 8), {}), ((np.nan, ext, 8), {}),
           ((0.0, ext, 8), {"column": 1}), ((0.0, ext, 8), {"column": -1}), ((0.0, ext, (1024, 1024, 512)), {}),
           ((0.0, ext, -3), {})]
    for args, kw in bad:
        for fn in (model.extract_isosurfaces, model.extract_isosurfaces_cuda):
            with pytest.raises(ValueError):
                fn(*args, **kw)
    with pytest.raises(ValueError):
        model.extract_isosurfaces(0.0, [-1, -1, 1, 1], 8)
    p2 = H.make_points(500, 2, "uniform", 19)
    m2 = fb.RBFInterpolator(p2, p2[:, 0] - 0.5, _settings())
    with pytest.raises(ValueError, match="3-D"):
        m2.extract_isosurfaces(0.0, ext, 8)
    assert np.array_equal(np.asarray(model.evaluate(pts[:50])), ref)
    assert len(model.extract_isosurfaces(0.0, ext, 8)[0][1]) > 0


def test_c4_albatite_zero_level_set():
    import ferreus_rbf_rs_b200 as fb
    d = np.load(H.__file__.replace("helpers.py", "golden/albatite_SD_points.npz"))
    pts, vals = d["points"], d["values"]
    ic = fb.interpolant_config
    model = fb.RBFInterpolator(pts, vals, ic.InterpolantSettings(ic.RBFKernelType.Cubic))
    lo, hi = np.floor(pts.min(0)), np.ceil(pts.max(0))
    ext = list(lo) + list(hi)
    v, f, n = model.extract_isosurfaces(0.0, ext, 128)[0]
    assert len(f) > 1000
    once, open_edges = oi.edge_use(f)
    assert once
    ends = v[np.array(sorted({e for pair in open_edges for e in pair}), dtype=np.int64)]
    on_box = (np.isclose(ends, lo, rtol=0, atol=1e-9) | np.isclose(ends, hi, rtol=0, atol=1e-9)).any(axis=1)
    assert on_box.all()
    v0, f0, _ = model.extract_isosurfaces(0.0, ext, 128, refine=False)[0]
    assert np.array_equal(f, f0)
    # The points lie inside the lattice box, so the evaluator on that box is the extraction's tree, and the refinement
    # converges on the sign change of the interpolant as that tree evaluates it.  At these UTM coordinates the cubic
    # kernel's sums cancel from ~1e9 and the FMM values jump by up to a few 1e-2 across leaf boundaries, where the exact
    # sum is continuous.  A vertex with a residual above 1e-5 max|value| must sit on such a jump: the evaluator changes
    # sign within 1e-5 along the vertex's edge, by more than the residual, and the exact kernel sum does not jump there.
    model.build_evaluator(ext)
    vmax = np.abs(vals).max()
    r = np.asarray(model.evaluate_targets(v)).ravel()
    big = np.flatnonzero(np.abs(r) > 1e-5 * vmax)
    assert big.size < 0.05 * len(v), big.size
    u = v[big] - v0[big]
    ulen = np.linalg.norm(u, axis=1)
    assert (ulen > 0).all()
    u /= ulen[:, None]
    delta = 1e-5
    fp = np.asarray(model.evaluate_targets(v[big] + delta * u)).ravel()
    fm = np.asarray(model.evaluate_targets(v[big] - delta * u)).ravel()
    jump = np.abs(fp - fm)
    assert (fp * fm < 0).all()
    assert (np.abs(r[big]) <= jump).all()
    assert jump.max() <= 1e-3 * vmax, jump.max()
    co, sp = model.coefficients.point_coefficients[:, 0], model.source_points
    sample = np.arange(big.size)[:: max(1, big.size // 100)]

    def kernel_sum(x):
        return (np.sqrt(((x[:, None, :] - sp[None]) ** 2).sum(-1)) ** 3) @ co

    exact_jump = np.abs(kernel_sum(v[big][sample] + delta * u[sample]) - kernel_sum(v[big][sample] - delta * u[sample]))
    assert (exact_jump < 0.1 * jump[sample]).all()
    one_shot = np.abs(np.asarray(model.evaluate(v)).ravel())
    assert one_shot.max() < np.abs(np.asarray(model.evaluate(v0)).ravel()).max()
    assert np.allclose(np.linalg.norm(n, axis=1), 1.0, rtol=0, atol=1e-12)
