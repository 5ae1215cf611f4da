"""Solids on the GPU: ferreus_rbf_rs_b200.lattice_solid against the numpy restatement of the specification
(tests/solid_oracle.py), and RBFInterpolator.extract_solids(_cuda) against extract_isosurfaces and against the oracle
solid of the lattice values that evaluate_cuda returns."""
import ctypes as C

import numpy as np
import pytest

from tests import helpers as H
from tests import isosurface_oracle as oi
from tests import solid_oracle as so

pytestmark = pytest.mark.gpu

EXT_IN = [-0.85, -0.8, -0.75, 0.8, 0.85, 0.9]    # inside the points' box, the sphere of radius 0.5 inside it
EXT_CUT = [-0.3, -0.85, -0.8, 0.85, 0.9, 0.2]     # cuts the sphere at x = -0.3 and z = 0.2


def _torch():
    import torch
    return torch


def _cuda(a):
    torch = _torch()
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda")


def _np(t):
    return t.detach().cpu().numpy()


def _box(ext):
    return float(np.prod(np.subtract(ext[3:], ext[:3])))


def _closed(faces):
    once, open_edges = oi.edge_use(faces)
    return once and not open_edges


def _gaussians(ext, res, seed):
    rng = np.random.default_rng(seed)
    x = oi.lattice_points(ext, res)
    v = np.zeros(x.shape[0])
    for _ in range(4):
        c = rng.uniform(ext[:3], ext[3:])
        w = rng.uniform(0.2, 0.6)
        v += rng.uniform(-1, 1) * np.exp(-((x - c) ** 2).sum(1) / (w * w))
    return v.reshape(res[2], res[1], res[0])


def _sd_model(n, seed, radius=0.5, cols=1, trend=None):
    """signed distance to a sphere (column 1: to a smaller one) from n points in [-1, 1]^3"""
    import ferreus_rbf_rs_b200 as fb
    ic = fb.interpolant_config
    pts = np.random.default_rng(seed).uniform(-1, 1, (n, 3))
    r = np.linalg.norm(pts, axis=1)
    vals = r - radius if cols == 1 else np.stack([r - radius, r - 0.6 * radius], axis=1)
    settings = ic.InterpolantSettings(ic.RBFKernelType(0), drift=ic.Drift(2))
    return fb.RBFInterpolator(pts, vals, settings, global_trend=trend), pts


def _away_from(vals, iso):
    """iso moved until it is at least 1e-8 from every lattice value: two evaluations classify every node alike"""
    while np.abs(vals - iso).min() < 1e-8:
        iso += 3e-8
    return iso


def _cap_normals(verts, ext):
    lo, hi = np.array(ext[:3]), np.array(ext[3:])
    n = (verts == hi).astype(float) - (verts == lo).astype(float)
    return n / np.linalg.norm(n, axis=1)[:, None]


# ------------------------------------------------------------------------------------------------- lattice level
@pytest.mark.parametrize("res,seed", [((2, 2, 2), 1), ((17, 23, 31), 2), ((64, 64, 64), 3)])
def test_lattice_solid_matches_the_oracle(res, seed):
    import ferreus_rbf_rs_b200 as fb
    ext = np.array([-1.1, -0.9, -1.0, 1.2, 0.8, 1.05])
    v = _gaussians(ext, res, seed)
    flat = np.sort(v.ravel())
    isos = [0.0, float(np.median(flat)), float(flat[len(flat) // 3]), float(flat[-1]), float(flat[0]),
            float(flat[0]) - 1.0]
    span = float(np.max(ext[3:] - ext[:3]))
    box = _box(ext)
    d = _cuda(v)
    for iso in isos:
        ov, of = fb.lattice_isosurface(d, ext, iso)
        vols = []
        for side in ("below", "above"):
            rv, rf, rnv, rnf = so.extract_solid(v, ext, iso, side)
            g = fb.lattice_solid(d, ext, iso, side=side)
            assert g.vertices.is_cuda and g.faces.dtype == _torch().int64 and g.normals is None
            gv, gf = _np(g.vertices), _np(g.faces)
            assert (g.n_surface_vertices, g.n_surface_faces) == (rnv, rnf)
            assert np.array_equal(gf, rf), (iso, side)
            assert gv.shape == rv.shape
            assert np.abs(gv - rv).max(initial=0.0) <= 1e-15 * span, (iso, side)
            # the isosurface part is the open mesh bit for bit
            assert np.array_equal(gv[:rnv], _np(ov))
            assert np.array_equal(gf[:rnf], _np(of) if side == "below" else _np(of)[:, [0, 2, 1]])
            rvol, rarea = so.volume(rv, rf, ext[:3]), oi.area(rv, rf[:rnf])
            assert abs(g.volume - rvol) <= 1e-12 * box, (iso, side, g.volume, rvol)
            assert abs(g.surface_area - rarea) <= 1e-12 * rarea, (iso, side)
            assert _closed(gf)
            again = fb.lattice_solid(d, ext, iso, side=side)
            assert again.volume == g.volume and again.surface_area == g.surface_area
            vols.append(g.volume)
        assert abs(vols[0] + vols[1] - box) <= 1e-12 * box


def test_lattice_solid_of_a_tie_lattice_is_closed():
    import ferreus_rbf_rs_b200 as fb
    ext = [-1.0, -1.0, -1.0, 1.0, 1.0, 1.0]
    x = oi.lattice_points(ext, (24, 24, 24))
    v = np.round(4.0 * np.linalg.norm(x, axis=1)).reshape(24, 24, 24)
    for side, chi in (("below", 2), ("above", 4)):
        g = fb.lattice_solid(_cuda(v), ext, 2.0, side=side)
        rv, rf, _, _ = so.extract_solid(v, ext, 2.0, side)
        assert np.array_equal(_np(g.faces), rf)
        assert _closed(rf) and oi.euler_characteristic(rv, rf) == chi


def test_solid_info_rejects_an_open_handle():
    import ferreus_rbf_rs_b200 as fb
    from ferreus_rbf_rs_b200 import _lib as L
    from ferreus_rbf_rs_b200.isosurface import Handle, lattice_args
    v = _cuda(_gaussians(np.array([0, 0, 0, 1, 1, 1.0]), (6, 7, 8), 4))
    ext, res = lattice_args([0, 0, 0, 1, 1, 1], (8, 7, 6))
    with Handle() as h:
        assert L.lib().fr_lattice_isosurface(v.data_ptr(), res.ctypes.data_as(C.POINTER(C.c_uint64)), L.dptr(ext), 0.0,
                                             L.cuda_stream(v.device), C.byref(h.h)) == L.FB_OK
        n, x = C.c_uint64(), C.c_double()
        assert L.lib().fr_isosurface_solid_info(h.h, 0, C.byref(n), C.byref(n), C.byref(x),
                                                C.byref(x)) == L.FB_ERR_INVALID_ARGUMENT
    with pytest.raises(ValueError, match="side"):
        fb.lattice_solid(v, [0, 0, 0, 1, 1, 1], 0.0, side="inside")


# --------------------------------------------------------------------------------------------------- model level
@pytest.mark.parametrize("ext", [EXT_IN, EXT_CUT])
def test_sphere_solids_through_the_fmm(ext):
    model, _ = _sd_model(6000, 12)   # more points than naive_solve_threshold: DDM fit, FMM evaluation
    res = (37, 41, 39)
    lat = oi.lattice_points(ext, res)
    vals = _np(model.evaluate_cuda(_cuda(lat)))
    iso = _away_from(vals, 0.0)
    lv = vals.reshape(res[2], res[1], res[0])
    cell = float(np.max((np.array(ext[3:]) - ext[:3]) / (np.array(res) - 1)))
    box = _box(ext)
    for refine in (False, True):
        mv, mf, mn = model.extract_isosurfaces(iso, ext, res, refine=refine)[0]
        vols = []
        for side in ("below", "above"):
            s = model.extract_solids(iso, ext, res, side=side, refine=refine)[0]
            nv, nf = s.n_surface_vertices, s.n_surface_faces
            assert (nv, nf) == (len(mv), len(mf))
            if side == "above" or ext is EXT_CUT:      # the box cuts the solid
                assert len(s.faces) > nf and len(s.vertices) > nv
            assert np.array_equal(s.faces[:nf], mf if side == "below" else mf[:, [0, 2, 1]])
            assert np.abs(s.vertices[:nv] - mv).max() <= 1e-12
            sign = 1.0 if side == "below" else -1.0
            assert np.abs(s.normals[:nv] - sign * mn).max() <= 1e-10
            assert np.abs(s.normals[nv:] - _cap_normals(s.vertices[nv:], ext)).max(initial=0.0) <= 1e-15
            assert _closed(s.faces), (refine, side)
            assert abs(so.volume(s.vertices, s.faces, ext[:3]) - s.volume) <= 1e-12 * box
            assert abs(oi.area(s.vertices, s.faces[:nf]) - s.surface_area) <= 1e-12 * s.surface_area
            if not refine:
                rv, rf, _, _ = so.extract_solid(lv, ext, iso, side)
                assert np.array_equal(s.faces, rf)
                assert np.array_equal(s.vertices[nv:], rv[nv:])   # cap nodes: exact lattice coordinates
                assert np.abs(s.vertices - rv).max() <= 1e-9 * cell
                # the lattice values of the extraction's tree and of evaluate_cuda's agree to rounding
                rvol = so.volume(rv, rf, ext[:3])
                print(f"{ext} {side}: volume {s.volume!r}, oracle of evaluate_cuda's lattice {rvol!r}")
                assert abs(s.volume - rvol) <= 1e-12 * box, (s.volume, rvol)
            vols.append(s.volume)
        assert abs(vols[0] + vols[1] - box) <= 1e-12 * box


def test_sphere_volume_at_96():
    model, _ = _sd_model(6000, 12)
    s = model.extract_solids(0.0, EXT_IN, 96)[0]
    ref = 4.0 / 3.0 * np.pi * 0.5 ** 3
    err = s.volume / ref - 1.0
    print(f"volume of {{f < 0}} at 96^3: {s.volume:.9f}, 4/3 pi r^3 = {ref:.9f}, relative error {err:.3e}")
    assert _closed(s.faces)
    assert abs(err) < 0.01
    c = _torch()
    sc = model.extract_solids_cuda(0.0, EXT_IN, 96)[0]
    assert sc.vertices.is_cuda and sc.faces.dtype == c.int64 and sc.normals.is_cuda
    assert np.array_equal(_np(sc.faces), s.faces)
    assert abs(sc.volume - s.volume) <= 1e-12 * s.volume


def test_several_isovalues_and_a_second_column():
    model, _ = _sd_model(3000, 13, cols=2)
    isos = [-0.2, 0.0, 0.15, 0.3]
    above = model.extract_solids(isos, EXT_IN, (30, 31, 32), side="above")
    below = model.extract_solids(isos, EXT_IN, (30, 31, 32), side="below")
    va, vb = [s.volume for s in above], [s.volume for s in below]
    assert all(_closed(s.faces) for s in above + below)
    assert (np.diff(va) < 0).all() and (np.diff(vb) > 0).all()
    for a, b in zip(va, vb):
        assert abs(a + b - _box(EXT_IN)) <= 1e-12 * _box(EXT_IN)
    one = model.extract_solids([0.15], EXT_IN, (30, 31, 32), side="above")[0]
    assert np.array_equal(one.faces, above[2].faces)
    c1 = model.extract_solids(0.0, EXT_IN, (30, 31, 32), column=1)[0]
    assert _closed(c1.faces) and 0 < c1.volume < vb[1]


def test_global_trend_model_caps_in_user_coordinates():
    import ferreus_rbf_rs_b200 as fb
    gt = fb.GlobalTrend.three(25.0, 70.0, 15.0, 2.0, 1.5, 1.0)
    model, _ = _sd_model(3000, 15, trend=gt)
    res = (27, 25, 29)
    lat = oi.lattice_points(EXT_CUT, res)
    vals = _np(model.evaluate_cuda(_cuda(lat)))
    iso = _away_from(vals, 0.0)
    for side in ("below", "above"):
        s0 = model.extract_solids(iso, EXT_CUT, res, side=side, refine=False)[0]
        rv, rf, _, _ = so.extract_solid(vals.reshape(res[2], res[1], res[0]), EXT_CUT, iso, side)
        assert np.array_equal(s0.faces, rf)
        assert np.array_equal(s0.vertices[s0.n_surface_vertices:], rv[s0.n_surface_vertices:])
        s = model.extract_solids(iso, EXT_CUT, res, side=side)[0]
        assert np.array_equal(s.faces, s0.faces) and _closed(s.faces)
        n = s.normals[s.n_surface_vertices:]
        assert np.allclose(np.linalg.norm(s.normals, axis=1), 1.0, rtol=0, atol=1e-12)
        centre = 0.5 * (np.array(EXT_CUT[:3]) + EXT_CUT[3:])
        assert (np.einsum("ij,ij->i", n, s.vertices[s.n_surface_vertices:] - centre) > 0).all()   # out of the box


def test_rejected_arguments_leave_the_model_usable():
    model, pts = _sd_model(1500, 18)
    ref = np.asarray(model.evaluate(pts[:50]))
    ext = [-1, -1, -1, 1, 1, 1]
    for fn in (model.extract_solids, model.extract_solids_cuda):
        for bad in ("inside", 1, None):
            with pytest.raises(ValueError, match="side"):
                fn(0.0, ext, 8, side=bad)
        for args, kw in (((0.0, ext, 1), {}), ((np.nan, ext, 8), {}), ((0.0, ext, 8), {"column": 1}),
                         ((0.0, [-1, -1, -1, 1, -1, 1], 8), {})):
            with pytest.raises(ValueError):
                fn(*args, side="above", **kw)
    assert np.array_equal(np.asarray(model.evaluate(pts[:50])), ref)
    s = model.extract_solids(0.0, ext, 8, side="above")[0]
    assert len(s.faces) > 0 and _closed(s.faces)


def test_c4_albatite_zero_level_set_is_closed():
    import ferreus_rbf_rs_b200 as fb
    d = np.load(H.__file__.replace("helpers.py", "golden/albatite_SD_points.npz"))
    pts, vals = d["points"], d["values"]
    ic = fb.interpolant_config
    model = fb.RBFInterpolator(pts, vals, ic.InterpolantSettings(ic.RBFKernelType.Cubic))
    lo, hi = np.floor(pts.min(0)), np.ceil(pts.max(0))
    ext = list(lo) + list(hi)
    box = _box(ext)
    vols = []
    for side in ("below", "above"):
        s = model.extract_solids(0.0, ext, 128, side=side)[0]
        assert len(s.faces) > 1000 and _closed(s.faces)
        assert 0 < s.volume < box
        vols.append(s.volume)
    print(f"C4 at 128^3: volume below {vols[0]:.6e}, above {vols[1]:.6e}, box {box:.6e}")
    assert abs(vols[0] + vols[1] - box) <= 1e-9 * box
