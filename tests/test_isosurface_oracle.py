"""The lattice isosurface specification (tests/isosurface_oracle.py) on analytic fields, and argument checks of the
isosurface entry points that need no device."""
import ctypes as C

import numpy as np
import pytest

from tests import isosurface_oracle as oi

EXT = [-1.3, -1.2, -1.1, 1.25, 1.35, 1.15]


def field(f, ext, res):
    x = oi.lattice_points(ext, res)
    return f(x[:, 0], x[:, 1], x[:, 2]).reshape(res[2], res[1], res[0])


@pytest.mark.parametrize("ext,res", [([0, 0, 0, 1, 1, 1], (2, 2, 2)), (EXT, (17, 23, 31)),
                                     ([-3.7, 1e-3, 12.5, 0.1, 0.3, 99.0], (64, 5, 129))])
def test_lattice_is_linspace_bit_for_bit(ext, res):
    x = oi.lattice_points(ext, res)
    for d in range(3):
        ref = np.linspace(ext[d], ext[3 + d], res[d])
        assert np.array_equal(np.unique(x[:, d]), np.unique(ref))
        assert np.array_equal(oi.axes(ext, res)[d], ref)
    # x fastest, then y, then z
    nx, ny = res[0], res[1]
    assert x[1, 0] > x[0, 0] and x[nx, 1] > x[0, 1] and x[nx * ny, 2] > x[0, 2]


def test_swap_table_uses_120_entries_and_depends_on_parity():
    t = oi.swap_table()
    used = sum(len(oi.triangles_of(m)) for m in range(1, 15)) * 6
    assert used == 120
    assert np.array_equal(t[0], t[3]) and np.array_equal(t[0], t[4])
    assert np.array_equal(t[1], t[2]) and np.array_equal(t[1], t[5])


def test_sphere_is_closed_oriented_and_accurate():
    r = 0.9
    res = (64, 64, 64)
    v = field(lambda x, y, z: np.sqrt(x * x + y * y + z * z) - r, EXT, res)
    verts, faces = oi.extract(v, EXT, 0.0)
    once, open_edges = oi.edge_use(faces)
    assert once and not open_edges
    assert oi.euler_characteristic(verts, faces) == 2
    n = oi.face_normals(verts, faces)
    c = verts[faces].mean(axis=1)
    assert (np.einsum("ij,ij->i", n, c) > 0).all()   # the gradient of |x| - r points outward
    assert abs(oi.area(verts, faces) / (4 * np.pi * r * r) - 1) < 0.01
    assert faces.dtype == np.int64 and np.unique(faces).size == len(verts)


def test_torus_has_euler_characteristic_zero():
    res = (48, 48, 40)
    v = field(lambda x, y, z: (np.sqrt(x * x + y * y) - 0.8) ** 2 + z * z - 0.3 ** 2, EXT, res)
    verts, faces = oi.extract(v, EXT, 0.0)
    once, open_edges = oi.edge_use(faces)
    assert once and not open_edges
    assert oi.euler_characteristic(verts, faces) == 0


def test_linear_field_vertices_lie_on_the_plane():
    res = (19, 21, 23)
    a = np.array([0.3, -0.7, 0.5])
    v = field(lambda x, y, z: a[0] * x + a[1] * y + a[2] * z, EXT, res)
    verts, faces = oi.extract(v, EXT, 0.1)
    assert len(faces) > 0
    assert np.abs(verts @ a - 0.1).max() < 1e-14
    once, open_edges = oi.edge_use(faces)
    assert once   # an open sheet: its boundary is on the lattice's faces
    ends = verts[np.array(sorted({e for pair in open_edges for e in pair}))]
    lo, hi = np.array(EXT[:3]), np.array(EXT[3:])
    assert (np.isclose(ends, lo, rtol=0, atol=1e-12) | np.isclose(ends, hi, rtol=0, atol=1e-12)).any(axis=1).all()


def test_isovalue_outside_the_range_gives_an_empty_mesh():
    v = field(lambda x, y, z: x * x + y, EXT, (9, 10, 11))
    for iso in (v.min() - 1.0, v.max() + 1.0, v.min()):
        verts, faces = oi.extract(v, EXT, iso)
        assert verts.shape == (0, 3) and faces.shape == (0, 3)


def test_ties_are_oriented_consistently():
    # integer values: many nodes equal the isovalue, so some triangles are degenerate
    res = (20, 20, 20)
    v = field(lambda x, y, z: np.round(3.0 * np.sqrt(x * x + y * y + z * z)), EXT, res)
    for iso in (1.0, 2.0, 3.0):
        assert (v == iso).any()
        verts, faces = oi.extract(v, EXT, iso)
        once, open_edges = oi.edge_use(faces)
        assert once and not open_edges
        assert oi.euler_characteristic(verts, faces) == 2


def _lib():
    from ferreus_rbf_rs_b200 import _lib as L
    return L


def test_entry_points_reject_invalid_arguments_without_a_device():
    L = _lib()
    lib = L.lib()
    out = C.c_void_p()
    u64 = C.POINTER(C.c_uint64)
    ext = np.array(EXT)
    res = np.array([4, 4, 4], dtype=np.uint64)
    iso = np.array([0.0])
    bad = C.c_void_p(16)  # never dereferenced: the arguments are rejected first
    assert lib.fr_isosurface_extract(None, L.dptr(ext), res.ctypes.data_as(u64), L.dptr(iso), 1, 0, 1,
                                     C.byref(out)) == L.FB_ERR_INVALID_ARGUMENT
    assert "model" in L.last_error() and not out.value
    assert lib.fr_lattice_isosurface(None, res.ctypes.data_as(u64), L.dptr(ext), 0.0, None,
                                     C.byref(out)) == L.FB_ERR_INVALID_ARGUMENT
    for r, e, msg in (([1, 4, 4], EXT, "resolution"), ([4, 4, 4], [0, 0, 0, 1, 0, 1], "lo < hi"),
                      ([4, 4, 4], [0, 0, 0, 1, np.nan, 1], "finite"), ([1 << 10, 1 << 10, 1 << 9], EXT, "2^28")):
        rr, ee = np.array(r, dtype=np.uint64), np.array(e, dtype=np.float64)
        assert lib.fr_lattice_isosurface(bad, rr.ctypes.data_as(u64), L.dptr(ee), 0.0, None,
                                         C.byref(out)) == L.FB_ERR_INVALID_ARGUMENT
        assert msg in L.last_error(), L.last_error()
    assert lib.fr_lattice_isosurface(bad, res.ctypes.data_as(u64), L.dptr(ext), float("nan"), None,
                                     C.byref(out)) == L.FB_ERR_INVALID_ARGUMENT
    assert lib.fr_lattice_isosurface(bad, None, L.dptr(ext), 0.0, None, C.byref(out)) == L.FB_ERR_INVALID_ARGUMENT
    assert lib.fr_lattice_isosurface(bad, res.ctypes.data_as(u64), L.dptr(ext), 0.0, None,
                                     None) == L.FB_ERR_INVALID_ARGUMENT
    n = C.c_uint64()
    assert lib.fr_isosurface_counts(None, 0, C.byref(n), C.byref(n)) == L.FB_ERR_INVALID_ARGUMENT
    assert lib.fr_isosurface_copy(None, 0, None, None, None) == L.FB_ERR_INVALID_ARGUMENT
    assert lib.fr_isosurface_timing(None, L.dptr(np.zeros(4))) == L.FB_ERR_INVALID_ARGUMENT
    assert lib.fr_isosurface_refine_stats(None, 0, C.byref(n), C.byref(n)) == L.FB_ERR_INVALID_ARGUMENT
    lib.fr_isosurface_free(None)


def test_python_rejects_non_cuda_values():
    torch = pytest.importorskip("torch")
    import ferreus_rbf_rs_b200 as fb
    with pytest.raises(TypeError):
        fb.lattice_isosurface(torch.zeros((4, 4, 4), dtype=torch.float64), EXT, 0.0)
    with pytest.raises(TypeError):
        fb.lattice_isosurface(np.zeros((4, 4, 4)), EXT, 0.0)
