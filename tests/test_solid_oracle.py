"""The solid specification (tests/solid_oracle.py) on analytic fields: closed, with the right topology and the volume of
the piecewise-linear interpolant's sublevel set; and the rejection of a bad side before any device call."""
import ctypes as C

import numpy as np
import pytest

from tests import isosurface_oracle as oi
from tests import solid_oracle as so

EXT = [-1.3, -1.2, -1.1, 1.25, 1.35, 1.15]
BOX = float(np.prod(np.subtract(EXT[3:], EXT[:3])))


def field(f, ext, res):
    x = oi.lattice_points(ext, res)
    return f(x[:, 0], x[:, 1], x[:, 2]).reshape(res[2], res[1], res[0])


def sphere(c, r):
    return lambda x, y, z: np.sqrt((x - c[0]) ** 2 + (y - c[1]) ** 2 + (z - c[2]) ** 2) - r


def torus(x, y, z):
    return (np.sqrt(x * x + y * y) - 0.8) ** 2 + z * z - 0.3 ** 2


def plane(x, y, z):
    return 0.3 * x - 0.7 * y + 0.5 * z


def ties(x, y, z):
    return np.round(4.0 * np.sqrt(x * x + y * y + z * z))


# (field, resolution, isovalue, Euler characteristic of the below solid, of the above solid)
CASES = {
    "sphere inside": (sphere((0.1, 0.0, -0.05), 0.7), (21, 19, 17), 0.0, 2, 4),
    "sphere cut by two faces": (sphere((1.0, 1.1, 0.0), 0.9), (21, 19, 17), 0.0, 2, 2),
    "torus": (torus, (32, 30, 24), 0.0, 0, 2),
    "plane": (plane, (13, 15, 11), 0.1, 2, 2),
    "tie lattice": (ties, (18, 18, 18), 2.0, 2, 4),
}


def closed(faces):
    once, open_edges = oi.edge_use(faces)
    return once and not open_edges


@pytest.mark.parametrize("name", sorted(CASES))
def test_solids_are_closed_with_the_expected_topology(name):
    f, res, iso, chi_below, chi_above = CASES[name]
    v = field(f, EXT, res)
    vols = []
    for side, chi in (("below", chi_below), ("above", chi_above)):
        verts, faces, nvs, nfs = so.extract_solid(v, EXT, iso, side)
        assert closed(faces), side
        assert oi.euler_characteristic(verts, faces) == chi, side
        assert np.unique(faces).size == len(verts)    # every cap node is used
        vols.append(so.volume(verts, faces, EXT[:3]))
    assert vols[0] > 0 and vols[1] > 0
    assert abs(vols[0] + vols[1] - BOX) <= 1e-12 * BOX


def test_surface_part_is_the_isosurface():
    v = field(sphere((1.0, 1.1, 0.0), 0.9), EXT, (21, 19, 17))
    sv, sf = oi.extract(v, EXT, 0.0)
    for side in ("below", "above"):
        verts, faces, nvs, nfs = so.extract_solid(v, EXT, 0.0, side)
        assert (nvs, nfs) == (len(sv), len(sf))
        assert np.array_equal(verts[:nvs], sv)
        assert np.array_equal(faces[:nfs], sf if side == "below" else sf[:, [0, 2, 1]])
        assert (faces[nfs:] >= 0).all()


def test_empty_and_full_sides():
    v = field(sphere((0.0, 0.0, 0.0), 0.5), EXT, (9, 10, 11))
    for iso in (v.min(), v.min() - 1.0, v.max() + 1.0):
        below = so.extract_solid(v, EXT, iso, "below")
        above = so.extract_solid(v, EXT, iso, "above")
        empty, full = (below, above) if iso <= v.min() else (above, below)
        assert empty[0].shape == (0, 3) and empty[1].shape == (0, 3)
        assert so.volume(empty[0], empty[1], EXT[:3]) == 0.0
        assert closed(full[1]) and oi.euler_characteristic(full[0], full[1]) == 2
        assert abs(so.volume(full[0], full[1], EXT[:3]) - BOX) <= 1e-13 * BOX
        # the box surface: 2 triangles per boundary square
        nx, ny, nz = 9, 10, 11
        squares = 2 * ((nx - 1) * (ny - 1) + (nx - 1) * (nz - 1) + (ny - 1) * (nz - 1))
        assert len(full[1]) == 2 * squares
        dx, dy, dz = np.subtract(EXT[3:], EXT[:3])
        assert abs(oi.area(full[0], full[1]) - 2 * (dx * dy + dx * dz + dy * dz)) <= 1e-13 * BOX


@pytest.mark.parametrize("res,seed", [((4, 5, 3), 1), ((6, 5, 7), 2)])
def test_volume_is_the_clip_of_the_piecewise_linear_interpolant(res, seed):
    v = np.random.default_rng(seed).normal(size=(res[2], res[1], res[0]))
    for iso in (-0.4, 0.0, 0.7):
        for side in ("below", "above"):
            verts, faces, _, _ = so.extract_solid(v, EXT, iso, side)
            ref = so.clip_volume(v, EXT, iso, side)
            assert abs(so.volume(verts, faces, EXT[:3]) - ref) <= 1e-12 * max(ref, BOX), (iso, side)


def test_linear_field_gives_the_box_cut_by_a_half_space():
    a = np.array([0.3, 0.7, 0.5])
    v = field(lambda x, y, z: a[0] * x + a[1] * y + a[2] * z, EXT, (11, 13, 9))
    lo, hi = np.array(EXT[:3]), np.array(EXT[3:])
    for c in (-0.6, 0.1, 0.9):
        # volume of {a . x < c} in the box by inclusion-exclusion over its corners (all a > 0)
        exact = 0.0
        for s in range(8):
            bits = np.array([(s >> d) & 1 for d in range(3)])
            corner = np.where(bits == 1, hi, lo)
            exact += (-1) ** bits.sum() * max(0.0, c - a @ corner) ** 3
        exact /= 6 * a.prod()
        verts, faces, _, _ = so.extract_solid(v, EXT, c, "below")
        assert abs(so.volume(verts, faces, EXT[:3]) - exact) <= 1e-12 * BOX, c


def test_volumes_are_monotone_in_the_isovalue():
    v = field(torus, EXT, (20, 21, 16))
    isos = np.linspace(v.min() - 0.1, v.max() + 0.1, 12)
    below = [so.volume(*so.extract_solid(v, EXT, iso, "below")[:2], EXT[:3]) for iso in isos]
    above = [so.volume(*so.extract_solid(v, EXT, iso, "above")[:2], EXT[:3]) for iso in isos]
    assert below[0] == 0.0 and abs(below[-1] - BOX) <= 1e-13 * BOX
    assert (np.diff(below) > 0).all() and (np.diff(above) < 0).all()


def test_cap_table_orients_every_cap_face_out_of_the_box():
    v = np.random.default_rng(3).normal(size=(6, 7, 8))
    lo, hi = np.array(EXT[:3]), np.array(EXT[3:])
    for iso in (-0.3, 0.2):
        for side in ("below", "above"):
            verts, faces, _, nfs = so.extract_solid(v, EXT, iso, side)
            cap = faces[nfs:]
            assert len(cap) > 0
            n = oi.face_normals(verts, cap)
            x = verts[cap]
            out = np.zeros_like(n)
            for d in range(3):
                out[(x[:, :, d] == lo[d]).all(axis=1), d] = -1.0
                out[(x[:, :, d] == hi[d]).all(axis=1), d] = 1.0
            assert (np.abs(out).sum(axis=1) == 1).all()     # every cap face lies in one box face
            assert (np.einsum("ij,ij->i", n, out) > 0).all()


def test_table_is_derived_from_the_unit_square():
    t = so.cap_swap_table()
    used = sum(len(so.clip(m)) for m in range(1, 8)) * 2 * 6
    assert used == 120
    used_entries = np.zeros((2, 8, 2), dtype=bool)
    for m in range(1, 8):
        used_entries[:, m, :len(so.clip(m))] = True
    # the lo and hi face of an axis face opposite ways; the y faces see the (u, v) = (x, z) plane mirrored
    for w in range(3):
        assert (t[2 * w] != t[2 * w + 1])[used_entries].all()
    assert np.array_equal(t[0], t[3]) and np.array_equal(t[0], t[4])
    assert np.array_equal(t[1], t[2]) and np.array_equal(t[1], t[5])


def test_python_rejects_a_bad_side_before_any_device_call():
    import ferreus_rbf_rs_b200 as fb
    from ferreus_rbf_rs_b200 import isosurface as iso
    for bad in ("inside", "Below", 0, None):
        with pytest.raises(ValueError, match="side"):
            fb.lattice_solid(np.zeros((4, 4, 4)), EXT, 0.0, side=bad)
        with pytest.raises(ValueError, match="side"):
            iso.side_code(bad)
    assert iso.side_code("below") == 0 and iso.side_code("above") == 1


def test_entry_points_reject_a_bad_side_without_a_device():
    from ferreus_rbf_rs_b200 import _lib as L
    lib = L.lib()
    out = C.c_void_p()
    u64 = C.POINTER(C.c_uint64)
    ext = np.array(EXT)
    res = np.array([4, 4, 4], dtype=np.uint64)
    isos = np.array([0.0])
    bad = C.c_void_p(16)  # never dereferenced: the arguments are rejected first
    for side in (-1, 2, 7):
        assert lib.fr_lattice_solid(bad, res.ctypes.data_as(u64), L.dptr(ext), 0.0, side, None,
                                    C.byref(out)) == L.FB_ERR_INVALID_ARGUMENT
        assert "side" in L.last_error() and not out.value
        assert lib.fr_isosurface_extract_solid(bad, L.dptr(ext), res.ctypes.data_as(u64), L.dptr(isos), 1, 0, 1, side,
                                               C.byref(out)) == L.FB_ERR_INVALID_ARGUMENT
        assert "side" in L.last_error() and not out.value
    # the other arguments are checked as fr_lattice_isosurface checks them
    r1 = np.array([1, 4, 4], dtype=np.uint64)
    assert lib.fr_lattice_solid(bad, r1.ctypes.data_as(u64), L.dptr(ext), 0.0, 0, None,
                                C.byref(out)) == L.FB_ERR_INVALID_ARGUMENT
    assert "resolution" in L.last_error()
    assert lib.fr_lattice_solid(bad, res.ctypes.data_as(u64), L.dptr(ext), float("nan"), 1, None,
                                C.byref(out)) == L.FB_ERR_INVALID_ARGUMENT
    assert lib.fr_isosurface_extract_solid(None, L.dptr(ext), res.ctypes.data_as(u64), L.dptr(isos), 1, 0, 1, 0,
                                           C.byref(out)) == L.FB_ERR_INVALID_ARGUMENT
    assert "model" in L.last_error()
    n, x = C.c_uint64(), C.c_double()
    assert lib.fr_isosurface_solid_info(None, 0, C.byref(n), C.byref(n), C.byref(x),
                                        C.byref(x)) == L.FB_ERR_INVALID_ARGUMENT
