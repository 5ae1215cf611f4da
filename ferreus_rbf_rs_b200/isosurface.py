"""Isosurface meshes of lattices and of fitted 3-D interpolants (fr_isosurface_* / fr_lattice_isosurface,
include/ferreus_rbf_b200.h).  The meshes are built and held on the GPU; this module reads them out of the handle."""
import ctypes as C
from collections import namedtuple

import numpy as np

from . import _lib

_u64p = C.POINTER(C.c_uint64)


def lattice_args(extents, resolution):
    """extents [x0, y0, z0, x1, y1, z1] and resolution (an int or (nx, ny, nz)) as the C arrays; the library validates
    the values"""
    ext = np.ascontiguousarray(np.asarray(extents, dtype=np.float64).ravel())
    if ext.size != 6:
        raise ValueError("extents must be [x0, y0, z0, x1, y1, z1]")
    res = [resolution] * 3 if np.ndim(resolution) == 0 else list(resolution)
    if len(res) != 3:
        raise ValueError("resolution must be an int or a 3-tuple")
    # a negative count cannot be a uint64: pass 0, which the library rejects with the other counts below 2
    return ext, np.array([max(int(r), 0) for r in res], dtype=np.uint64)


Solid = namedtuple("Solid", "vertices faces normals volume surface_area n_surface_vertices n_surface_faces")
Solid.__doc__ = """A level set closed at the lattice box into a solid: vertices (V, 3) float64, faces (F, 3) int64 pointing out of
the solid, normals (V, 3) float64 or None; the first n_surface_vertices / n_surface_faces rows are the isosurface, the
rest the caps on the box faces.  volume is the enclosed volume, surface_area the area of the isosurface faces."""


def side_code(side):
    """0 for "below" (the region {f < iso}, the inside of a signed distance), 1 for "above" ({f >= iso})"""
    if isinstance(side, str) and side in ("below", "above"):
        return 0 if side == "below" else 1
    raise ValueError(f'side must be "below" or "above", not {side!r}')


def check(rc):
    if rc != _lib.FB_OK:
        raise (ValueError if rc == _lib.FB_ERR_INVALID_ARGUMENT else RuntimeError)(_lib.last_error())


class Handle:
    """An fr_isosurface handle, freed when the `with` block ends."""

    def __init__(self):
        self.h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        if self.h.value:
            _lib.lib().fr_isosurface_free(self.h)
            self.h = C.c_void_p()

    def mesh(self, which, normals, device=None):
        """(vertices (V, 3) float64, faces (F, 3) int64, normals (V, 3) float64 or None): numpy arrays, or torch
        tensors on `device`"""
        L = _lib.lib()
        nv, nf = C.c_uint64(), C.c_uint64()
        check(L.fr_isosurface_counts(self.h, which, C.byref(nv), C.byref(nf)))
        nv, nf = nv.value, nf.value
        if device is None:
            v, f = np.empty((nv, 3)), np.empty((nf, 3), dtype=np.int64)
            nr = np.empty((nv, 3)) if normals else None
            ptr = lambda a: a.ctypes.data if a is not None and a.size else None  # noqa: E731
        else:
            import torch
            v = torch.empty((nv, 3), dtype=torch.float64, device=device)
            f = torch.empty((nf, 3), dtype=torch.int64, device=device)
            nr = torch.empty((nv, 3), dtype=torch.float64, device=device) if normals else None
            ptr = lambda a: a.data_ptr() if a is not None and a.numel() else None  # noqa: E731
        check(L.fr_isosurface_copy(self.h, which, ptr(v), ptr(f), ptr(nr)))
        return v, f, nr

    def timing(self):
        """milliseconds of lattice evaluation (tree included), extraction, refinement, normals"""
        ms = np.zeros(4)
        check(_lib.lib().fr_isosurface_timing(self.h, _lib.dptr(ms)))
        return [float(x) for x in ms]

    def solid(self, which, normals, device=None):
        """the Solid `which` of a handle of solids"""
        v, f, nr = self.mesh(which, normals, device)
        nv, nf, vol, area = C.c_uint64(), C.c_uint64(), C.c_double(), C.c_double()
        check(_lib.lib().fr_isosurface_solid_info(self.h, which, C.byref(nv), C.byref(nf), C.byref(vol), C.byref(area)))
        return Solid(v, f, nr, vol.value, area.value, nv.value, nf.value)

    def refine_stats(self, which):
        """(trial points evaluated, iterations of the slowest vertex) of the refinement of surface `which`"""
        ev, it = C.c_uint64(), C.c_uint64()
        check(_lib.lib().fr_isosurface_refine_stats(self.h, which, C.byref(ev), C.byref(it)))
        return ev.value, it.value


def lattice_isosurface(values, extents, isovalue):
    """Mesh of the level set `isovalue` of lattice values: a float64 CUDA tensor of shape (nz, ny, nx) over the lattice
    of `extents` [x0, y0, z0, x1, y1, z1] (node (i, j, k) at np.linspace of each axis).  Returns (vertices (V, 3)
    float64, faces (F, 3) int64) as CUDA tensors on the values' device; vertices lie on the lattice edges at the linear
    interpolation of the values.  Ordered on torch's current stream, returns once the mesh is complete."""
    import torch
    if not isinstance(values, torch.Tensor) or not values.is_cuda or values.dtype != torch.float64 or values.dim() != 3:
        raise TypeError("Expected a 3D float64 CUDA tensor (nz, ny, nx) for values")
    v = values.contiguous()
    nz, ny, nx = v.shape
    ext, res = lattice_args(extents, (nx, ny, nz))
    with torch.cuda.device(v.device), Handle() as h:
        check(_lib.lib().fr_lattice_isosurface(v.data_ptr(), res.ctypes.data_as(_u64p), _lib.dptr(ext),
                                               float(isovalue), _lib.cuda_stream(v.device), C.byref(h.h)))
        verts, faces, _ = h.mesh(0, False, v.device)
    return verts, faces


def lattice_solid(values, extents, isovalue, *, side="below"):
    """The level set `isovalue` of lattice values (as lattice_isosurface) closed at the lattice box into the solid
    {f < isovalue} (side "below") or {f >= isovalue} ("above").  Returns a Solid of CUDA tensors on the values' device,
    with normals None; a side with no node gives no faces and volume 0, a side with every node the box."""
    sd = side_code(side)
    import torch
    if not isinstance(values, torch.Tensor) or not values.is_cuda or values.dtype != torch.float64 or values.dim() != 3:
        raise TypeError("Expected a 3D float64 CUDA tensor (nz, ny, nx) for values")
    v = values.contiguous()
    nz, ny, nx = v.shape
    ext, res = lattice_args(extents, (nx, ny, nz))
    with torch.cuda.device(v.device), Handle() as h:
        check(_lib.lib().fr_lattice_solid(v.data_ptr(), res.ctypes.data_as(_u64p), _lib.dptr(ext), float(isovalue), sd,
                                          _lib.cuda_stream(v.device), C.byref(h.h)))
        return h.solid(0, False, v.device)
