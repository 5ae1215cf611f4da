"""Mirror of the reference class ``ferreus_rbf.RBFInterpolator`` over the C ABI of include/ferreus_rbf_b200.h
(py_ferreus_rbf/src/python_bindings.rs:696-930).  All compute is in libferreus_b200.so."""
import ctypes as C
import json

import numpy as np

from . import _lib
from .config import Params
from .interpolant_config import InterpolantSettings
from .progress import DuplicatesRemoved, Message, SolverIteration


class GlobalTrend:
    """Mirror of ``ferreus_rbf.GlobalTrend`` (py_ferreus_rbf/ferreus_rbf/__init__.pyi:21-159; global_trend.rs:36-126):
    anisotropy by rotation and axis ratios about the centroid of the points; angles in degrees."""

    def __init__(self, dim, angles, ratios):
        self.dim, self.angles, self.ratios = int(dim), [float(a) for a in angles], [float(r) for r in ratios]

    @classmethod
    def one(cls, major_ratio):
        return cls(1, [], [major_ratio])

    @classmethod
    def two(cls, rotation_angle, major_ratio, minor_ratio):
        return cls(2, [rotation_angle], [major_ratio, minor_ratio])

    @classmethod
    def three(cls, dip, dip_direction, pitch, major_ratio, semi_major_ratio, minor_ratio):
        return cls(3, [dip, dip_direction, pitch], [major_ratio, semi_major_ratio, minor_ratio])

    def _c(self):
        t = _lib.FrGlobalTrend()
        t.dim = self.dim
        for i, a in enumerate(self.angles):
            t.angles[i] = a
        for i, r in enumerate(self.ratios):
            t.ratios[i] = r
        return t


class Coefficients:
    def __init__(self, point_coefficients, poly_coefficients):
        self.point_coefficients = point_coefficients
        self.poly_coefficients = poly_coefficients


def _one_col(a):
    """mat_to_numpy: a single value column comes back 1-D (python_bindings.rs:81-99)"""
    return a[:, 0].copy() if a.ndim == 2 and a.shape[1] == 1 else a


def _points2d(obj, what):
    if not isinstance(obj, np.ndarray) or obj.dtype != np.float64 or obj.ndim != 2:
        raise TypeError(f"Expected a 2D float64 array for {what}")
    return obj


class RBFInterpolator:
    """RBFInterpolator(points, values, interpolant_settings, *, params=None, global_trend=None,
    progress_callback=None) -> fr_fit"""

    def __init__(self, points, values, interpolant_settings, *, params=None, global_trend=None,
                 progress_callback=None):
        pts = _points2d(points, "points")
        if not isinstance(values, np.ndarray) or values.dtype != np.float64 or values.ndim not in (1, 2):
            raise TypeError("Expected a 1D/2D float64 array for values")
        vals = values[:, None] if values.ndim == 1 else values
        if vals.shape[0] != pts.shape[0]:
            raise ValueError("points and values must have the same number of rows")
        s: InterpolantSettings = interpolant_settings
        L = _lib.lib()
        cs = _lib.FrSettings()
        L.fr_settings_default(int(s.kernel_type), C.byref(cs))
        cs.drift = -1 if s.drift is None else int(s.drift)
        cs.spheroidal_order = int(s.spheroidal_order)
        cs.nugget, cs.base_range, cs.total_sill = s.nugget, s.base_range, s.total_sill
        cs.tolerance = s.fitting_accuracy.tolerance
        cs.tolerance_type = int(s.fitting_accuracy.tolerance_type)
        p: Params = params if params is not None else Params(s.kernel_type)
        cp = _lib.FrParams()
        L.fr_params_default(int(s.kernel_type), C.byref(cp))
        cp.solver_type = int(p.solver_type)
        cp.leaf_threshold = p.ddm_params.leaf_threshold
        cp.overlap_quota = p.ddm_params.overlap_quota
        cp.coarse_ratio = p.ddm_params.coarse_ratio
        cp.coarse_threshold = p.ddm_params.coarse_threshold
        cp.interpolation_order = p.fmm_params.interpolation_order
        cp.max_points_per_cell = p.fmm_params.max_points_per_cell
        cp.compression_type = int(p.fmm_params.compression_type)
        cp.epsilon = p.fmm_params.epsilon
        cp.eval_chunk_size = p.fmm_params.eval_chunk_size
        cp.naive_solve_threshold = p.naive_solve_threshold
        cp.test_unique = int(p.test_unique)
        self.params = p
        self.interpolant_settings = s
        self._progress = progress_callback

        def _cb(ev_ptr, _user):
            if self._progress is None:
                return
            ev = ev_ptr.contents
            if ev.kind == 1:
                self._progress._emit(SolverIteration(ev.iter, ev.residual, ev.progress))
            elif ev.kind == 0:
                self._progress._emit(DuplicatesRemoved(ev.iter))
            else:
                self._progress._emit(Message(ev.message.decode() if ev.message else ""))

        self._cb = _lib.FR_PROGRESS_CB(_cb)
        self._L = L
        self._h = C.c_void_p()
        pr, pc = _lib.strides_of(pts)
        vr, vc = _lib.strides_of(vals)
        ct = global_trend._c() if global_trend is not None else None
        rc = L.fr_fit_trend(_lib.dptr(pts), pts.shape[0], pts.shape[1], pr, pc, _lib.dptr(vals), vals.shape[1], vr, vc,
                            C.byref(cs), C.byref(cp), C.byref(ct) if ct is not None else None, self._cb, None,
                            C.byref(self._h))
        if rc != _lib.FB_OK:
            self._h = C.c_void_p()
            raise (ValueError if rc == _lib.FB_ERR_INVALID_ARGUMENT else RuntimeError)(_lib.last_error())
        info = self.info()
        self._n, self._cols, self._m, self._dim = info["n_points"], info["n_cols"], info["basis_size"], info["dim"]

    # ---- save_model / load_model (rbf.rs:1087-1171) ----------------------------------------------
    # The reference writes `serde_json` of the struct behind a flattened envelope {format, version, ...fields}
    # (rbf.rs:1469-1488).  Field names and enum variant names below are the reference's (rbf.rs:266-302,
    # interpolant_config.rs:18-218, config.rs:42-262, global_trend.rs:128-132).  faer 0.23.2's `Mat` (un-vendored
    # dependency, Cargo.lock:275-278) serialises as {"nrows", "ncols", "data": [row-major elements]} (faer's serde
    # implementation for MatRef); that layout is restated here without a fixture from the reference to pin it.
    _JSON_FORMAT_NAME = "ferreus_rbf.json"
    _JSON_VERSION = 1

    @staticmethod
    def _mat(a):
        a = np.atleast_2d(np.asarray(a, dtype=np.float64))
        return {"nrows": int(a.shape[0]), "ncols": int(a.shape[1]), "data": [float(v) for v in a.ravel(order="C")]}

    @staticmethod
    def _unmat(d):
        return np.asarray(d["data"], dtype=np.float64).reshape(int(d["nrows"]), int(d["ncols"]))

    def save_model(self, path):
        st = _lib.FrModelState()
        self._check(self._L.fr_get_state(self._h, C.byref(st)))
        dim, h = self._dim, self._dim + 1
        drift = ["None", "Constant", "Linear", "Quadratic"][st.settings.drift]
        sph = {3: "Three", 5: "Five", 7: "Seven", 9: "Nine"}[st.settings.spheroidal_order]
        co = self.coefficients
        vals = np.asarray(self.source_values, dtype=np.float64)
        trend = None
        if st.has_trend:
            trend = {"affine_transform": self._mat(np.array(st.affine_transform[: h * h]).reshape(h, h)),
                     "inverse_transform": self._mat(np.array(st.inverse_transform[: h * h]).reshape(h, h))}
        p = st.params
        doc = {
            "format": self._JSON_FORMAT_NAME, "version": self._JSON_VERSION,
            "points": self._mat(self.source_points),
            "point_values": self._mat(vals.reshape(self._n, self._cols)),
            "coefficients": {"point_coefficients": self._mat(co.point_coefficients),
                             "poly_coefficients": None if co.poly_coefficients is None else self._mat(co.poly_coefficients)},
            "interpolant_settings": {
                "kernel_type": ["Linear", "ThinPlateSpline", "Cubic", "Spheroidal"][st.settings.kernel_type],
                "spheroidal_order": sph, "drift": drift, "nugget": st.settings.nugget,
                "base_range": st.settings.base_range, "total_sill": st.settings.total_sill,
                "basis_size": st.basis_size, "polynomial_degree": st.polynomial_degree,
                "fitting_accuracy": {"tolerance": st.settings.tolerance,
                                     "tolerance_type": ["Relative", "Absolute"][st.settings.tolerance_type]}},
            "translation_factor": [st.translation_factor[d] for d in range(dim)] if st.basis_size else [],
            "scale_factor": [st.scale_factor[d] for d in range(dim)] if st.basis_size else [],
            "params": {
                "solver_type": ["DDM", "FGMRES"][p.solver_type],
                "ddm_params": {"leaf_threshold": p.leaf_threshold, "overlap_quota": p.overlap_quota,
                               "coarse_ratio": p.coarse_ratio, "coarse_threshold": p.coarse_threshold},
                "fmm_params": {"interpolation_order": p.interpolation_order,
                               "max_points_per_cell": p.max_points_per_cell,
                               "compression_type": ["None", "SVD", "ACA"][p.compression_type],
                               "epsilon": p.epsilon, "eval_chunk_size": p.eval_chunk_size},
                "naive_solve_threshold": p.naive_solve_threshold, "test_unique": bool(p.test_unique)},
            "global_trend": trend,
        }
        with open(path, "w") as f:
            json.dump(doc, f, indent=2)

    @staticmethod
    def load_model(path, progress_callback=None):
        with open(path) as f:
            doc = json.load(f)
        if doc.get("format") != RBFInterpolator._JSON_FORMAT_NAME:
            raise ValueError(f"{path}: format mismatch: found {doc.get('format')!r}, "
                             f"expected {RBFInterpolator._JSON_FORMAT_NAME!r}")
        if doc.get("version") != RBFInterpolator._JSON_VERSION:
            raise ValueError(f"{path}: version mismatch: found {doc.get('version')!r}, "
                             f"expected {RBFInterpolator._JSON_VERSION}")
        from . import config as cfg
        from . import interpolant_config as ic
        un = RBFInterpolator._unmat
        pts = np.ascontiguousarray(un(doc["points"]))
        vals = np.ascontiguousarray(un(doc["point_values"]))
        pc = np.ascontiguousarray(un(doc["coefficients"]["point_coefficients"]))
        poly_d = doc["coefficients"].get("poly_coefficients")
        poly = np.ascontiguousarray(un(poly_d)) if poly_d is not None else None
        s, p = doc["interpolant_settings"], doc["params"]
        st = _lib.FrModelState()
        st.settings.kernel_type = ["Linear", "ThinPlateSpline", "Cubic", "Spheroidal"].index(s["kernel_type"])
        st.settings.drift = ["None", "Constant", "Linear", "Quadratic"].index(s["drift"])
        st.settings.spheroidal_order = {"Three": 3, "Five": 5, "Seven": 7, "Nine": 9}[s["spheroidal_order"]]
        st.settings.nugget, st.settings.base_range, st.settings.total_sill = s["nugget"], s["base_range"], s["total_sill"]
        st.settings.tolerance = s["fitting_accuracy"]["tolerance"]
        st.settings.tolerance_type = ["Relative", "Absolute"].index(s["fitting_accuracy"]["tolerance_type"])
        st.params.solver_type = ["DDM", "FGMRES"].index(p["solver_type"])
        d, fp = p["ddm_params"], p["fmm_params"]
        st.params.leaf_threshold, st.params.overlap_quota = d["leaf_threshold"], d["overlap_quota"]
        st.params.coarse_ratio, st.params.coarse_threshold = d["coarse_ratio"], d["coarse_threshold"]
        st.params.interpolation_order, st.params.max_points_per_cell = fp["interpolation_order"], fp["max_points_per_cell"]
        st.params.compression_type = ["None", "SVD", "ACA"].index(fp["compression_type"])
        st.params.epsilon, st.params.eval_chunk_size = fp["epsilon"], fp["eval_chunk_size"]
        st.params.naive_solve_threshold, st.params.test_unique = p["naive_solve_threshold"], int(p["test_unique"])
        st.basis_size, st.polynomial_degree = s["basis_size"], s["polynomial_degree"]
        for i, v in enumerate(doc.get("translation_factor") or []):
            st.translation_factor[i] = v
        for i, v in enumerate(doc.get("scale_factor") or []):
            st.scale_factor[i] = v
        gt = doc.get("global_trend")
        st.has_trend = 0
        if gt is not None:
            st.has_trend = 1
            a, ai = un(gt["affine_transform"]).ravel(), un(gt["inverse_transform"]).ravel()
            for i in range(a.size):
                st.affine_transform[i], st.inverse_transform[i] = a[i], ai[i]
        self = RBFInterpolator.__new__(RBFInterpolator)
        L = _lib.lib()
        self._L, self._h, self._progress = L, C.c_void_p(), progress_callback
        self._cb = _lib.FR_PROGRESS_CB(lambda ev, user: None)
        rc = L.fr_model_restore(_lib.dptr(pts), pts.shape[0], pts.shape[1], _lib.dptr(vals), vals.shape[1], _lib.dptr(pc),
                                _lib.dptr(poly) if poly is not None else None, C.byref(st), self._cb, None,
                                C.byref(self._h))
        if rc != _lib.FB_OK:
            self._h = C.c_void_p()
            raise (ValueError if rc == _lib.FB_ERR_INVALID_ARGUMENT else RuntimeError)(_lib.last_error())
        kt = ic.RBFKernelType(st.settings.kernel_type)
        self.interpolant_settings = ic.InterpolantSettings(
            kt, drift=ic.Drift(st.settings.drift), nugget=st.settings.nugget,
            spheroidal_order=ic.SpheroidalOrder(st.settings.spheroidal_order), base_range=st.settings.base_range,
            total_sill=st.settings.total_sill,
            fitting_accuracy=ic.FittingAccuracy(st.settings.tolerance, ic.FittingAccuracyType(st.settings.tolerance_type)))
        self.params = cfg.Params(
            kt, solver_type=cfg.Solvers(st.params.solver_type),
            ddm_params=cfg.DDMParams(d["leaf_threshold"], d["overlap_quota"], d["coarse_ratio"], d["coarse_threshold"]),
            fmm_params=cfg.FmmParams(fp["interpolation_order"], fp["max_points_per_cell"],
                                     cfg.FmmCompressionType(st.params.compression_type), fp["epsilon"],
                                     fp["eval_chunk_size"]),
            naive_solve_threshold=p["naive_solve_threshold"], test_unique=bool(p["test_unique"]))
        info = self.info()
        self._n, self._cols, self._m, self._dim = info["n_points"], info["n_cols"], info["basis_size"], info["dim"]
        return self

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            self._L.fr_free(h)
            self._h = C.c_void_p()

    def _check(self, rc):
        if rc != _lib.FB_OK:
            msg = _lib.last_error()
            if rc == _lib.FB_ERR_POINT_OUTSIDE_TREE:
                raise ValueError(msg)
            raise (ValueError if rc == _lib.FB_ERR_INVALID_ARGUMENT else RuntimeError)(msg)

    # ---- fields ------------------------------------------------------------------------------
    def info(self):
        inf = _lib.FrModelInfo()
        self._check(self._L.fr_get_info(self._h, C.byref(inf)))
        d = {name: getattr(inf, name) for name, _ in inf._fields_ if name != "ddm_domains"}
        d["ddm_domains"] = list(inf.ddm_domains)[: inf.ddm_levels]
        return d

    @property
    def source_points(self):
        out = np.zeros((self._n, self._dim))
        self._check(self._L.fr_source_points(self._h, _lib.dptr(out), None))
        return out

    @property
    def source_values(self):
        out = np.zeros((self._n, self._cols))
        self._check(self._L.fr_source_points(self._h, None, _lib.dptr(out)))
        return _one_col(out)

    @property
    def coefficients(self):
        pc = np.zeros((self._n, self._cols))
        poly = np.zeros((max(self._m, 1), self._cols))
        self._check(self._L.fr_coefficients(self._h, _lib.dptr(pc), _lib.dptr(poly)))
        return Coefficients(pc, poly[: self._m] if self._m else None)

    # ---- evaluation --------------------------------------------------------------------------
    def _eval(self, fn, targets, grads):
        x = _points2d(targets, "target_points")
        m = x.shape[0]
        out = np.zeros((m, self._cols))
        g = np.zeros((m, self._cols * self._dim)) if grads else None
        xr, xc = _lib.strides_of(x)
        self._check(fn(self._h, _lib.dptr(x), m, xr, xc, _lib.dptr(out), _lib.dptr(g) if grads else None))
        return (_one_col(out), g) if grads else _one_col(out)

    def evaluate(self, target_points):
        return self._eval(self._L.fr_evaluate, target_points, False)

    def evaluate_with_gradients(self, target_points):
        return self._eval(self._L.fr_evaluate, target_points, True)

    def evaluate_at_source(self, *, add_nugget=False):
        out = np.zeros((self._n, self._cols))
        self._check(self._L.fr_evaluate_at_source(self._h, int(bool(add_nugget)), _lib.dptr(out)))
        return _one_col(out)

    def build_evaluator(self, extents=None):
        ext = None if extents is None else np.ascontiguousarray(np.asarray(extents, dtype=np.float64).ravel())
        self._check(self._L.fr_build_evaluator(self._h, _lib.dptr(ext) if ext is not None else None))

    def evaluate_targets(self, target_points):
        return self._eval(self._L.fr_evaluate_targets, target_points, False)

    def evaluate_targets_with_gradients(self, target_points):
        # python_bindings.rs:818-826 routes this to the one-shot evaluate_with_gradients (SURVEY.md quirk viii)
        return self._eval(self._L.fr_evaluate, target_points, True)

    # ---- torch CUDA tensors in and out (fr_evaluate*_device): no host round trip, ordered on torch's current stream --
    def _eval_cuda(self, fn, targets, gradients):
        import torch
        p, m, cols, rs, cs, dev = _lib.cuda_matrix(targets, "target_points")
        if cols != self._dim:
            raise ValueError(f"target_points must have {self._dim} columns, got {cols}")
        out = torch.empty((m, self._cols), dtype=torch.float64, device=dev)
        g = torch.empty((m, self._cols * self._dim), dtype=torch.float64, device=dev) if gradients else None
        self._check(fn(self._h, p, m, rs, cs, out.data_ptr(), g.data_ptr() if gradients else None,
                       _lib.cuda_stream(dev)))
        vals = out[:, 0] if self._cols == 1 else out
        return (vals, g) if gradients else vals

    def evaluate_cuda(self, targets, *, gradients=False):
        """evaluate / evaluate_with_gradients with a float64 CUDA tensor of targets (m x dim, any strides); returns
        tensors on its device.  Blocks until the results are complete (the one-shot tree is freed on return)."""
        return self._eval_cuda(self._L.fr_evaluate_device, targets, gradients)

    def evaluate_targets_cuda(self, targets, *, gradients=False):
        """evaluate_targets through the tree of build_evaluator, with a float64 CUDA tensor of targets; gradients come
        from that tree too.  Returns once the targets are binned; the results are ordered on torch's current stream."""
        return self._eval_cuda(self._L.fr_evaluate_targets_device, targets, gradients)

    # ---- isosurfaces (fr_isosurface_extract): one lattice evaluation and one transient tree for all isovalues ------
    def _isosurfaces(self, isovalues, extents, resolution, column, refine, device, sd=None):
        """(meshes, or Solids for side code sd 0 / 1 (isosurface.side_code), {"ms": stage times, "refine":
        [(evaluations, iterations)] per isovalue})"""
        from .isosurface import Handle, lattice_args
        ext, res = lattice_args(extents, resolution)
        iso = np.ascontiguousarray(np.atleast_1d(np.asarray(isovalues, dtype=np.float64)).ravel())
        args = (self._h, _lib.dptr(ext), res.ctypes.data_as(C.POINTER(C.c_uint64)), _lib.dptr(iso), iso.size,
                int(column), int(bool(refine)))
        with Handle() as h:
            if sd is None:
                self._check(self._L.fr_isosurface_extract(*args, C.byref(h.h)))
                meshes = [h.mesh(i, True, device) for i in range(iso.size)]
            else:
                self._check(self._L.fr_isosurface_extract_solid(*args, sd, C.byref(h.h)))
                meshes = [h.solid(i, True, device) for i in range(iso.size)]
            stats = {"ms": h.timing(), "refine": [h.refine_stats(i) for i in range(iso.size)]}
        return meshes, stats

    def extract_isosurfaces(self, isovalues, extents, resolution, *, column=0, refine=True):
        """Meshes of the level sets of value column `column` of a 3-D model: one (vertices (V, 3) float64, faces (F, 3)
        int64, normals (V, 3) float64) per isovalue.  The interpolant is evaluated on the lattice of `extents`
        [x0, y0, z0, x1, y1, z1] and `resolution` (an int or (nx, ny, nz)); every lattice cube is split into six
        tetrahedra, giving one vertex per crossing lattice edge.  With `refine` the vertices are moved along their edges
        onto the interpolant.  Faces are oriented, and normals point, along increasing value.  Every mesh edge is shared
        by two faces except on the lattice's boundary faces."""
        return self._isosurfaces(isovalues, extents, resolution, column, refine, None)[0]

    def extract_isosurfaces_cuda(self, isovalues, extents, resolution, *, column=0, refine=True):
        """extract_isosurfaces with the meshes as torch CUDA tensors on the current CUDA device.  Blocks until they
        are complete, like evaluate_cuda."""
        import torch
        dev = torch.device("cuda", torch.cuda.current_device())
        return self._isosurfaces(isovalues, extents, resolution, column, refine, dev)[0]

    def extract_solids(self, isovalues, extents, resolution, *, side="below", column=0, refine=True):
        """The level sets of extract_isosurfaces closed at the lattice box into solids: one Solid (vertices, faces,
        normals, volume, surface_area, n_surface_vertices, n_surface_faces) per isovalue, for the region {f < iso}
        (side "below", the inside of a signed distance) or {f >= iso} ("above", a grade shell).  The first
        n_surface_vertices / n_surface_faces rows are extract_isosurfaces' mesh for the same arguments (faces with their
        last two columns exchanged for "above"); the cap follows: the lattice's boundary nodes on the solid's side and
        the faces that close the mesh on the six box faces.  Every mesh edge is shared by exactly two faces, all faces
        and normals point out of the solid, and volume / surface_area (the area of the isosurface faces inside the box)
        are computed on the GPU from the final vertices."""
        from .isosurface import side_code
        return self._isosurfaces(isovalues, extents, resolution, column, refine, None, side_code(side))[0]

    def extract_solids_cuda(self, isovalues, extents, resolution, *, side="below", column=0, refine=True):
        """extract_solids with the arrays as torch CUDA tensors on the current CUDA device."""
        import torch
        from .isosurface import side_code
        sd = side_code(side)
        dev = torch.device("cuda", torch.cuda.current_device())
        return self._isosurfaces(isovalues, extents, resolution, column, refine, dev, sd)[0]

    # ---- introspection -----------------------------------------------------------------------
    def ddm_level(self, level):
        nd, npts = C.c_uint64(), C.c_uint64()
        u64 = C.POINTER(C.c_uint64)
        self._check(self._L.fr_ddm_level(self._h, level, C.byref(nd), C.byref(npts), None, None, None, None))
        lp = np.zeros(npts.value, dtype=np.uint64)
        ptr = np.zeros(nd.value + 1, dtype=np.uint64)
        self._check(self._L.fr_ddm_level(self._h, level, None, None, lp.ctypes.data_as(u64), ptr.ctypes.data_as(u64),
                                          None, None))
        idx = np.zeros(int(ptr[-1]), dtype=np.uint64)
        internal = np.zeros(int(ptr[-1]), dtype=np.uint8)
        self._check(self._L.fr_ddm_level(self._h, level, None, None, None, None, idx.ctypes.data_as(u64),
                                          internal.ctypes.data_as(C.POINTER(C.c_uint8))))
        return lp, ptr, idx, internal
