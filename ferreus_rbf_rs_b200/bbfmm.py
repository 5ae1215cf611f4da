"""Python surface of the reference module ``ferreus_bbfmm`` on top of the C ABI.

Mirrors py_ferreus_bbfmm/src/python_bindings.rs:66-389 (class and method names, signatures,
shapes, 1-D return for single-column results, error types and message texts).  All compute is
in libferreus_b200.so; there is no Python or CPU implementation behind these classes.
"""
import ctypes as C
import enum

import numpy as np

from . import _lib


class FmmKernelType(enum.IntEnum):  # python_bindings.rs:66-76 (pyclass eq_int: declaration order)
    LinearRbf = 0
    ThinPlateSplineRbf = 1
    CubicRbf = 2
    SpheroidalRbf = 3
    Laplacian = 4
    OneOverR2 = 5
    OneOverR4 = 6


class SpheroidalOrder(enum.IntEnum):  # python_bindings.rs:79-86
    Three = 0
    Five = 1
    Seven = 2
    Nine = 3


class M2LCompressionType(enum.IntEnum):  # python_bindings.rs:88-95
    None_ = 0
    SVD = 1
    ACA = 2


class FmmParams:
    """FmmParams(max_points_per_cell, compression_type, epsilon, eval_chunk_size) — python_bindings.rs:113-131"""

    def __init__(self, max_points_per_cell, compression_type, epsilon, eval_chunk_size):
        self.max_points_per_cell = int(max_points_per_cell)
        self.compression_type = M2LCompressionType(compression_type)
        self.epsilon = float(epsilon)
        self.eval_chunk_size = int(eval_chunk_size)

    def _c(self):
        return _lib.FbFmmParams(self.max_points_per_cell, int(self.compression_type), self.epsilon,
                                self.eval_chunk_size)


_REGISTRY = {  # registry index, ferreus_rbf_utils/src/utils.rs:558-571
    FmmKernelType.LinearRbf: 0, FmmKernelType.ThinPlateSplineRbf: 1, FmmKernelType.CubicRbf: 2,
    FmmKernelType.Laplacian: 7, FmmKernelType.OneOverR2: 8, FmmKernelType.OneOverR4: 9,
}


class KernelParams:
    """KernelParams(kernel_type, *, spheroidal_order=None, base_range=None, total_sill=None)
    python_bindings.rs:140-188; builder asserts kernel_helpers.rs:72-73."""

    def __init__(self, kernel_type, *, spheroidal_order=None, base_range=None, total_sill=None):
        kernel_type = FmmKernelType(kernel_type)
        if kernel_type == FmmKernelType.SpheroidalRbf:
            order = SpheroidalOrder(spheroidal_order) if spheroidal_order is not None else SpheroidalOrder.Three
            self.registry_index = 3 + int(order)
        else:
            self.registry_index = _REGISTRY[kernel_type]
        self.kernel_type = kernel_type
        self.base_range = 1.0 if base_range is None else float(base_range)
        self.total_sill = 1.0 if total_sill is None else float(total_sill)
        assert self.base_range > 0.0
        assert self.total_sill <= self.base_range

    def _c(self):
        return _lib.FbKernelParams(self.registry_index, self.base_range, self.total_sill)


def _as_matrix(obj, what):
    """numpy_to_matref (python_bindings.rs:20-36): 1-D or 2-D float64, 1-D becomes a column."""
    if not isinstance(obj, np.ndarray) or obj.dtype != np.float64 or obj.ndim not in (1, 2):
        raise TypeError(f"Expected a 1D/2D float64 array for {what}" if what == "source_points"
                        else f"Expected 1D/2D float64 for {what}")
    return obj[:, None] if obj.ndim == 1 else obj


def _to_numpy(mat):
    """mat_to_numpy (python_bindings.rs:39-64): one column comes back 1-D."""
    return mat.reshape(mat.shape[0]) if mat.shape[1] == 1 else mat  # a view: no second copy of the result


class FmmTree:
    """FmmTree(source_points, interpolation_order, kernel_params, adaptive_tree, sparse, *, extents=None,
    params=None) — python_bindings.rs:198-238 -> fb_tree_new."""

    def __init__(self, source_points, interpolation_order, kernel_params, adaptive_tree, sparse, *,
                 extents=None, params=None):
        pts = _as_matrix(source_points, "source_points")
        self._h = C.c_void_p()
        self._lib = _lib.lib()
        ext = None
        dim = pts.shape[1]
        if extents is not None:
            ext = np.ascontiguousarray(np.asarray(extents, dtype=np.float64).ravel())
            dim = ext.size // 2          # bbfmm.rs:291: dimensions come from the extents
            if ext.size != 2 * pts.shape[1]:
                raise ValueError("extents must hold [mins..., maxs...] for every column of source_points")
        kp = kernel_params._c()
        fp = params._c() if params is not None else None
        rs, cs = _lib.strides_of(pts)
        rc = self._lib.fb_tree_new(_lib.dptr(pts), pts.shape[0], dim, rs, cs, int(interpolation_order),
                                   C.byref(kp), int(bool(adaptive_tree)), int(bool(sparse)),
                                   _lib.dptr(ext) if ext is not None else None,
                                   C.byref(fp) if fp is not None else None, C.byref(self._h))
        if rc != _lib.FB_OK:
            self._h = C.c_void_p()
            raise (ValueError if rc == _lib.FB_ERR_INVALID_ARGUMENT else RuntimeError)(_lib.last_error())
        self._n = pts.shape[0]
        self._dim = dim
        self._nrhs = 1

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            self._lib.fb_tree_free(h)
            self._h = C.c_void_p()

    # -- helpers -------------------------------------------------------------------------------
    def _check(self, rc, bad=None, leaf=False):
        if rc == _lib.FB_OK:
            return
        if rc == _lib.FB_ERR_POINT_OUTSIDE_TREE:
            prefix = "FMM leaf evaluation failed" if leaf else "FMM evaluation failed"
            raise ValueError(f"{prefix}: target point at row {bad.value} lies outside the tree extents")
        if rc == _lib.FB_ERR_NO_GRADIENTS:
            raise ValueError("FMM evaluation failed: gradient evaluation requested but kernel does not "
                             "support gradients")
        if rc == _lib.FB_ERR_INVALID_ARGUMENT:
            raise ValueError(_lib.last_error())
        raise RuntimeError(_lib.last_error())

    # -- reference API -------------------------------------------------------------------------
    def set_weights(self, weights):
        w = _as_matrix(weights, "weights")
        rs, cs = _lib.strides_of(w)
        self._check(self._lib.fb_tree_set_weights(self._h, _lib.dptr(w), w.shape[0], w.shape[1], rs, cs))
        self._nrhs = w.shape[1]

    def set_local_coefficients(self, weights):
        w = _as_matrix(weights, "weights")
        rs, cs = _lib.strides_of(w)
        self._check(self._lib.fb_tree_set_local_coefficients(self._h, _lib.dptr(w), w.shape[0], w.shape[1], rs, cs))

    def _eval(self, fn, weights, target_points, grads, leaf, grad_leaf_msg=False):
        w = _as_matrix(weights, "weights")
        x = _as_matrix(target_points, "target_points")
        m = x.shape[0]
        out = _lib.pinned.empty((m, self._nrhs))  # the library writes every element
        g = np.zeros((m, self._nrhs * self._dim)) if grads else None
        bad = C.c_uint64(0)
        wr, wc = _lib.strides_of(w)
        xr, xc = _lib.strides_of(x)
        rc = fn(self._h, _lib.dptr(w), w.shape[0], w.shape[1], wr, wc, _lib.dptr(x), m, xr, xc, _lib.dptr(out),
                _lib.dptr(g) if grads else None, self._nrhs, 1, C.byref(bad))
        self._check(rc, bad, leaf and not grad_leaf_msg)
        return (_to_numpy(out), _to_numpy(g)) if grads else _to_numpy(out)

    def evaluate(self, weights, target_points):
        return self._eval(self._lib.fb_tree_evaluate, weights, target_points, False, False)

    def evaluate_with_gradients(self, weights, target_points):
        return self._eval(self._lib.fb_tree_evaluate, weights, target_points, True, False)

    def evaluate_leaves(self, weights, target_points):
        return self._eval(self._lib.fb_tree_evaluate_leaves, weights, target_points, False, True)

    def evaluate_leaves_with_gradients(self, weights, target_points):
        # python_bindings.rs:353-384 reports "FMM evaluation failed" for this variant
        return self._eval(self._lib.fb_tree_evaluate_leaves, weights, target_points, True, True, True)

    def source_points(self):
        out = np.zeros((self._n, self._dim))
        self._check(self._lib.fb_tree_source_points(self._h, _lib.dptr(out), self._dim, 1))
        return _to_numpy(out)

    # -- extensions (solver fast path, residency, introspection) ---------------------------------
    def evaluate_at_sources(self, weights, indices=None):
        """== evaluate(weights, source_points[indices]) without re-binning (rbf.rs:1357-1364)."""
        w = _as_matrix(weights, "weights")
        idx = None
        m = self._n
        if indices is not None:
            idx = np.ascontiguousarray(indices, dtype=np.uint64)
            m = idx.size
        out = _lib.pinned.empty((m, self._nrhs))
        wr, wc = _lib.strides_of(w)
        rc = self._lib.fb_tree_evaluate_at_sources(
            self._h, _lib.dptr(w), w.shape[0], w.shape[1], wr, wc,
            idx.ctypes.data_as(C.POINTER(C.c_uint64)) if idx is not None else None, m, _lib.dptr(out),
            self._nrhs, 1)
        self._check(rc)
        return _to_numpy(out)

    # -- torch CUDA tensors in and out (fb_tree_*_device): no host round trip, ordered on torch's current stream ----
    def set_weights_cuda(self, weights):
        """set_weights with a float64 CUDA tensor (n x nrhs, any strides)."""
        p, rows, cols, rs, cs, dev = _lib.cuda_matrix(weights, "weights")
        self._check(self._lib.fb_tree_set_weights_device(self._h, p, rows, cols, rs, cs, _lib.cuda_stream(dev)))
        self._nrhs = cols

    def evaluate_cuda(self, weights, targets, *, gradients=False):
        """evaluate / evaluate_with_gradients with float64 CUDA tensors; results are new tensors on the targets'
        device, shaped as the numpy methods return them."""
        import torch
        wp, wrows, wcols, wrs, wcs, _ = _lib.cuda_matrix(weights, "weights")
        xp, m, xcols, xrs, xcs, dev = _lib.cuda_matrix(targets, "target_points")
        if xcols != self._dim:
            raise ValueError(f"target_points must have {self._dim} columns, got {xcols}")
        out = torch.empty((m, self._nrhs), dtype=torch.float64, device=dev)
        g = torch.empty((m, self._nrhs * self._dim), dtype=torch.float64, device=dev) if gradients else None
        bad = C.c_uint64(0)
        rc = self._lib.fb_tree_evaluate_device(self._h, wp, wrows, wcols, wrs, wcs, xp, m, xrs, xcs, out.data_ptr(),
                                               g.data_ptr() if gradients else None, self._nrhs, 1,
                                               _lib.cuda_stream(dev), C.byref(bad))
        self._check(rc, bad)
        vals = out[:, 0] if self._nrhs == 1 else out
        return (vals, g[:, 0] if g.shape[1] == 1 else g) if gradients else vals

    def upload_weights(self, weights):
        w = _as_matrix(weights, "weights")
        rs, cs = _lib.strides_of(w)
        self._check(self._lib.fb_tree_upload_weights(self._h, _lib.dptr(w), w.shape[0], w.shape[1], rs, cs))
        self._nrhs = w.shape[1]

    def matvec_resident(self):
        self._check(self._lib.fb_tree_matvec_resident(self._h))

    def download_result(self):
        out = np.zeros((getattr(self, "_subset_n", None) or self._n, self._nrhs))
        self._check(self._lib.fb_tree_download_result(self._h, _lib.dptr(out), self._nrhs, 1))
        return _to_numpy(out)

    # -- NCCL partition (csrc/comm.cu): one process per GPU ------------------------------------------------
    def shard(self, comm):
        """Partition this tree across the ranks of `comm` (a Communicator, or None to drop the partition)."""
        self._check(self._lib.fb_tree_shard(self._h, comm._h if comm is not None else None))
        self._comm = comm

    def shard_as(self, comm, rank, world, exact=False):
        """Profiling / test aid: the share of `rank` of `world` ranks on a world-1 communicator (fb_tree_shard_as)."""
        self._check(self._lib.fb_tree_shard_as(self._h, comm._h, rank, world, 1 if exact else 0))
        self._comm = comm

    def shard_fork_mode(self, mode):
        self._check(self._lib.fb_tree_shard_fork_mode(self._h, int(mode)))

    def shard_rows(self, rank):
        a, b = C.c_uint64(), C.c_uint64()
        self._check(self._lib.fb_tree_shard_rows(self._h, rank, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def matvec_sharded(self):
        self._check(self._lib.fb_tree_matvec_sharded(self._h))

    def sharded_timing(self):
        ms = np.zeros(4)
        self._check(self._lib.fb_tree_sharded_timing(self._h, _lib.dptr(ms)))
        return dict(zip(("upward_exchange", "downward", "near_field_join_l2p", "result_allreduce"), ms.tolist()))

    def sharded_download(self):
        out = _lib.pinned.empty((self._n, self._nrhs))
        self._check(self._lib.fb_tree_sharded_download(self._h, _lib.dptr(out)))
        return _to_numpy(out)

    # -- sharding by Morton-contiguous leaf ranges (include/ferreus_b200.h, multi-GPU section) ---------
    def leaf_work(self):
        nl = self.info()["n_leaves"]
        ptr = np.zeros(nl + 1, dtype=np.uint64)
        work = np.zeros(nl)
        self._check(self._lib.fb_tree_leaf_work(self._h, ptr.ctypes.data_as(C.POINTER(C.c_uint64)), _lib.dptr(work)))
        return ptr.astype(np.int64), work

    def morton_order(self):
        order = np.zeros(self._n, dtype=np.uint64)
        self._check(self._lib.fb_tree_morton_order(self._h, order.ctypes.data_as(C.POINTER(C.c_uint64))))
        return order.astype(np.int64)

    def set_target_subset(self, indices):
        if indices is None or len(indices) == 0:
            self._check(self._lib.fb_tree_set_target_subset(self._h, None, 0))
            self._subset_n = None
            return
        idx = np.ascontiguousarray(indices, dtype=np.uint64)
        self._check(self._lib.fb_tree_set_target_subset(self._h, idx.ctypes.data_as(C.POINTER(C.c_uint64)), idx.size))
        self._subset_n = idx.size

    def result_device(self):
        """(device pointer, rows, cols) of the last resident matvec result"""
        ptr, rows, cols = C.c_void_p(), C.c_uint64(), C.c_uint64()
        self._check(self._lib.fb_tree_result_device(self._h, C.byref(ptr), C.byref(rows), C.byref(cols)))
        return ptr.value, rows.value, cols.value

    def last_matvec_ms(self):
        ms = C.c_double(0.0)
        self._check(self._lib.fb_tree_last_matvec_ms(self._h, C.byref(ms)))
        return ms.value

    def set_timing(self, enabled):
        self._check(self._lib.fb_tree_set_timing(self._h, int(bool(enabled))))

    def last_timing(self):
        ms = np.zeros(8)
        self._check(self._lib.fb_tree_last_timing(self._h, _lib.dptr(ms)))
        # "wx": P2L (fused with the M2P transpose when the targets are all sources); "leaf": P2P (+ M2P otherwise)
        return dict(zip(["p2m", "m2m", "m2l", "wx", "l2l", "l2p", "leaf", "total"], ms.tolist()))

    def info(self):
        inf = _lib.FbTreeInfo()
        self._check(self._lib.fb_tree_get_info(self._h, C.byref(inf)))
        d = {name: getattr(inf, name) for name, _ in inf._fields_ if name != "center"}
        d["center"] = list(inf.center)[: inf.dim]
        return d

    def dump_cells(self):
        inf = self.info()
        nc = inf["n_cells"]
        keys = np.zeros(nc, dtype=np.uint64)
        flags = np.zeros(nc, dtype=np.uint8)
        ptr = np.zeros(nc + 1, dtype=np.uint64)
        idx = np.zeros(max(1, inf["n_points"]), dtype=np.uint64)
        u64 = C.POINTER(C.c_uint64)
        self._check(self._lib.fb_tree_dump_cells(self._h, keys.ctypes.data_as(u64),
                                                 flags.ctypes.data_as(C.POINTER(C.c_uint8)),
                                                 ptr.ctypes.data_as(u64), idx.ctypes.data_as(u64)))
        return keys, flags, ptr, idx[: int(ptr[-1])]

    def dump_list(self, which):
        inf = self.info()
        nc = inf["n_cells"]
        total = [inf["n_u"], inf["n_v"], inf["n_w"], inf["n_x"]][which]
        ptr = np.zeros(nc + 1, dtype=np.uint64)
        idx = np.zeros(max(1, total), dtype=np.uint64)
        u64 = C.POINTER(C.c_uint64)
        self._check(self._lib.fb_tree_dump_list(self._h, which, ptr.ctypes.data_as(u64), idx.ctypes.data_as(u64)))
        return ptr, idx[:total]

    def m2l_rank(self, level, ref):
        return self._lib.fb_tree_m2l_rank(self._h, level, ref)

    def m2l_stream_warps(self):
        """MMA warps of the streaming M2L kernel this tree runs (csrc/m2l.cu), 0 for the generic kernel"""
        return self._lib.fb_tree_m2l_stream_warps(self._h)

    def m2l_operator(self, level, ref):
        r = self.m2l_rank(level, ref)
        P = self.info()["order"] ** self._dim
        u = np.zeros(P * r)
        vt = np.zeros(r * P)
        self._check(self._lib.fb_tree_m2l_operator(self._h, level, ref, _lib.dptr(u), _lib.dptr(vt)))
        return u.reshape((r, P)).T.copy(), vt.reshape((P, r)).T.copy()


class Communicator:
    """NCCL communicator of the partitioned matvec (fb_comm, include/ferreus_b200.h).  `exchange` broadcasts rank 0's
    128-byte NCCL id to the other ranks: any callable bytes -> bytes, e.g. over torch.distributed or MPI."""

    def __init__(self, rank, world_size, exchange=None):
        L = _lib.lib()
        ident = (C.c_uint8 * 128)()
        if rank == 0:
            rc = L.fb_comm_unique_id(ident)
            if rc != 0:
                raise RuntimeError(_lib.last_error())
        if world_size > 1:
            if exchange is None:
                raise ValueError("world_size > 1 needs an `exchange` callable to broadcast the NCCL id")
            raw = exchange(bytes(ident))
            ident = (C.c_uint8 * 128).from_buffer_copy(raw)
        h = C.c_void_p()
        rc = L.fb_comm_init(ident, rank, world_size, C.byref(h))
        if rc != 0:
            raise RuntimeError(_lib.last_error())
        self._h, self._L, self.rank, self.world_size = h, L, rank, world_size

    @classmethod
    def from_torch_distributed(cls, dist):
        """ranks and the id broadcast taken from an initialised torch.distributed process group (any backend)"""
        import torch
        rank, world = dist.get_rank(), dist.get_world_size()

        def exchange(raw):
            dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
            t = torch.tensor(list(raw), dtype=torch.uint8, device=dev)
            dist.broadcast(t, src=0)
            return bytes(t.cpu().tolist())

        return cls(rank, world, exchange)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._L.fb_comm_free(h)
            self._h = None
