"""ctypes loader for libferreus_b200.so (the C ABI declared in include/ferreus_b200.h).

The product path has no CPU fallback: if the shared library is missing this raises.
"""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libferreus_b200.so")
CSRC = os.path.join(_HERE, "csrc")

FB_OK = 0
FB_ERR_POINT_OUTSIDE_TREE = 1
FB_ERR_NO_GRADIENTS = 2
FB_ERR_INVALID_ARGUMENT = 3
FB_ERR_CUDA = 4


class FbKernelParams(C.Structure):
    _fields_ = [("kernel_type", C.c_int32), ("base_range", C.c_double), ("total_sill", C.c_double)]


class FbFmmParams(C.Structure):
    _fields_ = [("max_points_per_cell", C.c_uint64), ("compression_type", C.c_int32),
                ("epsilon", C.c_double), ("eval_chunk_size", C.c_uint64)]


class FbTreeInfo(C.Structure):
    _fields_ = [("n_points", C.c_uint64), ("n_cells", C.c_uint64), ("n_leaves", C.c_uint64),
                ("depth", C.c_uint64), ("n_u", C.c_uint64), ("n_v", C.c_uint64), ("n_w", C.c_uint64),
                ("n_x", C.c_uint64), ("dim", C.c_int32), ("order", C.c_int32), ("nrhs", C.c_int32),
                ("radius", C.c_double), ("center", C.c_double * 3), ("p2p_pairs", C.c_uint64),
                ("m2p_pairs", C.c_uint64), ("p2l_pairs", C.c_uint64)]


class FrSettings(C.Structure):
    _fields_ = [("kernel_type", C.c_int32), ("drift", C.c_int32), ("spheroidal_order", C.c_int32),
                ("nugget", C.c_double), ("base_range", C.c_double), ("total_sill", C.c_double),
                ("tolerance", C.c_double), ("tolerance_type", C.c_int32)]


class FrParams(C.Structure):
    _fields_ = [("solver_type", C.c_int32), ("leaf_threshold", C.c_uint64), ("overlap_quota", C.c_double),
                ("coarse_ratio", C.c_double), ("coarse_threshold", C.c_uint64), ("interpolation_order", C.c_uint64),
                ("max_points_per_cell", C.c_uint64), ("compression_type", C.c_int32), ("epsilon", C.c_double),
                ("eval_chunk_size", C.c_uint64), ("naive_solve_threshold", C.c_uint64), ("test_unique", C.c_int32)]


class FrGlobalTrend(C.Structure):
    _fields_ = [("dim", C.c_int32), ("angles", C.c_double * 3), ("ratios", C.c_double * 3)]


class FrModelState(C.Structure):
    _fields_ = [("settings", FrSettings), ("params", FrParams), ("basis_size", C.c_int32),
                ("polynomial_degree", C.c_int32), ("translation_factor", C.c_double * 3),
                ("scale_factor", C.c_double * 3), ("has_trend", C.c_int32), ("affine_transform", C.c_double * 16),
                ("inverse_transform", C.c_double * 16)]


class FrEvent(C.Structure):
    _fields_ = [("kind", C.c_int32), ("iter", C.c_uint64), ("residual", C.c_double), ("progress", C.c_double),
                ("message", C.c_char_p)]


class FrModelInfo(C.Structure):
    _fields_ = [("n_points", C.c_uint64), ("n_duplicates", C.c_uint64), ("n_cols", C.c_uint64),
                ("basis_size", C.c_uint64), ("dim", C.c_uint64), ("iterations", C.c_uint64),
                ("last_residual", C.c_double), ("ddm_levels", C.c_uint64), ("ddm_domains", C.c_uint64 * 8),
                ("fit_seconds", C.c_double), ("setup_seconds", C.c_double), ("solve_seconds", C.c_double),
                ("matvecs", C.c_uint64)]


FR_PROGRESS_CB = C.CFUNCTYPE(None, C.POINTER(FrEvent), C.c_void_p)


def build(force=False, jobs=8):
    """Compile the library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    if force:
        subprocess.check_call(["make", "-C", CSRC, "clean"])
    subprocess.check_call(["make", "-C", CSRC, f"-j{jobs}"])
    return LIB_PATH


_lib = None

_dp = C.POINTER(C.c_double)
_u64p = C.POINTER(C.c_uint64)
_u8p = C.POINTER(C.c_uint8)
_i32p = C.POINTER(C.c_int32)
_sz = C.c_size_t
_pd = C.c_ssize_t

# symbol -> (restype, argtypes); every symbol declared in include/ferreus_b200.h
SIGNATURES = {
    "fb_last_error": (C.c_char_p, []),
    "fb_kernel_launch_count": (C.c_uint64, []),
    "fb_set_device": (C.c_int, [C.c_int]),
    "fb_host_alloc": (C.c_void_p, [C.c_size_t]),
    "fb_host_free": (None, [C.c_void_p]),
    "fb_set_sqrt_mode": (C.c_int, [C.c_int]),
    "fb_get_sqrt_mode": (C.c_int, []),
    "fb_trim_memory": (C.c_uint64, []),
    "fb_tree_new": (C.c_int, [_dp, _sz, C.c_int, _pd, _pd, C.c_int, C.POINTER(FbKernelParams), C.c_int, C.c_int,
                              _dp, C.POINTER(FbFmmParams), C.POINTER(C.c_void_p)]),
    "fb_tree_free": (None, [C.c_void_p]),
    "fb_tree_set_weights": (C.c_int, [C.c_void_p, _dp, _sz, _sz, _pd, _pd]),
    "fb_tree_set_local_coefficients": (C.c_int, [C.c_void_p, _dp, _sz, _sz, _pd, _pd]),
    "fb_tree_evaluate": (C.c_int, [C.c_void_p, _dp, _sz, _sz, _pd, _pd, _dp, _sz, _pd, _pd, _dp, _dp, _pd, _pd,
                                   _u64p]),
    "fb_tree_set_weights_device": (C.c_int, [C.c_void_p, C.c_void_p, _sz, _sz, _pd, _pd, C.c_void_p]),
    "fb_tree_evaluate_device": (C.c_int, [C.c_void_p, C.c_void_p, _sz, _sz, _pd, _pd, C.c_void_p, _sz, _pd, _pd,
                                          C.c_void_p, C.c_void_p, _pd, _pd, C.c_void_p, _u64p]),
    "fb_tree_evaluate_leaves": (C.c_int, [C.c_void_p, _dp, _sz, _sz, _pd, _pd, _dp, _sz, _pd, _pd, _dp, _dp, _pd,
                                          _pd, _u64p]),
    "fb_tree_evaluate_at_sources": (C.c_int, [C.c_void_p, _dp, _sz, _sz, _pd, _pd, _u64p, _sz, _dp, _pd, _pd]),
    "fb_tree_upload_weights": (C.c_int, [C.c_void_p, _dp, _sz, _sz, _pd, _pd]),
    "fb_tree_matvec_resident": (C.c_int, [C.c_void_p]),
    "fb_tree_download_result": (C.c_int, [C.c_void_p, _dp, _pd, _pd]),
    "fb_tree_set_timing": (C.c_int, [C.c_void_p, C.c_int]),
    "fb_tree_last_timing": (C.c_int, [C.c_void_p, _dp]),
    "fb_tree_last_matvec_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_double)]),
    "fb_measure_fp64_tflops": (C.c_int, [_dp]),
    "fb_measure_fp64_dmma_tflops": (C.c_int, [_dp]),
    "fb_tree_m2l_flops": (C.c_int, [C.c_void_p, _dp]),
    "fb_tree_source_points": (C.c_int, [C.c_void_p, _dp, _pd, _pd]),
    "fb_tree_get_info": (C.c_int, [C.c_void_p, C.POINTER(FbTreeInfo)]),
    "fb_tree_dump_cells": (C.c_int, [C.c_void_p, _u64p, _u8p, _u64p, _u64p]),
    "fb_tree_dump_list": (C.c_int, [C.c_void_p, C.c_int, _u64p, _u64p]),
    "fb_tree_m2l_rank": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "fb_tree_m2l_operator": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _dp, _dp]),
    "fb_m2l_stream_warps": (C.c_int, [C.c_int, C.c_int]),
    "fb_tree_m2l_stream_warps": (C.c_int, [C.c_void_p]),
    "fb_p2p_blocked_launch_count": (C.c_uint64, []),
    "fb_tree_leaf_work": (C.c_int, [C.c_void_p, _u64p, _dp]),
    "fb_tree_morton_order": (C.c_int, [C.c_void_p, _u64p]),
    "fb_tree_set_target_subset": (C.c_int, [C.c_void_p, _u64p, _sz]),
    "fb_tree_result_device": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), _u64p, _u64p]),
    "fb_comm_unique_id": (C.c_int, [_u8p]),
    "fb_comm_init": (C.c_int, [_u8p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "fb_comm_free": (None, [C.c_void_p]),
    "fb_comm_rank": (C.c_int, [C.c_void_p]),
    "fb_comm_world_size": (C.c_int, [C.c_void_p]),
    "fb_tree_shard": (C.c_int, [C.c_void_p, C.c_void_p]),
    "fb_tree_shard_as": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "fb_tree_shard_fork_mode": (C.c_int, [C.c_void_p, C.c_int]),
    "fb_tree_shard_rows": (C.c_int, [C.c_void_p, C.c_int, _u64p, _u64p]),
    "fb_tree_matvec_sharded": (C.c_int, [C.c_void_p]),
    "fb_tree_sharded_timing": (C.c_int, [C.c_void_p, _dp]),
    "fb_tree_sharded_result_device": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "fb_tree_sharded_download": (C.c_int, [C.c_void_p, _dp]),
    "fb_partition_by_work": (C.c_int, [_dp, _sz, C.c_int, _u64p]),
    "fb_host_tree_new": (C.c_int, [_dp, _sz, C.c_int, _pd, _pd, _dp, C.c_uint64, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "fb_host_tree_free": (None, [C.c_void_p]),
    "fb_host_tree_counts": (C.c_int, [C.c_void_p, _u64p, _u64p, _i32p, _u64p]),
    "fb_host_tree_dump_cells": (C.c_int, [C.c_void_p, _u64p, _u8p, _u64p, _u64p]),
    "fb_host_tree_dump_list": (C.c_int, [C.c_void_p, C.c_int, _u64p, _u64p]),
    "fb_ops_new": (C.c_int, [C.c_int, C.c_int, C.c_double, C.c_int, C.POINTER(FbKernelParams), C.c_int, C.c_double,
                             C.POINTER(C.c_void_p)]),
    "fb_ops_free": (None, [C.c_void_p]),
    "fb_ops_rank": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "fb_ops_get": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _dp, _dp]),
    "fb_ops_tables": (C.c_int, [C.c_void_p, _i32p, _i32p, _i32p, _i32p, _i32p, _i32p, _dp]),
}


SOLVER_SIGNATURES = {
    "fr_settings_default": (None, [C.c_int32, C.POINTER(FrSettings)]),
    "fr_params_default": (None, [C.c_int32, C.POINTER(FrParams)]),
    "fr_fit": (C.c_int, [_dp, _sz, C.c_int, _pd, _pd, _dp, _sz, _pd, _pd, C.POINTER(FrSettings), C.POINTER(FrParams),
                         FR_PROGRESS_CB, C.c_void_p, C.POINTER(C.c_void_p)]),
    "fr_fit_trend": (C.c_int, [_dp, _sz, C.c_int, _pd, _pd, _dp, _sz, _pd, _pd, C.POINTER(FrSettings), C.POINTER(FrParams),
                               C.POINTER(FrGlobalTrend), FR_PROGRESS_CB, C.c_void_p, C.POINTER(C.c_void_p)]),
    "fr_get_state": (C.c_int, [C.c_void_p, C.POINTER(FrModelState)]),
    "fr_model_restore": (C.c_int, [_dp, _sz, C.c_int, _dp, _sz, _dp, _dp, C.POINTER(FrModelState), FR_PROGRESS_CB,
                                   C.c_void_p, C.POINTER(C.c_void_p)]),
    "fr_free": (None, [C.c_void_p]),
    "fr_get_info": (C.c_int, [C.c_void_p, C.POINTER(FrModelInfo)]),
    "fr_source_points": (C.c_int, [C.c_void_p, _dp, _dp]),
    "fr_coefficients": (C.c_int, [C.c_void_p, _dp, _dp]),
    "fr_evaluate": (C.c_int, [C.c_void_p, _dp, _sz, _pd, _pd, _dp, _dp]),
    "fr_evaluate_at_source": (C.c_int, [C.c_void_p, C.c_int, _dp]),
    "fr_build_evaluator": (C.c_int, [C.c_void_p, _dp]),
    "fr_evaluate_targets": (C.c_int, [C.c_void_p, _dp, _sz, _pd, _pd, _dp, _dp]),
    "fr_evaluate_device": (C.c_int, [C.c_void_p, C.c_void_p, _sz, _pd, _pd, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fr_evaluate_targets_device": (C.c_int, [C.c_void_p, C.c_void_p, _sz, _pd, _pd, C.c_void_p, C.c_void_p,
                                             C.c_void_p]),
    "fr_isosurface_extract": (C.c_int, [C.c_void_p, _dp, _u64p, _dp, C.c_int, C.c_int, C.c_int,
                                        C.POINTER(C.c_void_p)]),
    "fr_lattice_isosurface": (C.c_int, [C.c_void_p, _u64p, _dp, C.c_double, C.c_void_p, C.POINTER(C.c_void_p)]),
    "fr_isosurface_counts": (C.c_int, [C.c_void_p, C.c_int, _u64p, _u64p]),
    "fr_isosurface_copy": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fr_isosurface_timing": (C.c_int, [C.c_void_p, _dp]),
    "fr_isosurface_refine_stats": (C.c_int, [C.c_void_p, C.c_int, _u64p, _u64p]),
    "fr_isosurface_free": (None, [C.c_void_p]),
    "fr_isosurface_extract_solid": (C.c_int, [C.c_void_p, _dp, _u64p, _dp, C.c_int, C.c_int, C.c_int, C.c_int,
                                              C.POINTER(C.c_void_p)]),
    "fr_lattice_solid": (C.c_int, [C.c_void_p, _u64p, _dp, C.c_double, C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "fr_isosurface_solid_info": (C.c_int, [C.c_void_p, C.c_int, _u64p, _u64p, _dp, _dp]),
    "fr_dense_spd_solve": (C.c_int, [_dp, C.c_int, _dp, C.c_int, _dp, _i32p]),
    "fr_ddm_level_solve": (C.c_int, [_dp, _sz, C.c_int, C.POINTER(FrSettings), C.POINTER(FrParams), C.c_int, C.c_int,
                                     _dp, C.c_int, _dp, _u64p, _u64p]),
    "fr_evaluate_monomials": (C.c_int, [_dp, _sz, C.c_int, C.c_int, _dp, _dp, _dp, _i32p]),
    "fr_ddm_level": (C.c_int, [C.c_void_p, C.c_int, _u64p, _u64p, _u64p, _u64p, _u64p, _u8p]),
    "fr_host_ddm_new": (C.c_int, [_dp, _sz, C.c_int, _pd, _pd, C.POINTER(FrSettings), C.POINTER(FrParams),
                                  C.POINTER(C.c_void_p)]),
    "fr_host_ddm_free": (None, [C.c_void_p]),
    "fr_host_ddm_counts": (C.c_int, [C.c_void_p, _u64p, _u64p]),
    "fr_host_ddm_kept": (C.c_int, [C.c_void_p, _u64p]),
    "fr_host_ddm_level": (C.c_int, [C.c_void_p, C.c_int, _u64p, _u64p, _u64p, _u64p, _u64p, _u8p]),
}


def lib():
    """Load the shared library (once).  Raises if it has not been built: there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C ferreus_rbf_rs_b200/csrc`). The CUDA library is the only implementation.")
    l = C.CDLL(LIB_PATH)
    for name, (res, args) in list(SIGNATURES.items()) + list(SOLVER_SIGNATURES.items()):
        fn = getattr(l, name)
        fn.restype = res
        fn.argtypes = args
    _lib = l
    return l


def last_error():
    msg = lib().fb_last_error()
    return msg.decode() if msg else ""


def dptr(a):
    return a.ctypes.data_as(_dp)


class _PinnedPool:
    """Result matrices backed by page-locked blocks (fb_host_alloc): the device -> host copy lands in them directly and a
    block returns to the pool when the array that owns it is collected.  Small results and anything beyond the pool cap
    use ordinary numpy memory."""
    MIN_BYTES = 1 << 20
    CAP_BYTES = 1 << 30

    def __init__(self):
        self.free = {}   # nbytes -> [ptr]
        self.held = 0    # bytes currently owned by the pool (handed out or free)

    def _release(self, ptr, nbytes):
        self.free.setdefault(nbytes, []).append(ptr)

    def empty(self, shape):
        import weakref
        import numpy as np
        count = int(np.prod(shape))
        nbytes = count * 8
        if nbytes < self.MIN_BYTES:
            return np.empty(shape)
        lst = self.free.get(nbytes)
        if lst:
            ptr = lst.pop()
        else:
            if self.held + nbytes > self.CAP_BYTES:
                for sz, ptrs in list(self.free.items()):   # drop cached blocks of other sizes first
                    while ptrs:
                        lib().fb_host_free(ptrs.pop())
                        self.held -= sz
                if self.held + nbytes > self.CAP_BYTES:
                    return np.empty(shape)
            ptr = lib().fb_host_alloc(nbytes)
            if not ptr:
                return np.empty(shape)
            self.held += nbytes
        block = (C.c_double * count).from_address(ptr)
        fin = weakref.finalize(block, self._release, ptr, nbytes)
        fin.atexit = False
        return np.frombuffer(block, dtype=np.float64, count=count).reshape(shape)


pinned = _PinnedPool()


def strides_of(a):
    """element strides (row, col) of a 2-D float64 array"""
    return a.strides[0] // 8, a.strides[1] // 8


def cuda_matrix(obj, what):
    """A 1-D or 2-D float64 CUDA tensor as (data_ptr, rows, cols, row_stride, col_stride, device); 1-D is a column.
    torch is imported here, not when the package is, so the numpy API works without it."""
    import torch
    if not isinstance(obj, torch.Tensor) or not obj.is_cuda or obj.dtype != torch.float64 or obj.dim() not in (1, 2):
        raise TypeError(f"Expected a 1D/2D float64 CUDA tensor for {what}")
    if obj.dim() == 1:
        return obj.data_ptr(), obj.shape[0], 1, obj.stride(0), 1, obj.device
    return obj.data_ptr(), obj.shape[0], obj.shape[1], obj.stride(0), obj.stride(1), obj.device


def cuda_stream(device):
    """handle of torch's current stream on `device` (0 for the legacy default stream)"""
    import torch
    return torch.cuda.current_stream(device).cuda_stream
