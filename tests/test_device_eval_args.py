"""CPU tier of the device-memory evaluation entry points (fb_tree_*_device, fr_evaluate*_device): argument checks
that come before any CUDA call, the tensor validation of the Python layer, and an import that does not pull in torch."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from ferreus_rbf_rs_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cuda_matrix_rejects_what_is_not_a_float64_cuda_tensor():
    torch = pytest.importorskip("torch")
    for obj in (np.zeros((4, 3)), torch.zeros((4, 3), dtype=torch.float64), torch.zeros((2, 2, 3), dtype=torch.float64),
                [[0.0, 1.0]]):
        with pytest.raises((TypeError, ValueError), match="float64 CUDA tensor for target_points"):
            _lib.cuda_matrix(obj, "target_points")


def _fake(n=1):
    # a host address the library must never dereference: every call below fails its argument checks first
    buf = (C.c_double * n)()
    return C.cast(buf, C.c_void_p), buf


def test_null_handle_null_pointers_and_empty_targets_are_invalid_arguments():
    L = _lib.lib()
    p, _keep = _fake(8)
    bad = C.c_uint64(0)
    calls = [
        lambda: L.fb_tree_set_weights_device(None, p, 4, 1, 1, 1, None),
        lambda: L.fb_tree_evaluate_device(None, p, 4, 1, 1, 1, p, 4, 3, 1, p, None, 1, 1, None, C.byref(bad)),
        lambda: L.fb_tree_evaluate_device(None, p, 4, 1, 1, 1, None, 4, 3, 1, p, None, 1, 1, None, C.byref(bad)),
        lambda: L.fb_tree_evaluate_device(None, p, 4, 1, 1, 1, p, 0, 3, 1, p, None, 1, 1, None, C.byref(bad)),
        lambda: L.fr_evaluate_device(None, p, 4, 3, 1, p, None, None),
        lambda: L.fr_evaluate_device(None, None, 4, 3, 1, p, None, None),
        lambda: L.fr_evaluate_device(None, p, 0, 3, 1, p, None, None),
        lambda: L.fr_evaluate_targets_device(None, p, 4, 3, 1, p, None, None),
        lambda: L.fr_evaluate_targets_device(None, None, 4, 3, 1, p, None, None),
        lambda: L.fr_evaluate_targets_device(None, p, 0, 3, 1, p, None, None),
    ]
    for call in calls:
        assert call() == _lib.FB_ERR_INVALID_ARGUMENT
        assert _lib.last_error()


def test_package_import_does_not_import_torch():
    code = "import sys, ferreus_rbf_rs_b200; assert 'torch' not in sys.modules, 'torch imported'"
    subprocess.run([sys.executable, "-c", code], cwd=ROOT, check=True)
