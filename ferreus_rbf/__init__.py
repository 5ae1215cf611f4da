"""Importable stand-in for the reference's PyO3 module ``ferreus_rbf`` (py_ferreus_rbf/src/lib.rs:15-87): the same
top-level classes and the ``config`` / ``interpolant_config`` / ``progress`` submodules registered in ``sys.modules``
exactly as the Rust module init does, all re-exported from the B200 mirror (``ferreus_rbf_rs_b200``).  The reference's
isosurfacing (``ferreus_rbf.isosurfacing``, ``build_isosurface(s)``, ``Mesh``, ``BoundaryClosure``: the regularised
surface following of ``ferreus_rmt``) is absent, and no function takes those names.  Isosurfaces of 3-D models come
from ``RBFInterpolator.extract_isosurfaces`` / ``extract_isosurfaces_cuda`` instead: lattice marching tetrahedra with the
vertices refined onto the interpolant, which gives different meshes."""
import sys

import numpy as np

from ferreus_rbf_rs_b200 import config, interpolant_config, progress  # noqa: F401
from ferreus_rbf_rs_b200.rbf import Coefficients, GlobalTrend, RBFInterpolator  # noqa: F401

# lib.rs:27-60: sys.modules["ferreus_rbf.config"] = cfg, ... so `from ferreus_rbf.config import Params` works
sys.modules[__name__ + ".config"] = config
sys.modules[__name__ + ".interpolant_config"] = interpolant_config
sys.modules[__name__ + ".progress"] = progress


class RBFTestFunctions:
    """The two analytic test functions the reference examples and BASELINE config C3 use
    (ferreus_rbf/src/rbf_test_functions.rs:44-99 franke_2d, :102-151 f1_3d); harness data, not product code."""

    @staticmethod
    def franke_2d(points):
        p = np.asarray(points, dtype=np.float64)
        assert p.ndim == 2 and p.shape[1] == 2
        x, y = 9.0 * p[:, 0], 9.0 * p[:, 1]
        return (0.75 * np.exp(-((x - 2.0) ** 2 + (y - 2.0) ** 2) / 4.0)
                + 0.75 * np.exp(-((x + 1.0) ** 2) / 49.0 - ((y + 1.0) ** 2) / 10.0)
                + 0.5 * np.exp(-((x - 7.0) ** 2 + (y - 3.0) ** 2) / 4.0)
                - 0.2 * np.exp(-((x - 4.0) ** 2 + (y - 7.0) ** 2)))[:, None]

    @staticmethod
    def f1_3d(points):
        p = np.asarray(points, dtype=np.float64)
        assert p.ndim == 2 and p.shape[1] == 3
        x, y, z = 9.0 * p[:, 0], 9.0 * p[:, 1], 9.0 * p[:, 2]
        return (0.75 * np.exp(-((x - 2.0) ** 2 + (y - 2.0) ** 2 + (z - 2.0) ** 2) / 4.0)
                + 0.75 * np.exp(-((x + 1.0) ** 2) / 49.0 - ((y + 1.0) ** 2) / 10.0 - ((z + 1.0) ** 2) / 10.0)
                + 0.5 * np.exp(-((x - 7.0) ** 2 + (y - 3.0) ** 2 + (z - 5.0) ** 2) / 4.0)
                - 0.2 * np.exp(-((x - 4.0) ** 2 + (y - 7.0) ** 2 + (z - 5.0) ** 2)))[:, None]


__all__ = ["RBFInterpolator", "Coefficients", "GlobalTrend", "RBFTestFunctions", "config", "interpolant_config",
           "progress"]
