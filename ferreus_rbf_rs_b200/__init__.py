"""ferreus_rbf_rs_b200 — B200-native (sm_100a) drop-in for the BBFMM matvec + RBF solve hot path of
graphic-goose/ferreus_rbf_rs.  The package is a thin host-side mirror of the reference's Python
modules (``ferreus_bbfmm``, ``ferreus_rbf``) over the C ABI in ``include/ferreus_b200.h``."""
from . import _lib  # noqa: F401
from .bbfmm import (Communicator, FmmKernelType, FmmParams, FmmTree, KernelParams,  # noqa: F401
                    M2LCompressionType, SpheroidalOrder)
from . import config, interpolant_config, progress  # noqa: F401,E402
from .rbf import Coefficients, GlobalTrend, RBFInterpolator  # noqa: F401,E402
from .isosurface import Solid, lattice_isosurface, lattice_solid  # noqa: F401,E402


def set_sqrt_mode(fast: bool) -> None:
    """Square-root refinement of the direct-sum hot loops for trees / models built afterwards
    (fb_set_sqrt_mode, include/ferreus_b200.h): True = second order (default, <= 1.3e-12 per kernel value),
    False = third order (~1 ulp).  The integer 3 = True plus the tensor-core P2P distance experiment
    (csrc/p2p_mma.cu)."""
    _lib.lib().fb_set_sqrt_mode(3 if fast == 3 else (1 if fast else 0))


def get_sqrt_mode() -> int:
    return int(_lib.lib().fb_get_sqrt_mode())
