"""Which (dim, order) the streaming M2L kernel serves, and that the cases of tests/test_gpu_m2l_stream.py exercise its
rank pieces (host only, no GPU needed).

k_m2l_stream (csrc/m2l.cu) takes P = order^dim when its register-resident operator slices fit: floor(KS / NW) >= 6,
ceil(KS / NW) <= 8 and ceil(MTU / NW) <= 4 for KS = ceil(P / 4) k-steps and MTU = ceil(P / 8) row tiles, with NW = 8
or 11 MMA warps.  A tree takes orders 1..MAX_ORDER only (kMaxOrder, csrc/fmm.h), so pairs the rule serves beyond that
(2-D orders 17 and 18) never reach the kernel.  If the window or the order limit changes, the first test fails and names
the (dim, order) that test_gpu_m2l_stream.SERVED has to gain or lose.
"""
import ctypes as C

import numpy as np
import pytest

from ferreus_rbf_rs_b200 import _lib
from oracle import morton
from tests import helpers as H
from tests import test_gpu_m2l_stream as S

MAX_ORDER = 16  # Chebyshev nodes per axis a tree accepts


def served_pairs():
    """{(dim, order, MMA warps): compression types} over dim 1-3, order 1-20"""
    L = _lib.lib()
    served = {}
    for comp in (0, 1, 2):
        for dim in (1, 2, 3):
            for order in range(1, 21):
                nw = L.fb_m2l_stream_warps(order ** dim, comp)
                if comp == 0:
                    assert nw == 0, f"uncompressed operators streamed at dim {dim}, order {order}"
                elif nw:
                    served.setdefault((dim, order, nw), set()).add(comp)
    return served


def test_served_orders_are_exactly_the_tested_ones():
    served = served_pairs()
    assert all(comps == {1, 2} for comps in served.values())
    reachable = {c for c in served if c[1] <= MAX_ORDER}
    expected = {(d, p, nw) for d, p, nw in S.SERVED}
    assert reachable - expected == set(), "served but not in SERVED"
    assert expected - reachable == set(), "in SERVED but not served"


def test_served_orders_beyond_the_order_limit_are_rejected_by_the_tree():
    """the rule also serves P = 289 and 324 (2-D orders 17 and 18); fb_tree_new refuses those orders before it touches
    a device, so they cannot reach the kernel untested"""
    L = _lib.lib()
    beyond = sorted({(d, p) for d, p, _ in served_pairs() if p > MAX_ORDER})
    assert beyond == [(2, 17), (2, 18)]
    for dim, order in beyond + [(3, MAX_ORDER + 1)]:
        pts = H.make_points(50, dim, "uniform", seed=1)
        kp = _lib.FbKernelParams(S.KERNEL, 1.0, 1.0)
        out = C.c_void_p()
        rc = L.fb_tree_new(_lib.dptr(pts), 50, dim, dim, 1, order, C.byref(kp), 1, 1, None, None, C.byref(out))
        assert rc == _lib.FB_ERR_INVALID_ARGUMENT and not out.value
        assert _lib.last_error() == f"interpolation_order must be in 1..{MAX_ORDER}"


@pytest.mark.parametrize("P,nw", [(188, 0), (189, 8), (256, 8), (257, 0), (260, 0), (261, 11), (352, 11), (353, 0),
                                  (125, 0), (0, 0)])
def test_window_edges(P, nw):
    assert _lib.lib().fb_m2l_stream_warps(P, 2) == nw


@pytest.mark.parametrize("dim,order,nw", S.SERVED, ids=S.IDS)
@pytest.mark.parametrize("comp", [1, 2])
def test_cases_run_several_rank_pieces(dim, order, nw, comp):
    """the host operator build, at the tree radius and depth of the GPU cases: some operator needs more than one
    24-row piece, and some needs a third piece or a padded rank tile"""
    L = _lib.lib()
    n, kind, max_pts = S.GEOMETRY[dim]
    pts = H.make_points(n, dim, kind, seed=7)
    ht = C.c_void_p()
    assert L.fb_host_tree_new(_lib.dptr(pts), n, dim, dim, 1, None, max_pts, 1, 1, C.byref(ht)) == 0
    nc, nl, depth, nlist = C.c_uint64(), C.c_uint64(), C.c_int32(), (C.c_uint64 * 4)()
    assert L.fb_host_tree_counts(ht, C.byref(nc), C.byref(nl), C.byref(depth), nlist) == 0
    L.fb_host_tree_free(ht)
    assert depth.value >= 4 and nlist[1] > 0
    _, radius = morton.calculate_tree_center_and_radius(list(pts.min(0)) + list(pts.max(0)))
    kp = _lib.FbKernelParams(S.KERNEL, 1.0, 1.0)
    ops = C.c_void_p()
    assert L.fb_ops_new(order, dim, radius, depth.value, C.byref(kp), comp, S.EPS, C.byref(ops)) == 0
    ranks = [L.fb_ops_rank(ops, lvl, r) for lvl in range(2, depth.value + 1) for r in range(S.n_ref(dim))]
    L.fb_ops_free(ops)
    assert min(ranks) > 0
    assert max(ranks) > S.PIECE
    assert max(ranks) > 2 * S.PIECE or any(np.asarray(ranks) % 8)
