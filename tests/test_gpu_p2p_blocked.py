"""The one-column symmetric P2P kernel blocked on whole 128-target tiles (k_p2p_sym_blocked in csrc/p2p_sym.cu) against
the two-target kernel it replaces (k_p2p_sym, forced with FB_GENERIC_P2P=1) and against the oracle.

The switch is read once per process, so each arm runs in a subprocess: this module, run as a script, evaluates every
case and writes the results to an .npz file.  The cases cover leaves whose sizes sit on every boundary of the
targets-per-lane choice (1, 2 or 4 per lane) and of the 128-target tile, clustered clouds with near-coincident points
and exact duplicates, 1-D / 2-D / 3-D trees, four kernel families in both square-root modes, and the 3- and 5-rank
shares of a partitioned tree.  Small clouds split every tile's sources over several warps (split > 1); the 300 000-point
cloud runs with split = 3.  Only the summation order of the P2P sums differs between the arms: they must agree to 1e-13,
and each must match the oracle to the usual 1e-10.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tests import helpers as H  # noqa: E402

ORDER = 5
MATVEC_TOL = 1e-10
AB_TOL = 1e-13
COMP = 0  # dense M2L operators: no truncation choices between the product and the oracle
EPS = 1e-8
# leaf sizes on every boundary of NT (32, 64 targets) and of the tile (128, 256 targets)
BOUNDARY_SIZES = (1, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256)
BOUNDARY_MAX_PTS = 256
KERNELS = (0, 2, 3, 1)  # linear, cubic, spheroidal (fast square-root paths), thin-plate spline (no fast path)
WORLDS = (3, 5)


def boundary_points():
    """One cluster per size, each alone in a depth-3 cell.  The clusters are grouped under four adjacent depth-2 cells
    that each hold more than BOUNDARY_MAX_PTS points, so the adaptive tree splits them and every cluster becomes one
    leaf of exactly its size; leaves in neighbouring cells are U-list neighbours."""
    rng = np.random.default_rng(7)
    groups = {(1, 1, 1): (256, 1), (2, 1, 1): (255, 31), (1, 2, 1): (129, 128), (2, 2, 1): (127, 65, 64, 63, 33, 32)}
    out = []
    for parent, sizes in groups.items():
        for c, size in enumerate(sizes):
            child = np.array(parent) * 2 + np.array([c & 1, (c >> 1) & 1, c >> 2])
            out.append((child + 0.5) / 8.0 + rng.uniform(-0.05, 0.05, (size, 3)))
    return np.ascontiguousarray(np.concatenate(out))


UNIT_CUBE = (0.0, 0.0, 0.0, 1.0, 1.0, 1.0)  # root cell of the boundary cloud: depth-3 cells are 1/8 wide


def near_points():
    """Clustered points, a near-coincident copy of each, and 60 exact duplicates spread over the cloud."""
    rng = np.random.default_rng(17)
    base = H.make_points(2500, 3, "clustered", seed=18)
    pts = np.concatenate([base, base + rng.standard_normal(base.shape) * 10.0 ** rng.uniform(-9, -3, (len(base), 1))])
    pts[-60:] = pts[rng.permutation(len(pts) - 60)[:60]]
    return np.ascontiguousarray(pts)


# (name, points, max points per leaf, extents, kernels) of the clouds compared with the oracle
def clouds():
    return [("bnd", boundary_points(), BOUNDARY_MAX_PTS, UNIT_CUBE, KERNELS),
            ("near", near_points(), 40, None, (0, 3)),
            ("d1", np.ascontiguousarray(H.make_points(3000, 1, "clustered", seed=19)), 30, None, (0, 1)),
            ("d2", np.ascontiguousarray(H.make_points(4000, 2, "clustered", seed=20)), 30, None, (0, 2))]


def _weights(n, seed):
    return np.random.default_rng(seed).random((n, 1)) - 0.5


def compute(path):
    """Every case on this process's P2P kernel -> npz at `path`."""
    import ferreus_rbf_rs_b200 as fb
    from ferreus_rbf_rs_b200 import _lib
    out = {}
    was = fb.get_sqrt_mode()
    launches0 = _lib.lib().fb_p2p_blocked_launch_count()
    try:
        for mode in (1, 0):
            fb.set_sqrt_mode(mode)
            for name, pts, max_pts, ext, kernels in clouds():
                n = len(pts)
                for kernel in kernels:
                    w = _weights(n, 30 + kernel)
                    pt = H.product_tree(pts, ORDER, kernel, True, True, max_pts, COMP, EPS, extents=ext)
                    pt.set_weights(w)
                    out[f"{name}_k{kernel}_m{mode}"] = np.asarray(pt.evaluate(w, pts)).reshape(n, 1)
            # shares of a partitioned tree: every unordered pair once across the ranks
            spts = H.make_points(12000, 3, "clustered", seed=21)
            w = _weights(len(spts), 22)
            pt = H.product_tree(spts, ORDER, 0, True, True, 30, COMP, EPS)
            pt.set_weights(w)
            out[f"shard_whole_m{mode}"] = np.asarray(pt.evaluate(w, spts)).reshape(len(spts), 1)
            pt.upload_weights(w)
            comm = fb.Communicator(0, 1)
            for world in WORLDS:
                for r in range(world):
                    pt.shard_as(comm, r, world, exact=True)
                    pt.matvec_sharded()
                    out[f"shard{world}_{r}_m{mode}"] = np.array(pt.sharded_download()).reshape(len(spts), 1)
            pt.shard(None)
        fb.set_sqrt_mode(1)
        big = np.ascontiguousarray(H.make_points(300_000, 3, "uniform", seed=23))
        w = _weights(len(big), 24)
        pt = H.product_tree(big, ORDER, 0, True, True, 64, 2, EPS)
        pt.set_weights(w)
        out["big"] = np.asarray(pt.evaluate(w, big)).reshape(len(big), 1)
    finally:
        fb.set_sqrt_mode(was)
    out["blocked_launches"] = np.array(_lib.lib().fb_p2p_blocked_launch_count() - launches0)
    np.savez(path, **out)


def _run_arm(tmp_path, generic):
    path = str(tmp_path / ("generic.npz" if generic else "blocked.npz"))
    env = dict(os.environ)
    env.pop("FB_GENERIC_P2P", None)
    if generic:
        env["FB_GENERIC_P2P"] = "1"
    env["PYTHONPATH"] = ROOT + os.pathsep + env.get("PYTHONPATH", "")
    subprocess.run([sys.executable, "-s", os.path.abspath(__file__), path], cwd=ROOT, env=env, check=True)
    return dict(np.load(path))


@pytest.fixture(scope="module")
def arms(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("p2p_ab")
    return _run_arm(tmp, True), _run_arm(tmp, False)


def test_boundary_cloud_has_every_leaf_size():
    """CPU: the host tree of the boundary cloud has a leaf of each size in BOUNDARY_SIZES."""
    from ferreus_rbf_rs_b200 import _lib
    L = _lib.lib()
    pts = boundary_points()
    n, dim = pts.shape
    h = C.c_void_p()
    ext = np.array(UNIT_CUBE)
    assert L.fb_host_tree_new(_lib.dptr(pts), n, dim, dim, 1, _lib.dptr(ext), BOUNDARY_MAX_PTS, 1, 1, C.byref(h)) == 0
    try:
        nc, nl, depth = C.c_uint64(), C.c_uint64(), C.c_int32()
        nlist = (C.c_uint64 * 4)()
        assert L.fb_host_tree_counts(h, C.byref(nc), C.byref(nl), C.byref(depth), nlist) == 0
        nc = int(nc.value)
        u64p = C.POINTER(C.c_uint64)
        keys = np.zeros(nc, dtype=np.uint64)
        flags = np.zeros(nc, dtype=np.uint8)
        ptr = np.zeros(nc + 1, dtype=np.uint64)
        idx = np.zeros(n, dtype=np.uint64)
        assert L.fb_host_tree_dump_cells(h, keys.ctypes.data_as(u64p), flags.ctypes.data_as(C.POINTER(C.c_uint8)),
                                         ptr.ctypes.data_as(u64p), idx.ctypes.data_as(u64p)) == 0
    finally:
        L.fb_host_tree_free(h)
    sizes = np.diff(ptr.astype(np.int64))[flags == 1]
    assert sorted(int(s) for s in sizes if s > 0) == sorted(BOUNDARY_SIZES)


@pytest.mark.gpu
def test_each_arm_ran_its_kernel(arms):
    gen, new = arms
    assert int(gen["blocked_launches"]) == 0
    assert int(new["blocked_launches"]) > 0


@pytest.mark.gpu
def test_blocked_matches_generic(arms):
    gen, new = arms
    assert sorted(gen) == sorted(new)
    for key in gen:
        if key != "blocked_launches":
            assert H.rel_l2(new[key], gen[key]) <= AB_TOL, key


@pytest.mark.gpu
def test_shares_add_up_to_the_matvec(arms):
    for res in arms:
        for mode in (1, 0):
            whole = res[f"shard_whole_m{mode}"]
            for world in WORLDS:
                parts = [res[f"shard{world}_{r}_m{mode}"] for r in range(world)]
                assert all(np.abs(p).max() > 0 for p in parts)
                assert H.rel_l2(sum(parts), whole) <= AB_TOL, (world, mode)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["bnd", "near", "d1", "d2"])
def test_both_arms_match_oracle(arms, name):
    (_, pts, max_pts, ext, kernels), = [c for c in clouds() if c[0] == name]
    for kernel in kernels:
        w = _weights(len(pts), 30 + kernel)
        ot = H.oracle_tree(pts, ORDER, kernel, True, True, max_pts, COMP, EPS, extents=ext)
        ot.set_weights(w)
        ref = ot.evaluate(w, pts)
        for res in arms:
            for mode in (1, 0):
                key = f"{name}_k{kernel}_m{mode}"
                assert H.rel_l2(res[key], ref) <= MATVEC_TOL, key


if __name__ == "__main__":
    compute(sys.argv[1])
