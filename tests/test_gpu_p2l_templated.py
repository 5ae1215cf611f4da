"""The order-templated W/X kernel (k_p2l_grid_t in csrc/p2l.cu, order 7 in 3-D) against the generic one (k_p2l_grid,
forced with FB_GENERIC_P2L=1) and against the oracle.

The switch is read once per process, so each arm runs in a subprocess: this module, run as a script, evaluates every
case and writes the results to an .npz file.  Clustered points and small leaves give X lists of short ranges, so most
tiles are partial and end in neutral padding rows.  The two arms run the same arithmetic in the same order: they must
agree to 1e-13 (in practice bit for bit), and each must match the oracle to the usual 1e-10.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tests import helpers as H  # noqa: E402

pytestmark = pytest.mark.gpu

ORDER = 7
MATVEC_TOL = 1e-10
AB_TOL = 1e-13
# (kernel registry index, right-hand sides): linear, cubic, spheroidal (fast square-root paths), thin-plate spline (no
# fast path); 3 = 2 + 1 and 8 = 4 + 4 right-hand sides per pass
CASES = [(0, 1), (0, 8), (2, 2), (3, 3), (1, 4)]
N, N_SHARD, MAX_PTS, EPS = 3000, 12000, 20, 1e-7
COMP = 0  # dense M2L operators: no truncation choices between the product and the oracle
SHARD_WORLD = 3


def _points():
    pts = H.make_points(N, 3, "clustered", seed=81)
    rng = np.random.default_rng(82)  # targets next to sources: inside the occupied leaves of a sparse tree
    tg = np.ascontiguousarray(pts[rng.permutation(N)[:500]] + 1e-7 * rng.standard_normal((500, 3)))
    idx = np.random.default_rng(83).permutation(N)[:400]
    return pts, tg, idx


def _weights(n, nrhs, seed):
    return np.random.default_rng(seed).random((n, nrhs)) - 0.5


def compute(path):
    """Every case on this process's W/X kernel, in both square-root modes -> npz at `path`."""
    import ferreus_rbf_rs_b200 as fb
    pts, tg, idx = _points()
    out = {}
    was = fb.get_sqrt_mode()
    try:
        for mode in (1, 0):
            fb.set_sqrt_mode(mode)
            for kernel, nrhs in CASES:
                key = f"k{kernel}_r{nrhs}_m{mode}"
                w = _weights(N, nrhs, 90 + kernel)
                pt = H.product_tree(pts, ORDER, kernel, True, True, MAX_PTS, COMP, EPS)
                pt.set_weights(w)
                out[key + "_self"] = np.asarray(pt.evaluate(w, pts)).reshape(N, nrhs)
                out[key + "_tg"] = np.asarray(pt.evaluate(w, tg)).reshape(len(tg), nrhs)
                out[key + "_sub"] = np.asarray(pt.evaluate_at_sources(w, idx)).reshape(len(idx), nrhs)
                pt.upload_weights(w)
                pt.matvec_resident()
                out[key + "_res"] = np.array(pt.download_result()).reshape(N, nrhs)
            # shares of a partitioned tree: the M2P half of a cell is applied by the rank owning its first point
            spts = H.make_points(N_SHARD, 3, "clustered", seed=84)
            w = _weights(N_SHARD, 1, 85)
            pt = H.product_tree(spts, ORDER, 0, True, True, MAX_PTS, COMP, EPS)
            pt.upload_weights(w)
            comm = fb.Communicator(0, 1)
            for r in range(SHARD_WORLD):
                pt.shard_as(comm, r, SHARD_WORLD, exact=True)
                pt.matvec_sharded()
                out[f"shard{r}_m{mode}"] = np.array(pt.sharded_download()).reshape(N_SHARD, 1)
            pt.shard(None)
    finally:
        fb.set_sqrt_mode(was)
    np.savez(path, **out)


def _run_arm(tmp_path, generic):
    path = str(tmp_path / ("generic.npz" if generic else "templated.npz"))
    env = dict(os.environ)
    env.pop("FB_GENERIC_P2L", None)
    if generic:
        env["FB_GENERIC_P2L"] = "1"
    env["PYTHONPATH"] = ROOT + os.pathsep + env.get("PYTHONPATH", "")
    subprocess.run([sys.executable, "-s", os.path.abspath(__file__), path], cwd=ROOT, env=env, check=True)
    return dict(np.load(path))


@pytest.fixture(scope="module")
def arms(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("p2l_ab")
    return _run_arm(tmp, True), _run_arm(tmp, False)


def test_templated_matches_generic(arms):
    gen, new = arms
    assert sorted(gen) == sorted(new)
    for key in gen:
        assert H.rel_l2(new[key], gen[key]) <= AB_TOL, key
    for mode in (1, 0):  # the shares are partial results: each is nonzero and they add up to the whole
        total = sum(new[f"shard{r}_m{mode}"] for r in range(SHARD_WORLD))
        assert all(np.abs(new[f"shard{r}_m{mode}"]).max() > 0 for r in range(SHARD_WORLD))
        gtotal = sum(gen[f"shard{r}_m{mode}"] for r in range(SHARD_WORLD))
        assert H.rel_l2(total, gtotal) <= AB_TOL


@pytest.mark.parametrize("kernel,nrhs", CASES)
def test_both_arms_match_oracle(arms, kernel, nrhs):
    pts, tg, idx = _points()
    w = _weights(N, nrhs, 90 + kernel)
    ot = H.oracle_tree(pts, ORDER, kernel, True, True, MAX_PTS, COMP, EPS)
    ot.set_weights(w)
    ref = ot.evaluate(w, pts)
    ref_tg = ot.evaluate(w, tg)
    for res in arms:
        for mode in (1, 0):
            key = f"k{kernel}_r{nrhs}_m{mode}"
            assert H.rel_l2(res[key + "_self"], ref) <= MATVEC_TOL, key
            assert H.rel_l2(res[key + "_res"], ref) <= MATVEC_TOL, key
            assert H.rel_l2(res[key + "_sub"], ref[idx]) <= MATVEC_TOL, key
            assert H.rel_l2(res[key + "_tg"], ref_tg) <= MATVEC_TOL, key


def test_shares_match_oracle(arms):
    spts = H.make_points(N_SHARD, 3, "clustered", seed=84)
    w = _weights(N_SHARD, 1, 85)
    ot = H.oracle_tree(spts, ORDER, 0, True, True, MAX_PTS, COMP, EPS)
    ot.set_weights(w)
    ref = ot.evaluate(w, spts)
    for res in arms:
        for mode in (1, 0):
            total = sum(res[f"shard{r}_m{mode}"] for r in range(SHARD_WORLD))
            assert H.rel_l2(total, ref) <= MATVEC_TOL


if __name__ == "__main__":
    compute(sys.argv[1])
