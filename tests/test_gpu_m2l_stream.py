"""The streaming M2L kernel (k_m2l_stream, csrc/m2l.cu) at every order it serves, against the oracle and against the
generic kernel (k_m2l in csrc/fmm_kernels.cuh, forced with FB_M2L_STREAM=0 when a tree is built).

The kernel serves 189 <= P <= 256 with 8 MMA warps and 261 <= P <= 352 with 11 (m2l_stream_warps).  A tree has at most
16 nodes per axis (kMaxOrder), so the (dim, order) pairs in those windows are 2-D orders 14-16 and 3-D order 6 (8 warps)
and 3-D order 7 (11 warps); P = 289 and 324 (2-D orders 17 and 18) are served by the rule but no tree reaches them.
SERVED lists the reachable pairs, tests/test_m2l_stream_dispatch.py checks that the list is complete.  With ACA / SVD at
epsilon 1e-12 the operator ranks exceed one rank piece (24 rows) and are not multiples of the 8-row tile, so the cases
run several pieces per group and padded rank tiles.

A whole-matvec error hides M2L under the near field, so every comparison is also made against the M2L contribution
alone: the oracle port (oracle/fast.py) run once as is and once with every M2L operator of rank 0.  A dropped piece,
stage, entry or right-hand-side column shows up as an error of order one relative to that contribution.
"""
import numpy as np
import pytest

from oracle import fast
from tests import helpers as H

pytestmark = pytest.mark.gpu

MATVEC_TOL = 1e-10  # whole matvec against the oracle (the project's bar)
M2L_TOL = 1e-11     # against the oracle, relative to the M2L contribution
AB_TOL = 1e-13      # streaming vs generic kernel / vs a fresh tree, relative to the M2L contribution
EPS = 1e-12
KERNEL = 0          # linear
PIECE = 24          # rank rows of one piece (kStreamMaxMt * 8)

# (dim, order, MMA warps): every (dim, order) of a tree whose P = order^dim the streaming kernel serves.  P = 196 and 216
# sit on the lower edge of the 8-warp window (floor(KS / NW) = 6), P = 225 is odd, P = 256 gives every warp a full
# 8-step slice, P = 343 runs 11 warps with ceil(KS / NW) = 8
SERVED = [(2, 14, 8), (3, 6, 8), (2, 15, 8), (2, 16, 8), (3, 7, 11)]
IDS = [f"d{d}p{p}" for d, p, _ in SERVED]
NW = {(d, p): nw for d, p, nw in SERVED}
# point clouds of depth >= 4 with many V-list entries per (level, transfer vector) group: n, kind, max points per leaf
GEOMETRY = {2: (5000, "uniform", 10), 3: (6000, "uniform", 8)}


def n_ref(dim):
    return {1: 2, 2: 7, 3: 16}[dim]


def weights(n, nrhs, seed):
    """columns of different magnitude: a column landing in another column's slot shows"""
    w = np.random.default_rng(seed).random((n, nrhs)) - 0.5
    return w * (2.0 ** np.arange(nrhs))[None, :]


class Setup:
    """points, the oracle port and its M2L-free twin for one (dim, order, compression, cloud)"""

    def __init__(self, dim, order, comp, n, kind, max_pts, seed=7):
        self.dim, self.order, self.comp, self.max_pts = dim, order, comp, max_pts
        self.pts = H.make_points(n, dim, kind, seed)
        self.n = n
        self.ot = H.oracle_tree(self.pts, order, KERNEL, True, True, max_pts, comp, EPS)
        self.ff = None
        self.cache = {}

    def product(self):
        pt = H.product_tree(self.pts, self.order, KERNEL, True, True, self.max_pts, self.comp, EPS)
        assert pt.info()["depth"] == self.ot.depth
        for lvl in range(2, self.ot.depth + 1):
            for r in range(n_ref(self.dim)):
                assert pt.m2l_rank(lvl, r) == self.ot.ops.rank(lvl, r), f"rank mismatch level {lvl} ref {r}"
        if self.comp == 1 and self.ff is None:
            # pure-SVD truncation through equal singular values is not unique (DESIGN.md 4.2): the oracle takes the
            # product's factors, so the rest of the pipeline is what is compared
            for lvl in range(2, self.ot.depth + 1):
                for r in range(n_ref(self.dim)):
                    self.ot.ops.u[lvl][r], self.ot.ops.vt[lvl][r] = pt.m2l_operator(lvl, r)
        return pt

    def ranks(self):
        return [self.ot.ops.rank(lvl, r) for lvl in range(2, self.ot.depth + 1) for r in range(n_ref(self.dim))]

    def reference(self, nrhs, seed):
        """(weights, oracle matvec at all sources, its M2L contribution)"""
        key = (nrhs, seed)
        if key not in self.cache:
            if self.ff is None:
                self.ff = fast.FastFmm(self.ot)
                self.ff0 = fast.FastFmm(self.ot)
                self.ff0._ranks = np.zeros_like(self.ff0._ranks)  # orc_m2l applies rank-0 operators: no M2L at all
            w = weights(self.n, nrhs, seed)
            ref = self.ff.matvec(w)
            self.cache[key] = (w, ref, ref - self.ff0.matvec(w))
        return self.cache[key]


_SETUPS = {}


def setup_for(dim, order, comp=2, geometry=None):
    n, kind, max_pts = geometry or GEOMETRY[dim]
    key = (dim, order, comp, n, kind, max_pts)
    if key not in _SETUPS:
        _SETUPS[key] = Setup(dim, order, comp, n, kind, max_pts)
    return _SETUPS[key]


def err(got, ref):
    return float(np.linalg.norm(np.asarray(got).reshape(ref.shape) - ref))


def check(got, ref, m2l, what, tol=M2L_TOL):
    """whole-matvec bar and the M2L-only bar, column by column"""
    got = np.asarray(got).reshape(ref.shape)
    assert H.rel_l2(got, ref) <= MATVEC_TOL, what
    for k in range(ref.shape[1]):
        nm = np.linalg.norm(m2l[:, k])
        assert nm > 1e-3 * np.linalg.norm(ref[:, k]), f"{what}: column {k} has no M2L contribution to test"
        e = err(got[:, k], ref[:, k])
        assert e <= tol * nm, f"{what}: column {k}: error {e / nm:.3e} of the M2L contribution"


def assert_several_pieces(s):
    ranks = s.ranks()
    assert max(ranks) > PIECE, f"no operator has more than one rank piece: ranks {sorted(set(ranks))}"
    assert max(ranks) > 2 * PIECE or any(r % 8 for r in ranks), \
        f"no operator has three pieces or a padded rank tile: ranks {sorted(set(ranks))}"


@pytest.mark.parametrize("dim,order,nw", SERVED, ids=IDS)
def test_every_served_order_matches_oracle_and_generic(dim, order, nw, monkeypatch):
    s = setup_for(dim, order)
    assert s.ot.depth >= 4
    assert_several_pieces(s)
    nrhs = 2
    w, ref, m2l = s.reference(nrhs, 11)
    pt = s.product()
    assert pt.m2l_stream_warps() == nw
    pt.set_weights(w)
    check(pt.evaluate(w, s.pts), ref, m2l, "evaluate")
    stream = np.asarray(pt.evaluate_at_sources(w)).reshape(s.n, nrhs)
    check(stream, ref, m2l, "evaluate_at_sources")
    pt.upload_weights(w)
    pt.matvec_resident()
    check(pt.download_result(), ref, m2l, "resident")
    # the same tree on the generic kernel: the same products in another summation order
    monkeypatch.setenv("FB_M2L_STREAM", "0")
    gt = s.product()
    monkeypatch.delenv("FB_M2L_STREAM")
    assert gt.m2l_stream_warps() == 0
    gt.set_weights(w)
    generic = np.asarray(gt.evaluate_at_sources(w)).reshape(s.n, nrhs)
    check(generic, ref, m2l, "generic kernel")
    for k in range(nrhs):
        assert err(stream[:, k], generic[:, k]) <= AB_TOL * np.linalg.norm(m2l[:, k]), k


@pytest.mark.parametrize("dim,order,nw", SERVED, ids=IDS)
def test_svd_compression(dim, order, nw):
    s = setup_for(dim, order, comp=1)
    assert_several_pieces(s)
    pt = s.product()  # copies the factors into the oracle before its first matvec
    assert pt.m2l_stream_warps() == nw
    w, ref, m2l = s.reference(3, 13)
    pt.set_weights(w)
    check(pt.evaluate_at_sources(w), ref, m2l, "svd")


@pytest.mark.parametrize("nrhs", [1, 3, 4, 5, 8])
@pytest.mark.parametrize("dim,order", [(2, 14), (2, 16), (3, 7)], ids=["d2p14", "d2p16", "d3p7"])
def test_right_hand_side_counts(dim, order, nrhs):
    s = setup_for(dim, order)
    w, ref, m2l = s.reference(nrhs, 20 + nrhs)
    pt = s.product()
    pt.set_weights(w)
    check(pt.evaluate_at_sources(w), ref, m2l, f"{nrhs} right-hand sides")


@pytest.mark.parametrize("dim,order", [(2, 14), (3, 7)], ids=["d2p14", "d3p7"])
def test_work_table_rebuilt_when_the_column_count_changes(dim, order):
    """one tree, nrhs 1 -> 3 -> 1 -> 8 -> 1: the item table is rebuilt at every change and the device item counter
    is reused by every launch; each result must equal a fresh tree's"""
    s = setup_for(dim, order)
    pt = s.product()
    for step, nrhs in enumerate([1, 3, 1, 8, 1]):
        w, ref, m2l = s.reference(nrhs, 40 + nrhs)
        pt.set_weights(w)
        got = np.asarray(pt.evaluate_at_sources(w)).reshape(s.n, nrhs)
        check(got, ref, m2l, f"step {step}, {nrhs} right-hand sides")
        fresh = s.product()
        fresh.set_weights(w)
        again = np.asarray(fresh.evaluate_at_sources(w)).reshape(s.n, nrhs)
        for k in range(nrhs):
            assert err(got[:, k], again[:, k]) <= AB_TOL * np.linalg.norm(m2l[:, k]), (step, k)


@pytest.mark.parametrize("dim,order", [(2, 15), (3, 6)], ids=["d2p15", "d3p6"])
def test_target_subsets(dim, order):
    """evaluate_at_sources(w, idx) restricts M2L to the cells with targets by a per-cell flag; set_target_subset does
    the same for the resident matvec.  The subset is a slab plus a few scattered points, so most cells are skipped."""
    s = setup_for(dim, order)
    nrhs = 2
    w, ref, m2l = s.reference(nrhs, 51)
    rng = np.random.default_rng(52)
    idx = np.union1d(np.flatnonzero(s.pts[:, 0] < 0.3), rng.permutation(s.n)[:50])
    pt = s.product()
    pt.set_weights(w)
    check(pt.evaluate_at_sources(w, idx), ref[idx], m2l[idx], "evaluate_at_sources(idx)")
    pt.upload_weights(w)
    pt.set_target_subset(idx)
    pt.matvec_resident()
    check(pt.download_result(), ref[idx], m2l[idx], "set_target_subset")
    pt.set_target_subset(None)
    pt.matvec_resident()
    check(pt.download_result(), ref, m2l, "all targets again")


@pytest.mark.parametrize("dim,order", [(2, 14), (3, 7)], ids=["d2p14", "d3p7"])
def test_shares_of_a_partition_add_up_to_the_matvec(dim, order):
    """fb_tree_shard_as (exact mode): a share runs the items cut from the entry spans [level_lo, level_hi) of every
    group; the full-length partial results of the shares add up to the unpartitioned matvec"""
    import ferreus_rbf_rs_b200 as fb
    s = setup_for(dim, order)
    nrhs, world = 2, 3
    w, ref, m2l = s.reference(nrhs, 61)
    pt = s.product()
    pt.upload_weights(w)
    pt.matvec_resident()
    whole = np.array(pt.download_result()).reshape(s.n, nrhs)
    comm = fb.Communicator(0, 1)
    total = np.zeros((s.n, nrhs))
    for r in range(world):
        pt.shard_as(comm, r, world, exact=True)
        pt.matvec_sharded()
        part = np.array(pt.sharded_download()).reshape(s.n, nrhs)
        assert H.rel_l2(part, whole) > 1e-3  # a share is not the whole
        total += part
    pt.shard(None)
    assert H.rel_l2(total, whole) <= 1e-13
    check(total, ref, m2l, "sum of the shares")


# depth 2-3 trees (groups shorter than the 16 columns of a stage, items of a single entry) and clustered clouds (a few
# long groups split into several items): dim, order, n, kind, max points per leaf
SMALL_AND_LOPSIDED = [(2, 14, 200, "uniform", 20), (3, 7, 600, "uniform", 60), (2, 15, 600, "uniform", 20),
                      (3, 6, 1500, "uniform", 12), (2, 16, 6000, "clustered", 12), (3, 6, 6000, "clustered", 12)]


@pytest.mark.parametrize("dim,order,n,kind,max_pts", SMALL_AND_LOPSIDED,
                         ids=[f"d{c[0]}p{c[1]}-{c[3]}{c[2]}" for c in SMALL_AND_LOPSIDED])
def test_small_and_lopsided_trees(dim, order, n, kind, max_pts):
    s = setup_for(dim, order, geometry=(n, kind, max_pts))
    if kind == "uniform":
        assert s.ot.depth <= 3
    nrhs = 3
    w, ref, m2l = s.reference(nrhs, 71)
    pt = s.product()
    assert pt.m2l_stream_warps() == NW[(dim, order)]
    pt.set_weights(w)
    check(pt.evaluate_at_sources(w), ref, m2l, f"depth {s.ot.depth}")
