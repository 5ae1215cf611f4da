"""The subdomain factorisations, the batched subdomain solves and one Schwarz preconditioner cycle against dense float64
references, at the sizes where the kernels change path.

References are plain numpy: for a domain with points X the bordered system

    [A + nugget I   P] [lambda]   [d]
    [P^T            0] [c     ] = [0]

with A from oracle.kernels and P the monomials of X in X's own Chebyshev-cube scaling (as Domain::factorise builds them,
domain.rs:168-175).  lambda does not depend on which special points the library picks, so the null-space construction
(special points, Q_top) does not enter the references.  Errors are bounded by the conditioning of that system:
|x_dev - x_ref| <= C_FWD * cond(K) * eps * |x_ref| per domain and per block (lambda, c), with cond the 2-norm condition
number and |x_ref| the norm of the domain's whole solution; where the whole output of a domain is visible (mode 1) its
normwise backward error in K is bounded as well.  Measured on a B200: the largest forward ratio is 2.4 (a 3 x 3 system
with cond 2.2), 0.74 on a level with indefinite domains and below 0.42 elsewhere; the largest backward ratio is 0.64.

  (a) single dense domain through the public API (naive fits): rank 0, 1, 3, 4 and 10, mm = n - rank from 1 to 513
      (k_dom_prep / k_dom_assemble / k_cholesky / k_dom_solve mode 1 below mm = 512, k_chol_big_* / k_tri_inv_* /
      k_tri_gemv / k_big_finish from 512 on), a rank-deficient domain, and mm = 0;
  (b) multi-domain levels through fr_ddm_level_solve: fine levels in mode 0 (internal-point scatter), the coarse level in
      mode 1 with and without the polynomial tail, and a level where only some domains take the indefinite fallback;
  (c) one stationary Schwarz iteration through the public API, whose coefficients are one preconditioner cycle, against
      the oracle's cycle on the same hierarchy.
"""
import ctypes as C

import numpy as np
import pytest

from ferreus_rbf_rs_b200 import _lib
from oracle import rbf as orbf
from tests import helpers as H

EPS = np.finfo(np.float64).eps
U64P = C.POINTER(C.c_uint64)

# forward error bound factor: |x_dev - x_ref| <= C_FWD * cond(K) * eps * |x_ref|
C_FWD = 10.0
# normwise backward error |K x - b| / (|K| |x| + |b|) <= C_BWD * eps (2-norms)
C_BWD = 8.0

LINEAR, TPS, CUBIC, SPHEROIDAL = 0, 1, 2, 3
NONE, CONSTANT, LIN, QUAD = 0, 1, 2, 3


# ---------------------------------------------------------------------------------------------------------- references
def oracle_settings(kernel, drift, dim, nugget=0.0, base_range=1.0):
    s = orbf.InterpolantSettings(kernel, drift=drift, nugget=nugget, base_range=base_range)
    s.set_basis_size(dim)
    return s


def bordered(X, s):
    """the bordered matrix of a domain with points X (its own monomial scaling)"""
    n, m = len(X), s.basis_size
    A = s.kernel().matrix(X, X) + s.nugget * np.eye(n)
    if m == 0:
        return A
    tr, sc = orbf.get_cheb_cube_scaling_factors(X)
    P = orbf.evaluate_monomials(X, s.polynomial_degree, m, tr, sc)
    return np.block([[A, P], [P.T, np.zeros((m, m))]])


def solve_bordered(K, d):
    """x = K^-1 [d; 0] for one or more right-hand sides d (columns)"""
    d = d.reshape(len(d), -1)
    return np.linalg.solve(K, np.vstack([d, np.zeros((K.shape[0] - len(d), d.shape[1]))]))


def fwd_ratio(got, ref, cond, scale=None):
    """|got - ref| / (cond * eps * |ref|): must stay below C_FWD"""
    scale = np.linalg.norm(ref) if scale is None else scale
    return float(np.linalg.norm(got - ref) / (cond * EPS * max(scale, 1e-300)))


def bwd_ratio(K, x, b):
    """normwise backward error in units of eps"""
    r = K @ x - b
    return float(np.linalg.norm(r) / ((np.linalg.norm(K, 2) * np.linalg.norm(x) + np.linalg.norm(b)) * EPS))


def values(pts):
    v = np.sin(3 * pts[:, 0]) + np.cos(2 * pts[:, -1])
    return np.stack([v, np.cos(4 * pts[:, 0] * pts[:, -1]) - 0.5], axis=1)


# ------------------------------------------------------------------------------------------------------- C structures
def c_settings(kernel, drift, nugget=0.0, base_range=1.0):
    st = _lib.FrSettings()
    _lib.lib().fr_settings_default(kernel, C.byref(st))
    st.drift, st.nugget, st.base_range = drift, nugget, base_range
    return st


def c_params(kernel, leaf, coarse, naive=100):
    pr = _lib.FrParams()
    _lib.lib().fr_params_default(kernel, C.byref(pr))
    pr.leaf_threshold, pr.overlap_quota, pr.coarse_ratio, pr.coarse_threshold = leaf, 0.5, 0.125, coarse
    pr.naive_solve_threshold = naive
    return pr


def host_levels(pts, st, pr):
    """[(level points, domain ptr, domain point indices, internal flags)] of the host hierarchy (no GPU)"""
    L = _lib.lib()
    n, dim = pts.shape
    h = C.c_void_p()
    assert L.fr_host_ddm_new(_lib.dptr(pts), n, dim, dim, 1, C.byref(st), C.byref(pr), C.byref(h)) == 0
    try:
        nk, nl = C.c_uint64(), C.c_uint64()
        assert L.fr_host_ddm_counts(h, C.byref(nk), C.byref(nl)) == 0
        assert nk.value == n, "the cases have no duplicate points"
        levels = []
        for li in range(nl.value):
            nd, npts = C.c_uint64(), C.c_uint64()
            assert L.fr_host_ddm_level(h, li, C.byref(nd), C.byref(npts), None, None, None, None) == 0
            lp = np.zeros(npts.value, dtype=np.uint64)
            ptr = np.zeros(nd.value + 1, dtype=np.uint64)
            assert L.fr_host_ddm_level(h, li, None, None, lp.ctypes.data_as(U64P), ptr.ctypes.data_as(U64P), None,
                                       None) == 0
            idx = np.zeros(int(ptr[-1]), dtype=np.uint64)
            internal = np.zeros(int(ptr[-1]), dtype=np.uint8)
            assert L.fr_host_ddm_level(h, li, None, None, None, None, idx.ctypes.data_as(U64P),
                                       internal.ctypes.data_as(C.POINTER(C.c_uint8))) == 0
            levels.append((lp.astype(np.int64), ptr.astype(np.int64), idx.astype(np.int64), internal.astype(bool)))
        return levels
    finally:
        L.fr_host_ddm_free(h)


def domains(level):
    _, ptr, idx, internal = level
    return [(idx[ptr[d]:ptr[d + 1]], internal[ptr[d]:ptr[d + 1]]) for d in range(len(ptr) - 1)]


def domain_rank(X, s):
    """number of special points of a domain: rank of its scaled monomials (threshold of domain.rs:187-204)"""
    if s.basis_size == 0:
        return 0
    tr, sc = orbf.get_cheb_cube_scaling_factors(X)
    r = np.linalg.qr(orbf.evaluate_monomials(X, s.polynomial_degree, s.basis_size, tr, sc), mode="r")
    d = np.abs(np.diag(r))
    return int(np.sum(d > 1e-10 * d.max()))


# ----------------------------------------------------------------------------------------------- (b) level cases
# (name, kernel, drift, dim, n, leaf_threshold, coarse_threshold, seed, spheroidal base_range).  Chosen on the host
# hierarchy (test_level_cases_cover_the_dispatch_edges checks it without a GPU):
#   pair       2 fine domains with mm = 576 (= 0 mod 32), coarse mm = 70
#   many       256 fine domains with mm 61..63 (63 = 31 mod 32), coarse mm = 1023 (spread coarse path)
#   quadratic  128 fine domains of rank 10 with mm 32..34 (32 = 0 mod 32), coarse mm = 374
#   odd        64 fine domains with mm 63..65 (65 = 1 mod 32), coarse mm = 319
LEVEL_CASES = [
    ("pair", CUBIC, LIN, 3, 580, 500, 100, 1, 1.0),
    ("many", LINEAR, CONSTANT, 3, 8000, 64, 1100, 1, 1.0),
    ("quadratic", CUBIC, QUAD, 3, 2758, 64, 400, 1, 1.0),
    ("odd", LINEAR, CONSTANT, 3, 2055, 64, 400, 1, 1.0),
]
# spheroidal kernel (no polynomial) with a negative nugget between the smallest eigenvalues of the domains' kernel
# matrices: some domains are indefinite and take the pivoted fallback, the others keep their Cholesky factor
MIXED_CASE = ("mixed", SPHEROIDAL, NONE, 3, 2000, 64, 400, 5, 0.05)


def level_case(case):
    name, kernel, drift, dim, n, leaf, coarse, seed, br = case
    pts = np.random.default_rng(seed).random((n, dim))
    s = oracle_settings(kernel, drift, dim, base_range=br)
    return pts, s, c_params(kernel, leaf, coarse)


def mixed_nugget(pts, s, levels):
    """the negative nugget in the middle of the widest gap between the fine domains' smallest kernel eigenvalues, and
    the number of domains below it (those whose A + nugget I is indefinite)"""
    ev = np.sort([np.linalg.eigvalsh(s.kernel().matrix(pts[ix], pts[ix]))[0] for ix, _ in domains(levels[0])])
    g = int(np.argmax(np.diff(ev)))
    return -0.5 * (ev[g] + ev[g + 1]), g + 1, float(ev[g + 1] - ev[g])


def test_level_cases_cover_the_dispatch_edges():
    """CPU: across LEVEL_CASES the fine domains' mm = n - rank takes values = 0, 1 and 31 (mod 32), there is a coarse
    domain on each side of 512, a level of 2 and one of 100+ domains; every point of a fine level is internal to exactly
    one domain; MIXED_CASE puts some but not all fine domains below its negative nugget."""
    fine_res, coarse_mm, n_domains = set(), [], set()
    for case in LEVEL_CASES:
        pts, s, pr = level_case(case)
        levels = host_levels(pts, c_settings(case[1], case[2], base_range=case[8]), pr)
        assert len(levels) >= 2
        for li, lvl in enumerate(levels):
            doms = domains(lvl)
            mms = [len(ix) - domain_rank(pts[ix], s) for ix, _ in doms]
            if li == len(levels) - 1:
                assert len(doms) == 1
                coarse_mm.append(mms[0])
                continue
            n_domains.add(len(doms))
            fine_res |= {mm % 32 for mm in mms}
            owners = np.concatenate([ix[f] for ix, f in doms])
            assert np.array_equal(np.sort(owners), np.sort(lvl[0])), "a level point is internal to != 1 domain"
    assert {0, 1, 31} <= fine_res, fine_res
    assert min(coarse_mm) < 512 <= max(coarse_mm), coarse_mm
    assert 2 in n_domains and max(n_domains) >= 100, n_domains
    pts, s, pr = level_case(MIXED_CASE)
    levels = host_levels(pts, c_settings(SPHEROIDAL, NONE, base_range=MIXED_CASE[8]), pr)
    nugget, below, gap = mixed_nugget(pts, s, levels)
    assert 0 < below < len(domains(levels[0])) and nugget < 0 and gap > 0.05


def level_solve(pts, st, pr, level, add_poly, res, n_domains):
    """fr_ddm_level_solve on the rows of res (nvec x (n + basis)); returns (out, n_fallback, ranks)"""
    n, dim = pts.shape
    out = np.full_like(res, np.nan)
    nf = C.c_uint64()
    ranks = np.zeros(n_domains, dtype=np.uint64)
    rc = _lib.lib().fr_ddm_level_solve(_lib.dptr(pts), n, dim, C.byref(st), C.byref(pr), level, add_poly,
                                       _lib.dptr(res), res.shape[0], _lib.dptr(out), C.byref(nf),
                                       ranks.ctypes.data_as(U64P))
    assert rc == 0, _lib.last_error()
    return out, int(nf.value), ranks.astype(np.int64)


def check_fine_level(pts, s, st, pr, levels, li, expect_fallback=None):
    """mode 0: a level point's row is its owning domain's lambda there; every other row stays 0"""
    n, m = len(pts), s.basis_size
    lvl = levels[li]
    doms = domains(lvl)
    res = np.random.default_rng(100 + li).standard_normal((2, n + m))
    out, nf, ranks = level_solve(pts, st, pr, li, 0, res, len(doms))
    if expect_fallback is not None:
        assert nf == expect_fallback
    outside = np.setdiff1d(np.arange(n), lvl[0])
    assert not out[:, outside].any() and not out[:, n:].any()
    worst, gap = 0.0, 0.0
    lam_at = {}
    for d, (ix, internal) in enumerate(doms):
        X = pts[ix]
        assert ranks[d] == domain_rank(X, s)
        K = bordered(X, s)
        cond = np.linalg.cond(K)
        lam = solve_bordered(K, res[:, ix].T)[:len(ix)]
        for v in range(res.shape[0]):
            worst = max(worst, fwd_ratio(out[v, ix[internal]], lam[internal, v], cond, np.linalg.norm(lam[:, v])))
        for p, val in zip(ix[~internal], lam[~internal, 0]):
            lam_at.setdefault(int(p), []).append(val)
    print(f"[ddm-solves] fine level {li}: {len(doms)} domains, n_fallback {nf}, max fwd ratio {worst:.3e}")
    assert worst <= C_FWD, worst
    if all(len(ix) < len(lvl[0]) for ix, _ in doms):
        # the overlap solutions differ from the owners' by far more than the bar, so a scatter of overlap rows shows
        # (two domains whose overlap takes the whole level solve the same system: nothing to tell apart there)
        gap = max(abs(out[0, p] - v) / abs(out[0, p]) for p, vs in lam_at.items() for v in vs)
        assert gap > 1e-3, gap


def check_coarse_level(pts, s, st, pr, levels):
    """mode 1: every coarse point's row, and with add_poly the polynomial in the last `rank` rows"""
    n, m = len(pts), s.basis_size
    li = len(levels) - 1
    (ix, _), = domains(levels[li])
    X = pts[ix]
    K = bordered(X, s)
    cond = np.linalg.cond(K)
    res = np.random.default_rng(7).standard_normal((2, n + m))
    ref = solve_bordered(K, res[:, ix].T)
    outside = np.setdiff1d(np.arange(n), ix)
    worst, worst_b = 0.0, 0.0
    for add_poly in (0, 1):
        out, nf, ranks = level_solve(pts, st, pr, li, add_poly, res, 1)
        assert nf == 0 and ranks[0] == m
        assert not out[:, outside].any()
        for v in range(res.shape[0]):
            scale = np.linalg.norm(ref[:, v])
            worst = max(worst, fwd_ratio(out[v, ix], ref[:len(ix), v], cond, scale))
            if add_poly and m:
                worst = max(worst, fwd_ratio(out[v, n:], ref[len(ix):, v], cond, scale))
                b = np.concatenate([res[v, ix], np.zeros(m)])
                worst_b = max(worst_b, bwd_ratio(K, np.concatenate([out[v, ix], out[v, n:]]), b))
            else:
                assert not out[v, n:].any()
    print(f"[ddm-solves] coarse level {li}: mm {len(ix) - m}, cond {cond:.2e}, max fwd ratio {worst:.3e}, "
          f"max bwd ratio {worst_b:.3e}")
    assert worst <= C_FWD, worst
    assert worst_b <= C_BWD, worst_b


@pytest.mark.gpu
@pytest.mark.parametrize("case", LEVEL_CASES, ids=[c[0] for c in LEVEL_CASES])
def test_level_solves_match_dense_domain_solves(case):
    pts, s, pr = level_case(case)
    st = c_settings(case[1], case[2], base_range=case[8])
    levels = host_levels(pts, st, pr)
    for li in range(len(levels) - 1):
        check_fine_level(pts, s, st, pr, levels, li, expect_fallback=0)
    check_coarse_level(pts, s, st, pr, levels)


@pytest.mark.gpu
def test_level_with_some_indefinite_domains():
    """0 < n_fallback < n_domains on one level: the per-domain use_inverse switch inside one k_dom_solve launch"""
    pts, s, pr = level_case(MIXED_CASE)
    levels = host_levels(pts, c_settings(SPHEROIDAL, NONE, base_range=MIXED_CASE[8]), pr)
    nugget, below, _ = mixed_nugget(pts, s, levels)
    s.nugget = nugget
    st = c_settings(SPHEROIDAL, NONE, nugget=nugget, base_range=MIXED_CASE[8])
    check_fine_level(pts, s, st, pr, levels, 0, expect_fallback=below)


# ------------------------------------------------------------------------------------------ (a) single dense domain
def naive_fit(pts, vals, kernel, drift, nugget=0.0, base_range=1.0):
    """a fit below naive_solve_threshold: one dense domain of all points, solved in mode 1 with the polynomial tail"""
    import ferreus_rbf_rs_b200 as fb
    ic, cfg = fb.interpolant_config, fb.config
    st = ic.InterpolantSettings(ic.RBFKernelType(kernel), drift=ic.Drift(drift), nugget=nugget, base_range=base_range)
    return fb.RBFInterpolator(pts, vals, st, params=cfg.Params(ic.RBFKernelType(kernel),
                                                                naive_solve_threshold=len(pts) + 1))


# (kernel, drift, dim, n, nugget, spheroidal base_range): rank = basis size (0, 1, 3, 4, 10), mm = n - rank
DENSE_CASES = [
    (SPHEROIDAL, NONE, 3, 32, 0.0, 0.3),     # rank 0,  mm 32
    (SPHEROIDAL, NONE, 3, 513, 0.01, 0.3),   # rank 0,  mm 513, nugget
    (LINEAR, CONSTANT, 3, 2, 0.0, 1.0),      # rank 1,  mm 1
    (LINEAR, CONSTANT, 2, 34, 0.0, 1.0),     # rank 1,  mm 33
    (TPS, LIN, 2, 34, 0.0, 1.0),             # rank 3,  mm 31
    (TPS, LIN, 2, 515, 0.0, 1.0),            # rank 3,  mm 512
    (CUBIC, LIN, 3, 36, 0.0, 1.0),           # rank 4,  mm 32
    (CUBIC, LIN, 3, 515, 0.0, 1.0),          # rank 4,  mm 511
    (LINEAR, LIN, 3, 517, 0.05, 1.0),        # rank 4,  mm 513, nugget
    (CUBIC, QUAD, 3, 43, 0.0, 1.0),          # rank 10, mm 33
    (CUBIC, QUAD, 3, 522, 0.0, 1.0),         # rank 10, mm 512
]


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,drift,dim,n,nugget,br", DENSE_CASES)
def test_dense_domain_matches_bordered_solve(kernel, drift, dim, n, nugget, br):
    pts = np.random.default_rng(1000 + n + dim).random((n, dim))
    vals = values(pts)
    co = naive_fit(pts, vals, kernel, drift, nugget, br).coefficients
    s = oracle_settings(kernel, drift, dim, nugget, br)
    m = s.basis_size
    assert domain_rank(pts, s) == m
    K = bordered(pts, s)
    cond = np.linalg.cond(K)
    ref = solve_bordered(K, vals)
    fwd, bwd = 0.0, 0.0
    for v in range(vals.shape[1]):
        x = co.point_coefficients[:, v]
        scale = np.linalg.norm(ref[:, v])
        fwd = max(fwd, fwd_ratio(x, ref[:n, v], cond, scale))
        if m:
            x = np.concatenate([x, co.poly_coefficients[:, v]])
            fwd = max(fwd, fwd_ratio(x[n:], ref[n:, v], cond, scale))
        bwd = max(bwd, bwd_ratio(K, x, np.concatenate([vals[:, v], np.zeros(m)])))
    print(f"[ddm-solves] dense rank {m} mm {n - m}: cond {cond:.2e}, fwd ratio {fwd:.3e}, bwd ratio {bwd:.3e}")
    assert fwd <= C_FWD, fwd
    assert bwd <= C_BWD, bwd


@pytest.mark.gpu
def test_rank_deficient_domain_keeps_the_reduced_polynomial_in_the_last_rows():
    """3-D points on a plane with a linear drift: the z monomial vanishes in the domain's scaling, the domain has rank 3,
    and the polynomial of the 3 remaining monomials [1, x, y] goes to the last 3 of the 4 tail rows (schwarz.rs:147-152,
    as the oracle's coarse solve writes it); the first tail row stays 0."""
    n = 60
    pts = np.random.default_rng(3).random((n, 3))
    pts[:, 2] = 0.5
    vals = values(pts[:, :2])
    co = naive_fit(pts, vals, CUBIC, LIN).coefficients
    s = oracle_settings(CUBIC, LIN, 3)
    assert domain_rank(pts, s) == 3
    K = bordered(pts, s)
    K = np.delete(np.delete(K, n + 3, axis=0), n + 3, axis=1)   # drop the zero z column / row
    cond = np.linalg.cond(K)
    ref = solve_bordered(K, vals)
    assert not co.poly_coefficients[0].any()
    fwd = max(max(fwd_ratio(co.point_coefficients[:, v], ref[:n, v], cond, np.linalg.norm(ref[:, v])),
                  fwd_ratio(co.poly_coefficients[1:, v], ref[n:, v], cond, np.linalg.norm(ref[:, v])))
              for v in range(2))
    print(f"[ddm-solves] rank-deficient domain: cond {cond:.2e}, fwd ratio {fwd:.3e}")
    assert fwd <= C_FWD, fwd


@pytest.mark.gpu
def test_domain_without_free_points():
    """n == basis size (4 points, cubic kernel, linear drift in 3-D): Q^T A Q is 0 x 0, lambda = 0 and the polynomial
    interpolates the data.  The oracle's Domain handles the empty factorisation and gives the same answer."""
    pts = np.array([[0.1, 0.2, 0.3], [0.9, 0.1, 0.4], [0.3, 0.8, 0.2], [0.5, 0.4, 0.95]])
    vals = values(pts)
    model = naive_fit(pts, vals, CUBIC, LIN)
    co = model.coefficients
    assert not co.point_coefficients.any()
    s = oracle_settings(CUBIC, LIN, 3)
    tr, sc = orbf.get_cheb_cube_scaling_factors(pts)
    P = orbf.evaluate_monomials(pts, 1, 4, tr, sc)
    c_ref = np.linalg.solve(P, vals)
    assert fwd_ratio(co.poly_coefficients, c_ref, np.linalg.cond(P)) <= C_FWD
    om = orbf.RBFInterpolator(pts, vals, s, orbf.Params(CUBIC, naive_solve_threshold=5))
    assert not om.point_coefficients.any()
    assert np.allclose(om.poly_coefficients, c_ref, rtol=1e-12, atol=1e-14)


# ------------------------------------------------------------------------------------- (c) one preconditioner cycle
# (kernel, drift, n, coarse_threshold, spheroidal base_range, levels) with leaf_threshold 128: basis 0, 1, 4, 10
CYCLE_CASES = [
    (SPHEROIDAL, NONE, 1500, 300, 0.3, 2),
    (LINEAR, CONSTANT, 2400, 100, 1.0, 3),
    (CUBIC, LIN, 1500, 300, 1.0, 2),
    (CUBIC, QUAD, 2400, 100, 1.0, 3),
]
# one stationary iteration stops below a relative residual of 0.5 (the oracle's first step reaches 0.01-0.05 on these
# cases), while |b| is far above it
CYCLE_TOLERANCE = 0.5
# the product's and the oracle's FMMs agree to ~1e-10 (order 8, epsilon 1e-10); after one cycle the relative difference of
# the coefficients measured on a B200 over seeds 11-14 is at most 2.6e-10 (lambda) and 2.2e-11 (polynomial), 4e-13 for
# the spheroidal case: the bar leaves a margin of about 40
CYCLE_BAR = 1e-8


def one_cycle(kernel, drift, n, coarse, br, levels, seed):
    """(product, oracle) coefficients [lambda; c] of a stationary DDM fit that stops after one iteration"""
    import ferreus_rbf_rs_b200 as fb
    ic, cfg = fb.interpolant_config, fb.config
    pts = H.make_points(n, 3, "uniform", seed=seed)
    vals = values(pts)[:, 0]
    st = ic.InterpolantSettings(ic.RBFKernelType(kernel), drift=ic.Drift(drift), base_range=br,
                                fitting_accuracy=ic.FittingAccuracy(CYCLE_TOLERANCE, ic.FittingAccuracyType.Relative))
    pr = cfg.Params(ic.RBFKernelType(kernel), solver_type=cfg.Solvers.DDM, ddm_params=cfg.DDMParams(128, 0.5, 0.125, coarse),
                    fmm_params=cfg.FmmParams(8, 40, cfg.FmmCompressionType.ACA, 1e-10, 1024), naive_solve_threshold=100)
    model = fb.RBFInterpolator(pts, vals, st, params=pr)
    info = model.info()
    assert info["iterations"] == 1 and info["ddm_levels"] == levels
    assert np.linalg.norm(vals) > CYCLE_TOLERANCE
    os_ = orbf.InterpolantSettings(kernel, drift=drift, base_range=br, tolerance=CYCLE_TOLERANCE)
    op = orbf.Params(kernel, solver_type=orbf.SOLVER_DDM, leaf_threshold=128, coarse_threshold=coarse,
                     naive_solve_threshold=100, interpolation_order=8, max_points_per_cell=40, epsilon=1e-10)
    om = orbf.RBFInterpolator(pts, vals, os_, op)
    assert om.iterations == 1 and len(om.ddm.levels) == levels
    co = model.coefficients
    got = np.concatenate([co.point_coefficients[:, 0], co.poly_coefficients[:, 0] if co.poly_coefficients is not None
                          else np.zeros(0)])
    ref = np.concatenate([om.point_coefficients[:, 0], om.poly_coefficients[:, 0] if om.poly_coefficients is not None
                          else np.zeros(0)])
    return got, ref, n


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,drift,n,coarse,br,levels", CYCLE_CASES)
def test_one_schwarz_cycle_matches_the_oracle(kernel, drift, n, coarse, br, levels):
    """Solvers.DDM stopped after one iteration: the coefficients are precon([f; 0]), the whole cycle (partial matvecs,
    fine-level solves, k_project_* against the global polynomial space, coarse steps with the tail on the last one)."""
    got, ref, n = one_cycle(kernel, drift, n, coarse, br, levels, seed=11)
    d_lam = H.rel_l2(got[:n], ref[:n])
    d_poly = H.rel_l2(got[n:], ref[n:]) if len(got) > n else 0.0
    print(f"[ddm-solves] one cycle kernel {kernel} basis {len(got) - n} levels {levels}: rel diff lambda {d_lam:.3e}, "
          f"poly {d_poly:.3e}")
    assert d_lam <= CYCLE_BAR and d_poly <= CYCLE_BAR
