"""The reference's reproducible known-answer tests (SURVEY.md section 8c), re-expressed against the library:
  * monomial bases, polynomials.rs:163-239 (9 exact cases incl. the column order)              CPU, host entry point
  * RFP Cholesky solve on the closed-form SPD matrix make_spd, linalg.rs:638-764                GPU, see below
  * the indefinite fallback of domain.rs:63-68 (linalg.rs:514-616)                              GPU, k_dom_solve
The SPD cases run k_cholesky + k_dom_solve below n = 512 and k_chol_big_* + k_tri_gemv (one domain spread over the GPU)
from there on.
"""
import ctypes as C

import numpy as np
import pytest

from ferreus_rbf_rs_b200 import _lib

MONOMIAL_CASES = [
    # points, degree, expected   (polynomials.rs:163-239)
    ([[1.0], [2.0]], 0, [[1.0], [1.0]]),
    ([[1.0], [2.0]], 1, [[1.0, 1.0], [1.0, 2.0]]),
    ([[1.0], [2.0]], 2, [[1.0, 1.0, 1.0], [1.0, 2.0, 4.0]]),
    ([[1.0, 2.0], [1.0, 2.0]], 0, [[1.0], [1.0]]),
    ([[1.0, 2.0], [3.0, 4.0]], 1, [[1.0, 1.0, 2.0], [1.0, 3.0, 4.0]]),
    ([[1.0, 2.0], [3.0, 4.0]], 2, [[1.0, 1.0, 2.0, 1.0, 2.0, 4.0], [1.0, 3.0, 4.0, 9.0, 12.0, 16.0]]),
    ([[1.0, 2.0, 3.0], [4.0, 5.0, 6.0]], 0, [[1.0], [1.0]]),
    ([[1.0, 2.0, 3.0], [4.0, 5.0, 6.0]], 1, [[1.0, 1.0, 2.0, 3.0], [1.0, 4.0, 5.0, 6.0]]),
    ([[1.0, 2.0, 3.0], [4.0, 5.0, 6.0]], 2,
     [[1.0, 1.0, 2.0, 3.0, 1.0, 2.0, 3.0, 4.0, 6.0, 9.0], [1.0, 4.0, 5.0, 6.0, 16.0, 20.0, 24.0, 25.0, 30.0, 36.0]]),
]


@pytest.mark.parametrize("points,degree,expected", MONOMIAL_CASES)
def test_monomial_bases_known_answers(points, degree, expected):
    from oracle import rbf as orbf
    pts = np.ascontiguousarray(points, dtype=np.float64)
    want = np.array(expected)
    n, dim = pts.shape
    basis = C.c_int32()
    out = np.zeros((n, want.shape[1]))
    rc = _lib.lib().fr_evaluate_monomials(_lib.dptr(pts), n, dim, degree, None, None, _lib.dptr(out), C.byref(basis))
    assert rc == 0 and basis.value == want.shape[1]
    assert np.allclose(out, want, rtol=1e-10, atol=1e-12)
    # the oracle restatement gives the same table (translation 0, scale 1 as in the reference test)
    ref = orbf.evaluate_monomials(pts, degree, want.shape[1], np.zeros(dim), np.ones(dim))
    assert np.allclose(ref, want, rtol=1e-10, atol=1e-12)


def test_monomials_scaled_and_degree_none():
    pts = np.array([[2.0, 10.0], [4.0, 30.0]])
    basis = C.c_int32(7)
    assert _lib.lib().fr_evaluate_monomials(_lib.dptr(pts), 2, 2, -1, None, None, None, C.byref(basis)) == 0
    assert basis.value == 0
    tr, sc = np.array([3.0, 20.0]), np.array([1.0, 10.0])
    out = np.zeros((2, 3))
    assert _lib.lib().fr_evaluate_monomials(_lib.dptr(pts), 2, 2, 1, _lib.dptr(tr), _lib.dptr(sc), _lib.dptr(out),
                                            C.byref(basis)) == 0
    assert np.allclose(out, [[1.0, -1.0, -1.0], [1.0, 1.0, 1.0]])


def make_spd(n, alpha):
    """linalg.rs:638-651: A = M M^T + max(alpha, 1e-3) I, M[i][j] = (sin x + 2 cos x) / (1 + i + j + 1), x = (i+1)(j+2)"""
    i, j = np.meshgrid(np.arange(n, dtype=np.float64), np.arange(n, dtype=np.float64), indexing="ij")
    x = (i + 1.0) * (j + 2.0)
    m = (np.sin(x) + 2.0 * np.cos(x)) / (1.0 + (i + j + 1.0))
    return m @ m.T + max(alpha, 1e-3) * np.eye(n)


def _solve(a, b):
    n, nrhs = b.shape
    x = np.zeros((n, nrhs))
    fb_used = C.c_int32()
    rc = _lib.lib().fr_dense_spd_solve(_lib.dptr(np.ascontiguousarray(a)), n, _lib.dptr(np.ascontiguousarray(b)), nrhs,
                                       _lib.dptr(x), C.byref(fb_used))
    assert rc == 0, _lib.last_error()
    return x, fb_used.value


def _backward_error(a, x, b):
    return np.abs(a @ x - b).max() / max(np.abs(a).max() * np.abs(x).max() + np.abs(b).max(), np.finfo(float).eps)


@pytest.mark.gpu
@pytest.mark.parametrize("n,nrhs", [(6, 2), (7, 3)])
def test_make_spd_cholesky_known_answers(n, nrhs):
    """linalg.rs:685-764: factor + solve on make_spd(n, 1e-2) with the test's right-hand sides; backward error <= 1e-12
    and agreement with a standard LL^T solve (atol 1e-12, rtol 1e-10)."""
    a = make_spd(n, 1e-2)
    i, j = np.meshgrid(np.arange(n, dtype=np.float64), np.arange(nrhs, dtype=np.float64), indexing="ij")
    b = (i + 1.0 + 3.0 * j) / (1.0 + i) if n == 6 else np.sin(i + j + 2.0)
    x, fb_used = _solve(a, b)
    assert fb_used == 0
    assert _backward_error(a, x, b) <= 1e-12
    l = np.linalg.cholesky(a)
    x_std = np.linalg.solve(l.T, np.linalg.solve(l, b))
    assert np.allclose(x, x_std, atol=1e-12, rtol=1e-10)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [33, 100, 513, 700, 1100])
def test_blocked_cholesky_sizes(n):
    """the same construction at sizes that cross the 32-wide blocks, the DMMA trailing update and (n >= 512) the
    whole-GPU factorisation of a single large domain; make_spd gets ill conditioned with n, hence alpha = 1"""
    a = make_spd(n, 1.0)
    b = np.sin(np.arange(n * 2, dtype=np.float64)).reshape(n, 2)
    x, fb_used = _solve(a, b)
    assert fb_used == 0
    assert _backward_error(a, x, b) <= 1e-12
    assert np.allclose(x, np.linalg.solve(a, b), atol=1e-10, rtol=1e-8)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [40, 300, 700])
def test_indefinite_matrix_takes_the_fallback(n):
    """domain.rs:63-68: a subdomain matrix that is not positive definite is solved by the pivoted fallback (n = 700: a
    single domain above the 512 threshold of the whole-GPU factorisation, whose spread solve the fallback bypasses)"""
    a = make_spd(n, 1.0) - 1.5 * np.eye(n)      # eigenvalues on both sides of zero
    ev = np.linalg.eigvalsh(a)
    assert ev[0] < -0.1 and ev[-1] > 0.1
    b = np.cos(np.arange(n * 2, dtype=np.float64)).reshape(n, 2)
    x, fb_used = _solve(a, b)
    assert fb_used == 1
    assert _backward_error(a, x, b) <= 1e-11
    assert np.allclose(x, np.linalg.solve(a, b), atol=1e-9, rtol=1e-8)
