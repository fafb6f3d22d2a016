"""The extended-precision reference (oracle/xprec.py) against mpmath at 40 digits, on exact integer cases, and the
backward errors LAPACK's FP64 Cholesky reaches on the matrix families tests/test_gpu_backward_error.py holds the device
to.  CPU only."""
import numpy as np
import pytest
import scipy.linalg

from oracle import sds_oracle as so
from oracle import xprec as xp

pytestmark = pytest.mark.skipif(not xp.AVAILABLE, reason=xp.REASON)

EPS_LD = float(np.finfo(np.longdouble).eps)


def ks(n, ell, sf, sn):
    """(K, diag S) of the sampler on the unit grid (sliceSample.py:104-105,183-190)."""
    x = np.arange(n, dtype=np.float64).reshape(n, 1)
    K = so.cov_matrix(x, np.array([ell, sf, sn]))
    return K, so.s_diagonal(np.diagonal(K), sn)


def ill_conditioned(n):
    """K+S at the corner of the bench bracket, R + 1e-11 I from it, and a graded D A D."""
    K, S = ks(n, 11.0, 20.0, 0.05)
    rs = np.random.RandomState(n)
    M = rs.standard_normal((n, n))
    d = np.logspace(-3, 3, n)
    G = d[:, None] * (M @ M.T / n + np.eye(n)) * d[None, :]
    return {'ks': xp.symmetric(K + np.diag(S)), 'r': xp.r_plus_jitter(K, S), 'graded': xp.symmetric(G)}


# ------------------------------------------------------------------ mpmath at 40 digits
mp = pytest.importorskip('mpmath')


def _mpf(v):
    # a longdouble is the exact sum of two doubles (64 = 53 + 11 significant bits)
    hi = float(v)
    return mp.mpf(hi) + mp.mpf(float(v - np.longdouble(hi)))


def _mp(A):
    return mp.matrix([[_mpf(v) for v in row] for row in np.asarray(A)])


def _mp_chol(A):
    with mp.workdps(40):
        return mp.cholesky(_mp(A))


@pytest.mark.parametrize('n', [7, 24, 40])
@pytest.mark.parametrize('family', ['ks', 'r', 'graded'])
def test_chol_trsv_loglik_against_mpmath(n, family):
    A = ill_conditioned(n)[family]
    g = np.random.RandomState(n + 1).standard_normal(n)
    L = xp.chol(A)
    z = xp.trsv(L.astype(np.float64), g)
    with mp.workdps(40):
        Lm = _mp_chol(A)
        # the factor: each entry to the conditioning of its column (forward error <= cond * eps_ld, column-scaled)
        Lref = np.array([[float(Lm[i, j]) for j in range(n)] for i in range(n)])
        cond = np.linalg.cond(A)
        err = np.abs(L.astype(np.float64) - Lref).max(axis=0) / np.abs(Lref).max(axis=0)
        assert err.max() <= 4 * cond * EPS_LD + 1e-300, (err.max(), cond)
        # backward error of the longdouble factor itself: a few longdouble ulps, 1/500 of one FP64 ulp
        Lx = _mp(L)
        Am = _mp(A)
        res = max(abs(Am[i, j] - sum(Lx[i, k] * Lx[j, k] for k in range(j + 1))) / sum(abs(Lx[i, k] * Lx[j, k]) for k in range(j + 1))
                  for i in range(n) for j in range(i + 1))
        assert float(res) <= 16 * EPS_LD, float(res)
        # trsv with the FP64-rounded factor: forward error within the conditioning of L at longdouble precision
        Lf = _mp(L.astype(np.float64))
        zm = mp.lu_solve(Lf, mp.matrix([mp.mpf(float(v)) for v in g]))
        zerr = max(abs(_mpf(z[i]) - zm[i]) for i in range(n)) / max(abs(zm[i]) for i in range(n))
        assert float(zerr) <= 4 * n * np.linalg.cond(L.astype(np.float64)) * EPS_LD
        # log N(g; 0, A) within the conditioning at longdouble precision: 2000 times closer than FP64 can be
        wm = mp.lu_solve(Lm, mp.matrix([mp.mpf(float(v)) for v in g]))
        ref = -(sum(w * w for w in wm) / 2 + sum(mp.log(Lm[i, i]) for i in range(n)) + n * mp.log(2 * mp.pi) / 2)
        got = xp.loglik(A, g)
        rel = abs(float((_mpf(got) - ref) / ref))
        print('%s n=%d cond %.1e: factor %.1e, trsv %.1e, loglik %.1e' % (family, n, cond, err.max(), float(zerr), rel))
        assert rel <= max(4 * EPS_LD, cond * EPS_LD)


# ------------------------------------------------------------------ exact cases
@pytest.mark.parametrize('n', [1, 9, 64, 65, 130])
def test_integer_factor_is_reproduced_exactly(n):
    # L with small integer entries: A = L L^T is exact in FP64, and so is every step of the Cholesky of A
    rs = np.random.RandomState(70 + n)
    L = np.tril(rs.randint(-3, 4, size=(n, n)).astype(np.float64), -1) + np.diag(rs.randint(1, 6, size=n).astype(np.float64))
    A = L @ L.T
    assert np.abs(A).max() < 2 ** 52
    assert np.array_equal(xp.chol(A).astype(np.float64), L)
    zi = rs.randint(-5, 6, size=n).astype(np.float64)
    g = L @ zi
    assert np.array_equal(xp.trsv(L, g).astype(np.float64), zi)
    assert xp.backward_error(A, L) == (0.0, 0.0)
    assert xp.solve_backward_error(L, g, zi) == 0.0
    with mp.workdps(40):
        want = -(mp.mpf(float(zi @ zi)) / 2 + sum(mp.log(int(v)) for v in np.diag(L)) + n * mp.log(2 * mp.pi) / 2)
        assert abs(float((_mpf(xp.loglik(A, g)) - want) / want)) < 4 * EPS_LD
    # the measure has teeth: L_00 off by 2^-48 relative puts 2^-47 |A_00| into the residual, 64 ulps
    Lb = L.copy()
    Lb[0, 0] *= 1 + 2.0 ** -48
    comp, norm = xp.backward_error(A, Lb)
    assert comp >= 60 and norm > 0


def test_non_positive_pivot_raises_at_its_row():
    rs = np.random.RandomState(5)
    L0 = np.tril(rs.uniform(-0.5, 0.5, (100, 100)), -1) + np.eye(100)
    d = np.ones(100)
    d[71] = -1e-6
    with pytest.raises(np.linalg.LinAlgError, match='minor 72 '):
        xp.chol(xp.symmetric(L0 @ np.diag(d) @ L0.T))


def test_banded_residual_equals_the_dense_one():
    # the envelope only skips exact zeros: a dense copy of the same product gives the same errors
    K, S = ks(300, 3.0, 4.0, 0.5)
    A = xp.symmetric(K + np.diag(S))
    assert xp.envelope(A).max() > 64
    L = scipy.linalg.cholesky(A, lower=True)
    Ld = L.astype(xp.LD)
    R = np.abs(np.tril(A.astype(xp.LD) - xp._mm(Ld, Ld.T))).astype(np.float64)
    D = np.abs(L) @ np.abs(L).T + xp.UNDERFLOW * 300
    comp, norm = xp.backward_error(A, L)
    # (the two sum the same products in different orders: they agree to the residual's longdouble rounding)
    assert comp == pytest.approx(float(np.where(R == 0, 0, R / D).max()) / xp.EPS, rel=1e-3)
    assert norm == pytest.approx(float(np.linalg.norm(R) / np.linalg.norm(np.tril(A))) / xp.EPS, rel=1e-3)
    Lbad = L.copy()
    Lbad[299, 0] = 1e-300                            # left of the envelope: Cholesky never puts a nonzero there
    with pytest.raises(AssertionError, match='left of the envelope'):
        xp.backward_error(A, Lbad)


# ------------------------------------------------------------------ LAPACK's calibration
LAPACK_COMP, LAPACK_NORM = 12.0, 3.0      # measured on x86-64 with OpenBLAS: 3.6-6.1 and 0.9-1.3 eps


@pytest.mark.parametrize('n', [129, 256])
def test_lapack_backward_error_on_the_families(n):
    mats = ill_conditioned(n)
    for ell in (3.0, 11.0):
        for sf in (4.0, 20.0):
            for sn in (0.05, 0.5):
                K, S = ks(n, ell, sf, sn)
                mats['ks_%g_%g_%g' % (ell, sf, sn)] = xp.symmetric(K + np.diag(S))
    for name, A in mats.items():
        comp, norm = xp.backward_error(A, scipy.linalg.cholesky(A, lower=True))
        print('%-18s LAPACK backward error: componentwise %.2f eps, normwise %.2f eps' % (name, comp, norm))
        assert comp < LAPACK_COMP and norm < LAPACK_NORM, (name, comp, norm)


def test_lapack_loglik_forward_error_at_the_bench_corner():
    # cond(K+S) ~ 4e6 at N = 1000: FP64 through LAPACK is ~1e-13 relative off the truth, far inside the 4e-10 that a
    # tolerance of eps * cond would allow
    n = 1000
    K, S = ks(n, 11.0, 20.0, 0.05)
    A = xp.symmetric(K + np.diag(S))
    g = 0.05 * np.random.RandomState(3).standard_normal(n)
    L = scipy.linalg.cholesky(A, lower=True)
    w = scipy.linalg.solve_triangular(L, g, lower=True)
    f64 = -(0.5 * w @ w + np.log(np.diag(L)).sum() + 0.5 * n * np.log(2 * np.pi))
    truth = xp.loglik(A, g)
    rel = float(abs((f64 - truth) / truth))
    print('LAPACK loglik relative error %.2e at cond %.1e' % (rel, np.linalg.cond(A)))
    assert 1e-16 < rel < 3e-12
    assert xp.solve_backward_error(L, g, w) < 4
