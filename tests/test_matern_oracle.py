"""CPU checks of the Matern covariance kinds (d = 1, 3, 5): the oracle's restatement of pyGPs 1.3.4 ``cov.Matern`` and
its gradient (oracle/matern_oracle.py) against mpmath at 40 digits, the oracle's kernel switch, and the host-side argument
handling of ``kcGP.covK.Matern``, ``kcGP.gpK.GPR.setPrior`` and the ``kind`` keyword of ``ops``."""
import numpy as np
import pytest

from oracle import kcgp_shim
from oracle import matern_oracle as mo
from oracle import sds_oracle as so

mpmath = pytest.importorskip('mpmath')
EPS = 2.0 ** -53


def _f_mp(d, t):
    if d == 1:
        return mpmath.mpf(1)
    if d == 3:
        return 1 + t
    return 1 + t + t * t / 3


def _k_mp(d, ell, sf, a, b):
    """K(a, b) at the working precision of mpmath, from the exact inputs."""
    s = mpmath.fsum((mpmath.sqrt(d) * (mpmath.mpf(p) - mpmath.mpf(q)) / ell) ** 2 for p, q in zip(a, b))
    t = mpmath.sqrt(s)
    return sf ** 2 * _f_mp(d, t) * mpmath.exp(-t), t


@pytest.mark.parametrize('d', [1, 3, 5])
@pytest.mark.parametrize('D', [1, 2])
def test_shim_matern_matches_mpmath(d, D):
    mpmath.mp.dps = 40
    rs = np.random.RandomState(10 * d + D)
    ell, sf = 0.7, 1.9
    x = rs.uniform(-3, 3, size=(12, D))
    # pairs whose t lies just below, at and past the point where exp(-t) underflows (t ~ 745.13)
    far = []
    for t in (700.0, 744.0, 744.9, 745.1, 745.2, 746.0, 800.0):
        far.append(np.full(D, t * ell / np.sqrt(d) / np.sqrt(D)))
    z = np.vstack([x[:3], np.zeros((1, D)), np.array(far)])
    cov = mo.Matern(np.log(ell), d, np.log(sf))
    for K, A, B in ((cov.getCovMatrix(x=x, mode='train'), x, x), (cov.getCovMatrix(x=x, z=z, mode='cross'), x, z)):
        assert K.shape == (A.shape[0], B.shape[0])
        for i in range(A.shape[0]):
            for j in range(B.shape[0]):
                ref, t = _k_mp(d, mpmath.mpf(np.exp(np.log(ell))), mpmath.mpf(np.exp(np.log(sf))), A[i], B[j])
                # the rounding of u and s is a relative error of a few eps in t, which exp(-t) turns into t times that in K;
                # where exp(-t) is subnormal it carries an absolute error of up to 2^-1074, which sf2 * f_d(t) scales
                tol = (float(t) + 8) * 8 * EPS * float(ref) + 2 * float(sf ** 2 * _f_mp(d, t)) * 2 ** -1074
                assert abs(K[i, j] - float(ref)) <= tol, (d, i, j, K[i, j], float(ref), float(t))
    # past the underflow point K is +0; on the diagonal it is sf2
    K0 = cov.getCovMatrix(x=np.zeros((1, D)), z=np.array(far), mode='cross')[0]
    assert K0[-1] == 0.0 and K0[-2] == 0.0 and K0[0] > 0.0
    np.testing.assert_array_equal(np.diagonal(cov.getCovMatrix(x=x, mode='train')), np.exp(2 * np.log(sf)))
    np.testing.assert_array_equal(cov.getCovMatrix(z=x, mode='self_test'), np.full((12, 1), np.exp(2 * np.log(sf))))


def test_shim_matern_rejects_other_d():
    for d in (0, 2, 4):
        with pytest.raises(ValueError):
            mo.Matern(0.0, d, 0.0)
        with pytest.raises(ValueError):
            with mo.kernel(d):
                pass


def test_kernel_switch_is_scoped():
    """mo.kernel(d) routes the restatements' isotropic kernel to the Matern one inside the block only, also when the
    block raises; the ARD kernel and the default are untouched."""
    rs = np.random.RandomState(5)
    x = rs.uniform(0, 9, size=(20, 1))
    hyp = np.array([1.7, 2.2, 0.4])
    rbf = kcgp_shim.RBF
    K = kcgp_shim.RBF(np.log(hyp[0]), np.log(hyp[1])).getCovMatrix(x=x, mode='train')
    np.testing.assert_array_equal(so.cov_matrix(x, hyp), K)
    Km = mo.cov_matrix(x, hyp, 3)
    np.testing.assert_array_equal(Km, mo.Matern(np.log(hyp[0]), 3, np.log(hyp[1])).getCovMatrix(x=x, mode='train'))
    assert not np.array_equal(Km, K)
    assert kcgp_shim.RBF is rbf
    np.testing.assert_array_equal(so.cov_matrix(x, hyp), K)
    with pytest.raises(RuntimeError):
        with mo.kernel(5):
            raise RuntimeError('inside')
    assert kcgp_shim.RBF is rbf
    with pytest.raises(ValueError):
        mo.cov_matrix(np.column_stack([x, x]), np.array([1.0, 2.0, 2.2, 0.4]), 3)


def _loglik_mp(x, g, hyp, d):
    """log N(g; 0, K + sn^2 I) with the Matern K at the working precision of mpmath."""
    n = x.shape[0]
    ell, sf, sn = hyp
    A = mpmath.matrix(n, n)
    for i in range(n):
        for j in range(n):
            A[i, j] = _k_mp(d, ell, sf, x[i], x[j])[0] + (sn ** 2 if i == j else 0)
    L = mpmath.cholesky(A)
    z = mpmath.lu_solve(L, mpmath.matrix([mpmath.mpf(v) for v in g]))
    quad = mpmath.fsum(z[i] ** 2 for i in range(n))
    logdet = 2 * mpmath.fsum(mpmath.log(L[i, i]) for i in range(n))
    return -(quad / 2 + logdet / 2 + n * mpmath.log(2 * mpmath.pi) / 2)


@pytest.mark.parametrize('d', [1, 3, 5])
@pytest.mark.parametrize('n,D,hyp', [(8, 1, (2.5, 1.7, 0.4)), (9, 2, (1.3, 0.8, 0.9))])
def test_matern_gradient_oracle_matches_mpmath_central_differences(d, n, D, hyp):
    mpmath.mp.dps = 40
    rs = np.random.RandomState(3 * n + d)
    x = np.arange(n, dtype=np.float64).reshape(n, 1) if D == 1 else rs.uniform(0, 5, size=(n, D))
    g = rs.standard_normal(n) * 1.3
    hyp = np.array(hyp)
    ll, grad = mo.loglik_grad(x, g, hyp, d, form='cho')
    ll2, grad2 = mo.loglik_grad(x, g, hyp, d, form='inv')
    h = mpmath.mpf('1e-15')
    for p in range(3):
        up = [mpmath.mpf(v) for v in hyp]
        dn = [mpmath.mpf(v) for v in hyp]
        up[p] += h * hyp[p]
        dn[p] -= h * hyp[p]
        ref = float((_loglik_mp(x, g, up, d) - _loglik_mp(x, g, dn, d)) / (2 * h * hyp[p]))
        for gr in (grad, grad2):
            assert abs(gr[p] - ref) <= 1e-10 * max(1.0, abs(ref)), (d, p, gr[p], ref)
    assert abs(ll - float(_loglik_mp(x, g, list(hyp), d))) <= 1e-12 * abs(ll)
    assert abs(ll - ll2) <= 1e-13 * abs(ll)


# ----------------------------------------------------------------------------------------- host-side arguments
def test_covk_matern_arguments(gp):
    covK = gp.kcGP.covK
    for d, kind in ((1, gp.ops.KIND_MATERN1), (3, gp.ops.KIND_MATERN3), (5, gp.ops.KIND_MATERN5)):
        k = covK.Matern(np.log(2.0), d, np.log(0.5))
        assert k.kind == kind and k.hyp == [np.log(2.0), np.log(0.5)]
    assert covK.Matern().d == 3
    for bad in (0, 2, 4, 7, 3.5, None):
        with pytest.raises(ValueError):
            covK.Matern(0.0, bad, 0.0)
    z = np.zeros((4, 1))
    np.testing.assert_array_equal(covK.Matern(0.0, 5, np.log(3.0)).getCovMatrix(z=z, mode='self_test'),
                                  np.full((4, 1), np.exp(2 * np.log(3.0))))
    with pytest.raises(ValueError):
        covK.Matern().getCovMatrix(x=z, mode='test')


def test_gpr_set_prior_accepts_matern(gp):
    covK = gp.kcGP.covK
    m = gp.kcGP.gpK.GPR()
    assert m._kind_kw() == {}
    k = covK.Matern(np.log(2.0), 5, np.log(1.0))
    m.setPrior(kernel=k)
    assert m.covfunc is k and m._kind_kw() == {'kind': gp.ops.KIND_MATERN5}
    m.setPrior(kernel=covK.RBF())
    assert m._kind_kw() == {}
    with pytest.raises(NotImplementedError):
        m.setPrior(kernel=object())


def test_ops_kind_inference_unchanged(gp):
    ops = gp.ops
    assert (ops.KIND_SE_ISO, ops.KIND_SE_ARD, ops.KIND_MATERN1, ops.KIND_MATERN3, ops.KIND_MATERN5) == (0, 1, 2, 3, 4)
    for D, P, kind in ((1, 3, 0), (4, 3, 0), (4, 6, 1), (2, 4, 1), (1, 3, 0)):
        assert ops.kind_of(D, P) == kind
        assert ops._kind(D, P, None) == kind
    with pytest.raises(ValueError):
        ops._kind(4, 5, None)
    assert ops._kind(1, 3, ops.KIND_MATERN3) == 3
    assert ops._kind(2, 3, np.int64(4)) == 4
