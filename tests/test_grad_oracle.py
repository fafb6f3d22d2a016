"""CPU checks of the log-likelihood gradient: the oracle (oracle/grad_oracle.py) against 40-digit central differences and
against its own longdouble form, and the host logic of ``kcGP.gpK.GPR`` (log-scale / sign conversion of ``dnlZ``,
restarts, where ``optimize`` lands) with the device call replaced by the oracle."""
import numpy as np
import pytest
import scipy.optimize

from oracle import grad_oracle as go
from oracle import xprec as xp

mpmath = pytest.importorskip('mpmath')


def _inputs(n, D, seed):
    rs = np.random.RandomState(seed)
    x = np.arange(n, dtype=np.float64).reshape(n, 1) if D == 1 else rs.uniform(0, 6, size=(n, D))
    return x, rs.standard_normal(n) * 1.3


def _loglik_mp(x, g, hyp):
    """log N(g; 0, K + sn^2 I) at the working precision of mpmath (S_ii = sn^2, as the gradient differentiates it)."""
    n, D = x.shape
    P = len(hyp)
    n_ell = P - 2
    ell = [hyp[0]] * D if n_ell == 1 else list(hyp[:n_ell])
    sf, sn = hyp[n_ell], hyp[n_ell + 1]
    A = mpmath.matrix(n, n)
    for i in range(n):
        for j in range(n):
            s = mpmath.fsum(((mpmath.mpf(x[i, d]) - mpmath.mpf(x[j, d])) / ell[d]) ** 2 for d in range(D))
            A[i, j] = sf ** 2 * mpmath.exp(-s / 2) + (sn ** 2 if i == j else 0)
    L = mpmath.cholesky(A)
    z = mpmath.lu_solve(L, mpmath.matrix([mpmath.mpf(v) for v in g]))           # L z = g
    quad = mpmath.fsum(z[i] ** 2 for i in range(n))
    logdet = 2 * mpmath.fsum(mpmath.log(L[i, i]) for i in range(n))
    return -(quad / 2 + logdet / 2 + n * mpmath.log(2 * mpmath.pi) / 2)


@pytest.mark.parametrize('n,D,ard,hyp', [
    (1, 1, False, (2.0, 1.5, 0.7)),
    (7, 1, False, (2.5, 3.0, 0.4)),
    (12, 1, False, (1.3, 0.8, 1.1)),
    (9, 2, False, (1.7, 2.0, 0.3)),
    (10, 2, True, (1.2, 3.1, 1.6, 0.5)),
    (12, 3, True, (0.9, 2.2, 4.0, 2.5, 0.8)),
])
def test_oracle_gradient_matches_mpmath_central_differences(n, D, ard, hyp):
    mpmath.mp.dps = 40
    x, g = _inputs(n, D, 7 + n)
    hyp = np.array(hyp)
    ll, grad = go.loglik_grad(x, g, hyp, form='cho')
    ll2, grad2 = go.loglik_grad(x, g, hyp, form='inv')
    h = mpmath.mpf('1e-15')
    for p in range(len(hyp)):
        up = [mpmath.mpf(v) for v in hyp]
        dn = [mpmath.mpf(v) for v in hyp]
        up[p] += h * hyp[p]
        dn[p] -= h * hyp[p]
        ref = float((_loglik_mp(x, g, up) - _loglik_mp(x, g, dn)) / (2 * h * hyp[p]))
        for gr in (grad, grad2):
            assert abs(gr[p] - ref) <= 1e-10 * max(1.0, abs(ref)), (p, gr[p], ref)
    assert abs(ll - float(_loglik_mp(x, g, list(hyp)))) <= 1e-12 * abs(ll)
    assert abs(ll - ll2) <= 1e-13 * abs(ll)


@pytest.mark.skipif(not xp.AVAILABLE, reason=xp.REASON)
@pytest.mark.parametrize('ard', [False, True])
def test_longdouble_gradient_matches_fp64_at_n200(ard):
    n = 200
    rs = np.random.RandomState(3)
    if ard:
        x = np.column_stack([np.arange(n, dtype=np.float64), rs.uniform(0, 20, n)])
        hyp = np.array([4.0, 7.0, 2.0, 0.6])
    else:
        x = np.arange(n, dtype=np.float64).reshape(n, 1)
        hyp = np.array([3.0, 2.0, 0.5])
    g = rs.standard_normal(n)
    ll_x, grad_x, mag = go.loglik_grad_xprec(x, g, hyp)
    for form in ('cho', 'inv'):
        ll, grad = go.loglik_grad(x, g, hyp, form=form)
        assert abs(ll - float(ll_x)) <= 1e-13 * abs(ll)
        err = np.abs(grad - np.asarray(grad_x, dtype=np.float64))
        assert np.all(err <= 1e-12 * np.asarray(mag, dtype=np.float64)), (form, err, mag)


# --------------------------------------------------------------------------------------------- GPR host logic
def _oracle_call(x, g, hyp, jitter_policy=None, workspace=None, max_wave=None):
    g = np.atleast_2d(np.asarray(g, dtype=np.float64))
    hyp = np.atleast_2d(np.asarray(hyp, dtype=np.float64))
    ll, grad, info = np.empty(len(hyp)), np.empty(hyp.shape), np.zeros(len(hyp), dtype=np.int32)
    for b in range(len(hyp)):
        try:
            ll[b], grad[b] = go.loglik_grad(x, g[b], hyp[b], form='cho')
        except np.linalg.LinAlgError:
            ll[b], grad[b], info[b] = np.nan, np.nan, -1
    return ll, grad, info


@pytest.fixture
def gpr_on_oracle(gp, monkeypatch):
    monkeypatch.setattr(gp.ops, 'loglik_grad_batched', _oracle_call)
    n = 80
    x, y = gp.synthetic.ih45_series(n)
    model = gp.kcGP.gpK.GPR()
    model.setData(x, y - y.mean())
    model.setPrior(kernel=gp.kcGP.covK.RBF(np.log(2.0), np.log(3.0)))
    model.setNoise(log_sigma=np.log(1.5))
    return model


def test_gpr_dnlz_is_the_log_scale_negative_gradient(gp, gpr_on_oracle):
    m = gpr_on_oracle
    nlZ, dnlZ, post = m.getPosterior()
    assert post is None and dnlZ.mean == []
    theta = np.array([2.0, 3.0, 1.5])
    ll, grad = go.loglik_grad(m.x, m.y[:, 0], theta)
    assert nlZ == -ll
    np.testing.assert_allclose(dnlZ.cov, -theta[:2] * grad[:2], rtol=1e-14)
    np.testing.assert_allclose(dnlZ.lik, [-theta[2] * grad[2]], rtol=1e-14)
    # and the derivative of nlZ along the log hyper-parameters by central differences
    h = 1e-6
    base = np.log(theta)
    for p, d in enumerate(list(dnlZ.cov) + list(dnlZ.lik)):
        up, dn = base.copy(), base.copy()
        up[p] += h
        dn[p] -= h
        fd = (-go.loglik_grad(m.x, m.y[:, 0], np.exp(up))[0] + go.loglik_grad(m.x, m.y[:, 0], np.exp(dn))[0]) / (2 * h)
        assert abs(fd - d) <= 1e-6 * max(1.0, abs(d)), (p, fd, d)
    with pytest.raises(NotImplementedError):
        m.setPrior(mean=object())


def test_gpr_restarts_keep_the_best(gp, gpr_on_oracle, monkeypatch):
    m = gpr_on_oracle
    runs = []
    real = scipy.optimize.minimize

    def spy(*a, **k):
        r = real(*a, **k)
        runs.append(r)
        return r

    monkeypatch.setattr(gp.kcGP.gpK.scipy.optimize, 'minimize', spy)
    m.setOptimizer(method='BFGS', num_restarts=3, covRange=[(-1.0, 3.0), (-1.0, 3.0)], likRange=[(-1.0, 2.0)])
    np.random.seed(11)
    nlZ, _, _ = m.optimize(numIterations=3)
    assert len(runs) == 4
    funs = [r.fun for r in runs]
    assert len(set(np.round(funs, 6))) > 1                     # the starts did lead to different places
    best = runs[int(np.argmin(funs))]
    assert nlZ == min(funs)
    np.testing.assert_array_equal(np.concatenate([m.covfunc.hyp, [np.log(m.likfunc.sn)]]), best.x)


def test_gpr_optimize_lands_where_scipy_lands_on_the_oracle(gp, gpr_on_oracle):
    m = gpr_on_oracle
    x, y = m.x, m.y[:, 0]
    h0 = np.log([2.0, 3.0, 1.5])

    def f(h):
        ll, grad = go.loglik_grad(x, y, np.exp(h))
        return -ll, -np.exp(h) * grad

    ref = scipy.optimize.minimize(f, h0, jac=True, method='L-BFGS-B', options={'maxiter': 40})
    nlZ, dnlZ, _ = m.optimize(numIterations=40)
    assert abs(nlZ - ref.fun) <= 1e-12 * abs(ref.fun)
    np.testing.assert_allclose(np.concatenate([m.covfunc.hyp, [np.log(m.likfunc.sn)]]), ref.x, rtol=1e-12, atol=1e-12)
    assert np.linalg.norm(list(dnlZ.cov) + list(dnlZ.lik)) < 1e-3
