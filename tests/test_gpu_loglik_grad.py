"""gpmc_loglik_grad_batched on the device: the gradient of the GP log marginal likelihood against the longdouble and FP64
oracles (oracle/grad_oracle.py), its loglik against gpmc_loglik_batched, exactness of the band skips, waves, failed
items, the C ABI, and kcGP.gpK.GPR built on it.  B200 only."""
import numpy as np
import pytest

from oracle import grad_oracle as go
from oracle import sds_oracle as so
from oracle import xprec as xp

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -53
# corners of the bench bracket (tests/test_gpu_backward_error.py) and a well-conditioned control
WORST, MILD, CONTROL = (11.0, 20.0, 0.05), (3.0, 4.0, 0.5), (1.5, 1.0, 1.0)


def _grad(gp, x, G, H, **kw):
    ll, grad, info = gp.ops.loglik_grad_batched(x, G, H, **kw)
    return ll.cpu().numpy(), grad.cpu().numpy(), info.cpu().numpy()


def _iso_items(n, seed):
    rs = np.random.RandomState(seed)
    x = np.arange(n, dtype=np.float64).reshape(n, 1)
    H = np.array([WORST, MILD, CONTROL])
    G = H[:, 2:3] * rs.standard_normal((3, n)) + 0.3
    return x, G, H


def _ard_items(n, seed):
    rs = np.random.RandomState(seed)
    x = np.column_stack([np.arange(n, dtype=np.float64), rs.uniform(0, 30, n)])
    H = np.array([[11.0, 6.0, 20.0, 0.05], [3.0, 5.0, 4.0, 0.5], [1.5, 2.5, 1.0, 1.0]])
    G = H[:, 3:4] * rs.standard_normal((3, n)) + 0.3
    return x, G, H


def _fp64_orders():
    """FP64 Cholesky factors summed in different orders: LAPACK's and left-looking panels of 8, 32 and 128 columns (the
    orders tests/test_gpu_backward_error.py measures FP64's own error over)."""
    from test_gpu_backward_error import FP64_ORDERS, _blocked_chol
    return [None if nb is None else (lambda A, nb=nb: _blocked_chol(A, nb)) for nb in FP64_ORDERS]


def _errors_vs_xprec(x, g, hyp, grad, ll, jitter=0.0):
    """Relative errors against the longdouble truth: (device gradient |err_p| / mag_p, worst FP64 |err_p| / mag_p over
    the two oracle forms on every summation order of the factor, device loglik, worst FP64 loglik).  mag_p = the sum of
    the magnitudes of component p's terms, 0.5 sum_ij |alpha_i alpha_j - W_ij| |dA_ij/dtheta_p|."""
    ll_t, g_t, mag = go.loglik_grad_xprec(x, g, hyp, jitter=jitter)
    ll_t, g_t, mag = float(ll_t), np.asarray(g_t, dtype=np.float64), np.asarray(mag, dtype=np.float64)
    rel = lambda e: np.where(e == 0, 0.0, e / np.where(mag > 0, mag, 1.0) + np.where(mag > 0, 0.0, np.inf))   # no terms: exact 0
    e_g, e_ll = np.zeros(len(hyp)), 0.0
    for chol in _fp64_orders():
        for form in ('cho', 'inv'):
            l_o, g_o = go.loglik_grad(x, g, hyp, form=form, jitter=jitter, chol=chol)
            e_g = np.maximum(e_g, rel(np.abs(g_o - g_t)))
            e_ll = max(e_ll, abs((l_o - ll_t) / ll_t))
    return rel(np.abs(grad - g_t)), e_g, abs((ll - ll_t) / ll_t), e_ll


def _hold(dev, f64, what):
    """The rule of tests/test_gpu_backward_error.py: within 8x the worst error FP64 itself makes on the batch (every item,
    every summation order, both forms), floor 16 eps.  One item's FP64 error is not FP64's error: which rounding pattern an
    item draws scatters it by 10x between orders, and the device's factor is held to 16x LAPACK's backward error there."""
    bound = max(8 * max(f64), 16 * EPS)
    assert max(dev) <= bound, (what, max(dev), max(f64))
    return max(dev) / max(max(f64), 16 * EPS)


@pytest.mark.skipif(not xp.AVAILABLE, reason=xp.REASON)
@pytest.mark.parametrize('n', [1, 2, 8, 33, 127, 128, 129, 200, 455, 512])
def test_gradient_vs_longdouble(gp, n):
    """Every gradient component and the loglik of ISO and ARD items (the bench bracket's corners and a control) against
    the longdouble truth."""
    errs = []
    for items in (_iso_items, _ard_items):
        x, G, H = items(n, 100 + n)
        ll, grad, info = _grad(gp, x, G, H)
        assert np.all(info == 0), info
        errs += [_errors_vs_xprec(x, G[b], H[b], grad[b], ll[b]) for b in range(len(H))]
    rg = _hold([e[0].max() for e in errs], [e[1].max() for e in errs], 'gradient')
    rl = _hold([e[2] for e in errs], [e[3] for e in errs], 'loglik')
    per_item = max(float(np.max(e[0] / np.maximum(e[1], 16 * EPS))) for e in errs)
    print('N=%d: worst error / worst FP64 error on the batch: gradient %.2f, loglik %.2f; worst per item and component %.2f'
          % (n, rg, rl, per_item))


@pytest.mark.parametrize('n', [1000, 2048, 4096])
def test_gradient_large_vs_fp64_oracle_and_central_difference(gp, n):
    rs = np.random.RandomState(n)
    x = np.arange(n, dtype=np.float64).reshape(n, 1)
    hyp = np.array(MILD)
    g = hyp[2] * rs.standard_normal(n)
    ll, grad, info = _grad(gp, x, g[None], hyp[None])
    assert info[0] == 0
    l_c, g_c = go.loglik_grad(x, g, hyp, form='cho')
    l_i, g_i = go.loglik_grad(x, g, hyp, form='inv')
    spread = np.abs(g_c - g_i)
    assert np.all(np.abs(grad[0] - g_c) <= 8 * spread + 1e-12 * np.abs(g_c)), (grad[0], g_c, g_i)
    assert abs(ll[0] - l_c) <= 1e-12 * abs(l_c)
    # central difference of gpmc_loglik_batched along a random direction in log space
    d = rs.standard_normal(3)
    h = 1e-4
    Hp = np.stack([hyp * np.exp(h * d), hyp * np.exp(-h * d)])
    lp, _ = gp.ops.loglik_batched(x, np.stack([g, g]), Hp)
    lp = lp.cpu().numpy()
    fd = (lp[0] - lp[1]) / (2 * h)
    an = float(np.dot(grad[0], hyp * d))
    assert abs(fd - an) <= 1e-6 * abs(an), (fd, an)


def test_loglik_output_matches_loglik_batched(gp):
    """The loglik of the gradient call against gpmc_loglik_batched on the same inputs (the bench shapes' dense layout and a
    compact-layout call): 1e-13 relative; whether they are bitwise equal is printed."""
    for n, B, nell in ((1024, 16, 1), (512, 64, 4), (4096, 4, 1)):
        x = gp.synthetic.ard_inputs(n, nell)[0] if nell > 1 else np.arange(n, dtype=np.float64).reshape(n, 1)
        G, H = gp.synthetic.loglik_batch(B, n, n_ell=nell)
        ll, _, info = _grad(gp, x, G, H)
        ref, info2 = gp.ops.loglik_batched(x, G, H)
        ref = ref.cpu().numpy()
        assert np.array_equal(info, info2.cpu().numpy())
        ok = info == 0
        assert np.all(np.abs(ll[ok] - ref[ok]) <= 1e-13 * np.abs(ref[ok]))
        print('N=%d B=%d D=%d: loglik bitwise equal to gpmc_loglik_batched: %s' % (n, B, nell, np.array_equal(ll[ok], ref[ok])))


@pytest.mark.parametrize('n,B,nell', [(2048, 4, 1), (1000, 6, 2), (300, 5, 1)])
def test_band_skips_are_exact_and_calls_repeat(gp, n, B, nell):
    rs = np.random.RandomState(n)
    x = np.arange(n, dtype=np.float64).reshape(n, 1) if nell == 1 else np.column_stack([np.arange(n, dtype=np.float64), rs.uniform(0, 50, n)])
    G, H = gp.synthetic.loglik_batch(B, n, n_ell=nell)
    on = _grad(gp, x, G, H)
    again = _grad(gp, x, G, H)
    try:
        gp.ops.set_tuning(15, 0)
        off = _grad(gp, x, G, H)
    finally:
        gp.ops.set_tuning(15, 1)
    for a, b, c in zip(on, again, off):
        assert np.array_equal(a, b, equal_nan=True)
        assert np.array_equal(a, c, equal_nan=True)
    assert np.all(np.isfinite(on[1][on[2] == 0]))


def test_waves_agree(gp):
    n, B = 700, 7
    x = np.arange(n, dtype=np.float64).reshape(n, 1)
    G, H = gp.synthetic.loglik_batch(B, n)
    ref = _grad(gp, x, G, H)
    for w in (1, 3):
        ll, grad, info = _grad(gp, x, G, H, max_wave=w, workspace=gp.ops.Workspace())
        assert np.array_equal(info, ref[2])
        ok = info == 0
        assert np.all(np.abs(ll[ok] - ref[0][ok]) <= 1e-12 * np.abs(ref[0][ok]))
        assert np.all(np.abs(grad[ok] - ref[1][ok]) <= 1e-12 * np.abs(ref[1][ok]).max(axis=1, keepdims=True))


def test_jitter_ladder_item_matches_oracle_at_the_jitter(gp):
    """An item whose K+S is numerically singular (sn = 1e-7, long length-scale): the ladder rescues it, and its loglik and
    gradient are those of A + jitter I for the rung the ladder stopped at (the jitter held constant)."""
    n = 200
    x = np.arange(n, dtype=np.float64).reshape(n, 1)
    rs = np.random.RandomState(5)
    H = np.array([MILD, (40.0, 10.0, 1e-7), CONTROL])
    G = rs.standard_normal((3, n))
    ll, grad, info = _grad(gp, x, G, H)
    assert np.all(info == 0) and np.all(np.isfinite(grad))
    _, K, A = go.matrix(x, H[1])
    mean = np.mean(np.diagonal(A))
    cands = [0.0] + [mean * 1e-6 * 10 ** k for k in range(5)]
    lls = []
    for j in cands:
        try:
            lls.append(go.loglik_grad(x, G[1], H[1], jitter=j)[0])
        except np.linalg.LinAlgError:
            lls.append(np.nan)
    k = int(np.nanargmin(np.abs(np.array(lls) - ll[1])))
    assert cands[k] > 0, 'the item did not need the ladder'
    e = _errors_vs_xprec(x, G[1], H[1], grad[1], ll[1], jitter=cands[k])
    _hold([e[0].max()], [e[1].max()], 'gradient')
    _hold([e[2]], [e[3]], 'loglik')
    # the other rows are what they are without the bad item
    H2 = H.copy()
    H2[1] = MILD
    ll2, grad2, _ = _grad(gp, x, G, H2)
    assert np.array_equal(ll[[0, 2]], ll2[[0, 2]]) and np.array_equal(grad[[0, 2]], grad2[[0, 2]])


def test_failed_and_invalid_items_give_nan_rows(gp):
    n = 200
    x = np.arange(n, dtype=np.float64).reshape(n, 1)
    rs = np.random.RandomState(6)
    good = np.array([MILD, CONTROL, WORST, MILD, CONTROL, MILD])
    G = rs.standard_normal((6, n))
    ll0, g0, _ = _grad(gp, x, G, good)
    # no jitter: the singular item fails with info > 0
    H = good.copy()
    H[1] = (40.0, 10.0, 1e-7)
    ll, grad, info = _grad(gp, x, G, H, jitter_policy=gp.JITTER_NONE)
    assert info[1] > 0 and np.isnan(ll[1]) and np.all(np.isnan(grad[1]))
    keep = [0, 2, 3, 4, 5]
    ll0n, g0n, _ = _grad(gp, x, G, good, jitter_policy=gp.JITTER_NONE)
    assert np.array_equal(ll[keep], ll0n[keep]) and np.array_equal(grad[keep], g0n[keep])
    # NaN / negative hyper-parameters: a NaN length-scale and a negative sf fail the factorisation (info = -1); a negative
    # sn leaves K+S positive definite, but the natural-scale gradient is defined for positive parameters only
    H = good.copy()
    H[1, 0] = np.nan
    H[3, 1] = -1.0
    H[4, 2] = -0.5
    ll, grad, info = _grad(gp, x, G, H)
    assert info[1] != 0 and info[3] != 0 and np.isnan(ll[1]) and np.isnan(ll[3])
    assert all(np.all(np.isnan(grad[b])) for b in (1, 3, 4))
    keep = [0, 2, 5]
    assert np.array_equal(ll[keep], ll0[keep]) and np.array_equal(grad[keep], g0[keep])


def test_c_abi(gp):
    import torch
    from gpmc_b200 import _lib
    lib = _lib.load()
    assert hasattr(lib, 'gpmc_loglik_grad_batched')
    n, B = 300, 3
    x = torch.arange(n, dtype=torch.float64, device='cuda').reshape(n, 1)
    G, H = gp.synthetic.loglik_batch(B, n)
    Gd, Hd = torch.tensor(G).cuda(), torch.tensor(H).cuda()
    ll = torch.empty(B, dtype=torch.float64, device='cuda')
    gr = torch.empty((B, 3), dtype=torch.float64, device='cuda')
    info = torch.empty(B, dtype=torch.int32, device='cuda')
    one = lib.gpmc_workspace_bytes(_lib.OP_LOGLIK_GRAD, n, 1, 1)
    allb = lib.gpmc_workspace_bytes(_lib.OP_LOGLIK_GRAD, n, 1, B)
    assert one >= 2 * n * n * 8 and allb >= one
    ws = torch.empty(allb, dtype=torch.uint8, device='cuda')

    def call(Bc=B, P=3, kind=_lib.KIND_SE_ISO, nbytes=allb):
        return lib.gpmc_loglik_grad_batched(x.data_ptr(), n, 1, Gd.data_ptr(), Hd.data_ptr(), Bc, P, kind, gp.JITTER_PYGPS,
                                            ll.data_ptr(), gr.data_ptr(), info.data_ptr(), ws.data_ptr(), nbytes, None)
    assert call() == 0
    first = gr.cpu().numpy().copy()
    assert call(Bc=0) == 0
    assert call(P=4) == -22 and len(lib.gpmc_last_error()) > 0
    assert call(kind=7) == -22
    assert call(nbytes=1024) == -12
    assert call() == 0 and np.array_equal(gr.cpu().numpy(), first)
    # a workspace of the one-item size serves a one-item call
    ws1 = torch.empty(one, dtype=torch.uint8, device='cuda')
    rc = lib.gpmc_loglik_grad_batched(x.data_ptr(), n, 1, Gd.data_ptr(), Hd.data_ptr(), 1, 3, _lib.KIND_SE_ISO, gp.JITTER_PYGPS,
                                      ll.data_ptr(), gr.data_ptr(), info.data_ptr(), ws1.data_ptr(), one, None)
    assert rc == 0 and np.array_equal(gr.cpu().numpy()[0], first[0])


# --------------------------------------------------------------------------------------------------------- GPR
def test_gpr_optimize_matches_scipy_on_the_oracle(gp):
    import scipy.optimize
    x, y = gp.synthetic.ih45_series(455)
    yc = y - y.mean()
    m = gp.kcGP.gpK.GPR()
    m.setData(x, yc)
    m.setPrior(kernel=gp.kcGP.covK.RBF(np.log(1.0), np.log(10.0)))
    m.setNoise(log_sigma=np.log(1.2))
    h0 = np.log([1.0, 10.0, 1.2])
    nlZ, dnlZ, post = m.optimize(numIterations=40)

    def f(h):
        ll, g = go.loglik_grad(x, yc, np.exp(h))
        return -ll, -np.exp(h) * g
    ref = scipy.optimize.minimize(f, h0, jac=True, method='L-BFGS-B', options={'maxiter': 40})
    print('GPR nlZ %.12f (oracle L-BFGS-B %.12f), theta %s' % (nlZ, ref.fun, np.exp(m.optim_result.x)))
    assert abs(nlZ - ref.fun) <= 1e-8 * abs(ref.fun)
    assert np.linalg.norm(list(dnlZ.cov) + list(dnlZ.lik)) <= 1e-4
    assert post is None


def test_gpr_predict_and_inf_mcmc(gp):
    import types
    n = 200
    x, y = gp.synthetic.ih45_series(n)
    yc = y - y.mean()
    xs = np.linspace(-3.5, n + 2.5, 37).reshape(-1, 1)
    m = gp.kcGP.gpK.GPR()
    m.setData(x, yc)
    m.setPrior(kernel=gp.kcGP.covK.RBF(np.log(5.0), np.log(4.0)))
    m.setNoise(log_sigma=np.log(2.5))
    ym, ys2, fm, fs2, lp = m.predict(xs, ys=np.zeros(37))
    assert m.xs.shape == (37, 1)
    hyp = np.array([5.0, 4.0, 2.5])
    fmu, fv, _ = gp.ops.predict_batched(x, xs, yc[None], hyp[None])
    np.testing.assert_allclose(fm[:, 0], fmu.cpu().numpy()[0], rtol=1e-10, atol=1e-10)
    np.testing.assert_allclose(fs2[:, 0], np.maximum(fv.cpu().numpy()[0], 0), rtol=1e-10, atol=1e-10)
    # oracle predictive with A = K + sn^2 I
    K = so.cov_matrix(x, hyp)
    Ks = so.kcgp_shim.RBF(np.log(5.0), np.log(4.0)).getCovMatrix(x=x, z=xs, mode='cross')
    A = K + np.eye(n) * 2.5 ** 2
    f_o = Ks.T @ np.linalg.solve(A, yc)
    v_o = 16.0 - np.einsum('ij,ij->j', Ks, np.linalg.solve(A, Ks))
    np.testing.assert_allclose(fm[:, 0], f_o, rtol=1e-10, atol=1e-10)
    np.testing.assert_allclose(fs2[:, 0], np.maximum(v_o, 0), rtol=1e-10, atol=1e-10)
    np.testing.assert_allclose(ys2, fs2 + 2.5 ** 2, rtol=1e-15)
    np.testing.assert_allclose(lp, -ym ** 2 / (2 * ys2) - 0.5 * np.log(2 * np.pi * ys2), rtol=1e-14)
    # inf_mcmc reads x, y, xs, meanfunc, covfunc, likfunc from a GPR as from the hand-built namespace
    f = 0.5 * yc[:, None] + 0.1 * np.random.RandomState(3).standard_normal((n, 4))
    lik = gp.kcGP.likK.TruncatedGauss2(upper=100 - y.mean(), lower=0 - y.mean(), log_sigma=np.log(2.5))
    m.setData(x, y)
    m.likfunc = lik
    zero = types.SimpleNamespace(getMean=lambda a: np.zeros((a.shape[0], 1)))
    ns = types.SimpleNamespace(x=x, y=y.reshape(-1, 1), xs=xs, meanfunc=zero, covfunc=gp.kcGP.covK.RBF(np.log(5.0), np.log(4.0)),
                               likfunc=lik)
    a = gp.kcMCMC.sliceSample.inf_mcmc(f, m)
    b = gp.kcMCMC.sliceSample.inf_mcmc(f, ns)
    for u, v in zip(a, b):
        assert np.array_equal(u, v)
