"""The Matern covariance kinds (GPMC_KIND_MATERN1/3/5, d = 2 nu = 1, 3, 5) on the device, against the oracle's restatement
of pyGPs 1.3.4 ``cov.Matern`` (oracle/matern_oracle.py): assembly, log-likelihood (band, envelope and compact layout bit for bit
against the dense path), gradient, GPR, prediction and the samplers, and the C ABI's kind validation.  B200 only."""
import ctypes

import numpy as np
import pytest

from oracle import matern_oracle as mo

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -53
DS = [1, 3, 5]
KIND = {1: 2, 3: 3, 5: 4}
ENV_ROWS, NB = 64, 128
RTOL_HYP = 1e-12
F_RES_FACTOR, F_ABS_CAP = 12.0, 5e-2        # the SDS f' policy of DESIGN.md section 4 (tests/test_gpu_sds.py)


def _t(x, z, ell, d):
    from scipy.spatial.distance import cdist
    return np.sqrt(cdist(np.sqrt(d) * x / ell, np.sqrt(d) * z / ell, 'sqeuclidean'))


def _f(t, d):
    return np.ones_like(t) if d == 1 else (1 + t if d == 3 else 1 + t * (1 + t / 3))


def _k_bound(ref, t, sf2, d):
    """Elementwise bound of |device K - oracle K|.  u and s are rounded in the same order on both sides, but the device's
    exp differs from numpy's by up to an ulp or two, and one ulp of ell or u is a relative error of eps * t in
    exp(-t) (DESIGN.md section 4 says the same of SE's s / 2): (t + 8) 8 eps relative.  Where exp(-t) is subnormal both
    sides carry an absolute error of 2^-1074 scaled by sf2 f_d(t) (and the device's exp returns +0 from t = 745 on, numpy's
    from 745.13)."""
    return (t + 8) * 8 * EPS * np.abs(ref) + 2 * sf2 * _f(t, d) * 2.0 ** -1074


def _inputs(n, D, seed, span=30.0):
    rs = np.random.RandomState(seed)
    return np.sort(rs.uniform(0, span, size=(n, D)), axis=0)


# ------------------------------------------------------------------------------------------------------ assembly
@pytest.mark.parametrize('d', DS)
@pytest.mark.parametrize('D', [1, 3, 5])
def test_assembly_train_cross_self_test_against_shim(gp, d, D):
    """D = 5 takes the generic-D instantiation, D = 1 and 3 the unrolled ones; ell from 0.02 (K mostly underflowed, both
    sides of the underflow point present) to 40."""
    x = _inputs(150, D, d + D, span=60.0)
    z = _inputs(37, D, 100 + d, span=70.0)
    for ell, sf in ((0.02, 1.3), (0.9, 2.5), (40.0, 0.4)):
        h = np.array([ell, sf, 0.5])
        K = gp.ops.cov_assemble(x, h[None], kind=KIND[d]).cpu().numpy()[0, :, :150]
        cov = mo.Matern(np.log(ell), d, np.log(sf))
        ref = cov.getCovMatrix(x=x, mode='train')
        ell_r, sf2 = np.exp(np.log(ell)), np.exp(2 * np.log(sf))
        assert np.all(np.abs(K - ref) <= _k_bound(ref, _t(x, x, ell_r, d), sf2, d))
        assert np.array_equal(np.diagonal(K), np.full(150, sf2))
        Kc = gp.ops.cov_cross(x, z, h, kind=KIND[d]).cpu().numpy()
        refc = cov.getCovMatrix(x=x, z=z, mode='cross')
        assert np.all(np.abs(Kc - refc) <= _k_bound(refc, _t(x, z, ell_r, d), sf2, d))
        # the kcGP stand-in routes the same calls
        m = gp.kcGP.covK.Matern(np.log(ell), d, np.log(sf))
        assert np.array_equal(m.getCovMatrix(x=x, mode='train'), K)
        assert np.array_equal(m.getCovMatrix(x=x, z=z, mode='cross'), Kc)
        assert np.array_equal(m.getCovMatrix(z=z, mode='self_test'), cov.getCovMatrix(z=z, mode='self_test'))


@pytest.mark.parametrize('d', DS)
def test_device_exp_is_zero_past_the_band_threshold(gp, d):
    """The Matern band rule needs K = +0 wherever t > 745.14: pairs at t just past it and far beyond."""
    ell = 0.75
    ts = np.array([744.0, 745.0, 745.1, 745.14, 745.2, 746.0, 800.0, 1e5])
    z = (ts * ell / np.sqrt(d)).reshape(-1, 1)
    K = gp.ops.cov_cross(np.zeros((1, 1)), z, np.array([ell, 1e3, 1.0]), kind=KIND[d]).cpu().numpy()[0]
    assert np.all(K[3:] == 0.0) and not np.any(np.signbit(K[3:])), K
    assert K[0] > 0.0


# ----------------------------------------------------------------------------------------------- log-likelihood
def _gershgorin_cond(x, h, d):
    from oracle import sds_oracle as so
    K = mo.cov_matrix(x, h, d)
    Sii = so.s_diagonal(np.diagonal(K), h[-1])
    return (np.abs(K).sum(axis=1) + Sii).max() / Sii.min()


def _loglik_case(n, B, d, seed, ell_range=(0.5, 6.0)):
    rs = np.random.RandomState(seed)
    x = np.arange(n, dtype=np.float64).reshape(n, 1) + rs.uniform(-0.3, 0.3, size=(n, 1))
    H = np.column_stack([rs.uniform(*ell_range, B), rs.uniform(0.5, 2.0, B), rs.uniform(0.8, 2.0, B)])
    G = rs.standard_normal((B, n)) * 2.0
    return x, G, H


@pytest.mark.parametrize('d', DS)
@pytest.mark.parametrize('n,B,max_wave', [(8, 5, None), (130, 9, 4), (1000, 6, 2), (4096, 3, 2)])
def test_loglik_against_oracle(gp, d, n, B, max_wave):
    """DESIGN.md section 4: 1e-10 relative where cond(K + S) <= 1e6 (the Gershgorin bound is checked here); several waves
    where max_wave is set."""
    from oracle import sds_oracle as so
    x, G, H = _loglik_case(n, B, d, 11 * n + d, ell_range=(0.5, 6.0) if n < 4096 else (0.5, 1.5))
    ll, info = gp.ops.loglik_batched(x, G, H, kind=KIND[d], max_wave=max_wave, workspace=gp.ops.Workspace())
    ll, info = ll.cpu().numpy(), info.cpu().numpy()
    assert np.all(info == 0)
    for b in range(B):
        assert _gershgorin_cond(x, H[b], d) <= 1e6
        ref = mo.loglik_unit(x, G[b], H[b], d, form='trsv')
        assert abs(ll[b] - ref) <= 1e-10 * abs(ref), (b, ll[b], ref)
    # the host-buffer entry point is the same computation
    llh, infoh = gp.ops.loglik_host(x, G, H, kind=KIND[d])
    assert np.all(infoh == 0)
    np.testing.assert_allclose(llh, ll, rtol=1e-13)


@pytest.mark.parametrize('d', DS)
def test_loglik_jitter_ladder_with_one_failing_item(gp, d):
    """One item the ladder cannot rescue (a NaN length-scale: every rung fails, info = GPMC_INFO_NOT_PD, loglik NaN) and,
    for d = 5, one it does rescue (300 points on [0, 3], ell = 80, sn = 1e-10: K + S has eigenvalues far below rounding,
    so the first factorisation fails on the device as in LAPACK, and jitter 1e-6 mean(diag) makes it positive definite);
    the other items equal those of a call without them (to rounding: the two calls' waves differ, and so may their
    schedules)."""
    import scipy.linalg
    from oracle import sds_oracle as so
    n, B = 300, 6
    x, G, H = _loglik_case(n, B, d, 77 + d)
    H[2] = [np.nan, 1.5, 0.5]
    bad = [2]
    if d == 5:
        x = np.linspace(0, 3, n).reshape(-1, 1)
        H[:, 0] = np.minimum(H[:, 0], 0.5) * 0.05                 # keep the other items well conditioned on the dense x
        H[4] = [80.0, 1.5, 1e-10]
        K = mo.cov_matrix(x, H[4], d)
        assert scipy.linalg.lapack.dpotrf(K + np.diag(so.s_diagonal(np.diagonal(K), H[4, -1])), lower=1)[1] != 0
        bad.append(4)
    ll, info = gp.ops.loglik_batched(x, G, H, kind=KIND[d], max_wave=2, workspace=gp.ops.Workspace())
    ll, info = ll.cpu().numpy(), info.cpu().numpy()
    assert info[2] == gp._lib.INFO_NOT_PD and np.isnan(ll[2])
    if d == 5:
        assert info[4] == 0
        ref = mo.loglik_unit(x, G[4], H[4], d, form='trsv')
        assert abs(ll[4] - ref) <= 1e-6 * abs(ref), (ll[4], ref)
    keep = [b for b in range(B) if b not in bad]
    assert np.all(info[keep] == 0)
    ll2, info2 = gp.ops.loglik_batched(x, G[keep], H[keep], kind=KIND[d], workspace=gp.ops.Workspace())
    assert np.all(info2.cpu().numpy() == 0)
    np.testing.assert_allclose(ll2.cpu().numpy(), ll[keep], rtol=1e-12)


def _band_w(x, h, d):
    """w[r] of band_bound_kernel for one Matern item with 1-D x (cov_assemble.cu)."""
    N = x.shape[0]
    nblk = (N + ENV_ROWS - 1) // ENV_ROWS
    ell = np.exp(np.log(h[0]))
    u = (np.sqrt(d) * x[:, 0]) / ell if d != 1 else x[:, 0] / ell
    bl = np.array([u[r * ENV_ROWS:(r + 1) * ENV_ROWS].min() for r in range(nblk)])
    bh = np.array([u[r * ENV_ROWS:(r + 1) * ENV_ROWS].max() for r in range(nblk)])
    lo = np.arange(nblk)
    for r in range(nblk):
        for c in range(r):
            g = max(0.0, bl[r] - bh[c], bl[c] - bh[r])
            if not (np.sqrt(g * g) * (1.0 - 1e-9) > 745.14):
                lo[r] = c
                break
    w = np.array([min(lo[max(r - 1, 0)], lo[r], lo[min(r + 1, nblk - 1)]) // (NB // ENV_ROWS) * (NB // ENV_ROWS)
                  for r in range(nblk)])
    return w


def _layout(gp):
    lib = gp._lib.load()
    W, waves = ctypes.c_int(-1), ctypes.c_int(-1)
    gp._lib.check(lib.gpmc_loglik_layout(ctypes.byref(W), ctypes.byref(waves)), 'gpmc_loglik_layout')
    return W.value, waves.value


@pytest.mark.parametrize('d', DS)
@pytest.mark.parametrize('ell,compact', [(0.1, True), (25.0, False)])
def test_band_envelope_compact_bitwise_equal_to_dense(gp, d, ell, compact):
    """Short ell: the band is narrow and the call takes the compact layout in one wave where the dense layout needs several;
    long ell (band about 745 ell / sqrt(d) rows, wider than the matrix): the dense fallback.  Either way loglik and info
    equal those of the dense path (keys 14, 15 and 17 off) bit for bit, and the dense K has no nonzero left of the band's
    first tile w[r]."""
    n, B, wave = 1000, 400, 200
    rs = np.random.RandomState(5 + d)
    x = np.arange(n, dtype=np.float64).reshape(n, 1) * 0.5
    H = np.column_stack([ell * np.sqrt(d) * rs.uniform(0.8, 1.2, B), rs.uniform(0.5, 2.0, B), rs.uniform(0.5, 1.5, B)])
    G = rs.standard_normal((B, n))
    ll, info = gp.ops.loglik_batched(x, G, H, kind=KIND[d], max_wave=wave, workspace=gp.ops.Workspace())
    W, waves = _layout(gp)
    assert (W > 0) == compact, (W, waves)
    if compact:
        widest = max(int((np.arange(len(w)) - w).max()) for w in (_band_w(x, h, d) for h in H))
        assert W == (NB + ENV_ROWS * widest + 15) // 16 * 16 and waves == 1, (W, widest, waves)
    else:
        assert waves >= 2
    for h in H[:4]:
        w = _band_w(x, h, d)
        K = gp.ops.cov_assemble(x, h[None], kind=KIND[d]).cpu().numpy()[0, :, :n]
        for r in range(len(w)):
            assert not np.any(K[r * ENV_ROWS:(r + 1) * ENV_ROWS, :w[r] * ENV_ROWS])
    for key in (14, 15, 17):
        gp.ops.set_tuning(key, 0)
    try:
        ll0, info0 = gp.ops.loglik_batched(x, G, H, kind=KIND[d], max_wave=wave, workspace=gp.ops.Workspace())
    finally:
        for key in (14, 15, 17):
            gp.ops.set_tuning(key, 1)
    assert np.all(info.cpu().numpy() == 0)
    assert np.array_equal(ll.cpu().numpy(), ll0.cpu().numpy()) and np.array_equal(info.cpu().numpy(), info0.cpu().numpy())


# ----------------------------------------------------------------------------------------------------- gradient
@pytest.mark.parametrize('d', DS)
@pytest.mark.parametrize('n,D', [(40, 1), (300, 1), (200, 2)])
def test_gradient_against_oracle_band_on_off_and_repeatable(gp, d, n, D):
    rs = np.random.RandomState(n + d)
    x = _inputs(n, D, n + d, span=n * 0.4)
    B = 4
    H = np.column_stack([rs.uniform(0.6, 4.0, B), rs.uniform(0.5, 2.0, B), rs.uniform(0.7, 1.5, B)])
    G = rs.standard_normal((B, n))
    ll, gr, info = gp.ops.loglik_grad_batched(x, G, H, kind=KIND[d])
    ll, gr, info = ll.cpu().numpy(), gr.cpu().numpy(), info.cpu().numpy()
    assert np.all(info == 0)
    for b in range(B):
        rl, rg = mo.loglik_grad(x, G[b], H[b], d, form='cho')
        rl2, rg2 = mo.loglik_grad(x, G[b], H[b], d, form='inv')
        assert abs(ll[b] - rl) <= 1e-10 * abs(rl)
        spread = np.abs(rg - rg2)
        assert np.all(np.abs(gr[b] - rg) <= 1e-9 * np.maximum(1.0, np.abs(rg)) + 100 * spread), (b, gr[b], rg)
    ll2, gr2, _ = gp.ops.loglik_grad_batched(x, G, H, kind=KIND[d])
    assert np.array_equal(gr2.cpu().numpy(), gr) and np.array_equal(ll2.cpu().numpy(), ll)
    gp.ops.set_tuning(15, 0)
    try:
        ll3, gr3, _ = gp.ops.loglik_grad_batched(x, G, H, kind=KIND[d])
    finally:
        gp.ops.set_tuning(15, 1)
    assert np.array_equal(gr3.cpu().numpy(), gr) and np.array_equal(ll3.cpu().numpy(), ll)


# ------------------------------------------------------------------------------------------------ GPR and predict
@pytest.mark.parametrize('d', DS)
def test_gpr_optimize_and_predict(gp, d):
    """Data drawn from a Matern GP: GPR.optimize lands where scipy lands on the oracle's nlZ from the same start, and
    GPR.predict matches the oracle's predictive mean / variance at the optimum."""
    import scipy.optimize
    from oracle import sds_oracle as so
    n = 120
    rs = np.random.RandomState(40 + d)
    x = np.sort(rs.uniform(0, 40, size=(n, 1)), axis=0)
    Kt = mo.cov_matrix(x, np.array([3.0, 1.5, 1.0]), d)
    y = np.linalg.cholesky(Kt + 1e-10 * np.eye(n)) @ rs.standard_normal(n) + 0.3 * rs.standard_normal(n)
    m = gp.kcGP.gpK.GPR()
    m.setData(x, y)
    m.setPrior(kernel=gp.kcGP.covK.Matern(np.log(1.0), d, np.log(1.0)))
    m.setNoise(log_sigma=np.log(0.5))
    h0 = m._log_hyp()
    m.optimize(numIterations=200)

    def nlz(lh):
        th = np.exp(lh)
        ll, g = mo.loglik_grad(x, y, th, d)
        return -ll, -th * g

    ref = scipy.optimize.minimize(nlz, h0, jac=True, method='L-BFGS-B', options={'maxiter': 200})
    got = m._log_hyp()
    assert abs(m.nlZ - ref.fun) <= 1e-6 * abs(ref.fun), (m.nlZ, ref.fun)
    np.testing.assert_allclose(got, ref.x, atol=1e-3)
    xs = np.linspace(-2, 42, 25).reshape(-1, 1)
    ym, ys2, fm, fs2, lp = m.predict(xs)
    th = np.exp(got)
    _, _, _, Fs2, Fmu = mo.inf_mcmc_unit(y, x, y, xs, th, d)
    np.testing.assert_allclose(fm[:, 0], Fmu[:, 0], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(fs2[:, 0], Fs2[:, 0], rtol=1e-8, atol=1e-10)


@pytest.mark.parametrize('d', DS)
@pytest.mark.parametrize('n,ns,S', [(130, 3, 2), (640, 70, 4)])
def test_predict_batched_against_oracle(gp, d, n, ns, S):
    from oracle import sds_oracle as so
    rs = np.random.RandomState(n + ns + d)
    x, y = gp.synthetic.ih45_series(n)
    xs = np.sort(rs.uniform(0, n, size=(ns, 1)), axis=0)
    Hyp = np.column_stack([rs.uniform(1.5, 7., S), rs.uniform(2., 9., S), rs.uniform(0.6, 2.8, S)])
    F = (y - y.mean())[:, None] * 0.7 + 0.3 * rs.standard_normal((n, S))
    fmu, fs2, info = gp.ops.predict_batched(x, xs, np.ascontiguousarray(F.T), Hyp, kind=KIND[d])
    assert np.all(info.cpu().numpy() == 0)
    fmu, fs2 = fmu.cpu().numpy(), fs2.cpu().numpy()
    for s in range(S):
        _, _, _, Fs2, Fmu = mo.inf_mcmc_unit(F[:, s], x, y, xs, Hyp[s], d)
        np.testing.assert_allclose(fmu[s], Fmu[:, 0], rtol=1e-9, atol=1e-9)
        np.testing.assert_allclose(np.maximum(fs2[s], 0), Fs2[:, 0], rtol=1e-8, atol=1e-10)


@pytest.mark.parametrize('d', DS)
def test_ess_sweep_against_oracle_on_tapes(gp, d):
    """nu on the tape: f' = f cos(theta) + nu sin(theta) to rounding; nu = chol(K) z on the device with the Matern K (a
    short length-scale keeps K well conditioned, so the first factorisation decides the same way as LAPACK's)."""
    import torch
    from gpmc_b200 import ops
    from oracle import sds_oracle as so
    from oracle.reference_loader import EssTape
    n, B = 150, 4
    x, y = gp.synthetic.ih45_series(n)
    rs = np.random.RandomState(90 + d)
    F0 = (y - y.mean())[None, :] * 0.5 + 0.3 * rs.standard_normal((B, n))
    H = np.column_stack([rs.uniform(0.8, 1.5, B), rs.uniform(2.0, 6.0, B), rs.uniform(1.0, 3.0, B)])
    Z, U, TH = rs.standard_normal((B, n)), rs.random_sample(B), rs.random_sample((B, 64))
    for mode in ('nu', 'z'):
        nus = np.stack([mo.ess_nu_from_z(x, H[c], Z[c], d) for c in range(B)])
        F = torch.tensor(F0.copy()).cuda()
        tape = ops.EssTape(U, TH, nu=nus if mode == 'nu' else None, z=Z if mode == 'z' else None)
        nt, st, info = ops.ess_sweep(x, y, F, H, tape=tape, max_trips=64, kind=KIND[d])
        assert np.all(st.cpu().numpy() == 0) and np.all(info.cpu().numpy() == 0)
        for c in range(B):
            of, ntr = so.elliptical_slice(F0[c], x, y, H[c], EssTape(nus[c], U[c], TH[c]))
            assert int(nt[c].item()) == ntr
            tol = 1e-12 if mode == 'nu' else 1e-9
            assert np.abs(F.cpu().numpy()[c] - of).max() <= tol * max(1.0, np.abs(of).max())


# --------------------------------------------------------------------------------------------------- SDS sampler
@pytest.mark.parametrize('d', DS)
def test_sds_sweep_against_tape_oracle(gp, d):
    """theta' (1e-12) and trip counts exact; f' within a multiple of the oracle's own resolution (literal vs reduced R,
    DESIGN.md section 4), capped at 5e-2."""
    import torch
    from gpmc_b200 import ops
    from oracle import sds_oracle as so
    from oracle.reference_loader import Tape
    n, B = 96, 4
    x, y = gp.synthetic.ih45_series(n)
    F0, H0 = gp.synthetic.chain_states(B, n)
    scale = np.array(gp.synthetic.SCALE)
    for it in (0, 700):
        rs = np.random.RandomState(31 + it + d)
        z, v, u0, U = rs.standard_normal((B, n)), rs.random_sample((B, 3)), rs.random_sample(B), rs.random_sample((B, 48, 3))
        F = torch.tensor(F0.copy()).cuda()
        H = torch.tensor(H0.copy()).cuda()
        nt, ll, st = ops.sds_sweep(x, y, F, H, scale, it, tape=ops.Tape(z, v, u0, U), max_trips=48, kind=KIND[d])
        assert np.all(st.cpu().numpy() == 0)
        for c in range(B):
            tr = so.SweepTrace()
            tape = Tape(z[c], v[c], u0[c], U[c])
            of, oh = mo.surrogate_slice_sampling(F0[c], x, y, H0[c], scale, it, tape, d, trace=tr, r_form='reduced')
            ofl, _ = mo.surrogate_slice_sampling(F0[c], x, y, H0[c], scale, it, tape, d, r_form='literal')
            assert int(nt[c].item()) == tr.n_trips
            np.testing.assert_allclose(H.cpu().numpy()[c], oh, rtol=RTOL_HYP)
            tol = min(F_ABS_CAP, max(1e-9, F_RES_FACTOR * float(np.abs(of - ofl).max())))
            assert np.abs(F.cpu().numpy()[c] - of).max() <= tol
            assert abs(float(ll[c].item()) - tr.propG_chol[-1]) <= 1e-9 * abs(tr.propG_chol[-1])


@pytest.mark.parametrize('d', DS)
def test_sds_run_equals_sweeps_and_chain_ensemble_runs(gp, d):
    import torch
    from gpmc_b200 import ops
    n, B, iters, it0 = 100, 7, 4, 498
    x, y = gp.synthetic.ih45_series(n)
    scale = np.array(gp.synthetic.SCALE)
    F0, H0 = gp.synthetic.chain_states(B, n)
    F = torch.tensor(F0.copy()).cuda(); H = torch.tensor(H0.copy()).cuda()
    ref_h, ref_f = [], []
    for k in range(iters):
        nt, ll, st = ops.sds_sweep(x, y, F, H, scale, it0 + k, seed=9, chain0=2, max_trips=48, kind=KIND[d])
        assert int((st != 0).sum().item()) == 0
        ref_h.append(H.cpu().numpy().copy()); ref_f.append(F.cpu().numpy().copy())
    F2 = torch.tensor(F0.copy()).cuda(); H2 = torch.tensor(H0.copy()).cuda()
    hh, hl, ht, hf, n_exh = ops.sds_run(x, y, F2, H2, scale, it0, iters, seed=9, chain0=2, max_trips=48, kind=KIND[d],
                                        workspace=ops.Workspace())
    assert n_exh == 0
    assert np.array_equal(F2.cpu().numpy(), ref_f[-1]) and np.array_equal(H2.cpu().numpy(), ref_h[-1])
    for k in range(iters):
        assert np.array_equal(hh.cpu().numpy()[:, k, :], ref_h[k])
    # the ensemble passes its kind through: its sweep is ops.sds_sweep with that kind.  theta' alone can coincide with the
    # SE sweep's (a first proposal that is accepted does not depend on the kernel), log N(g; 0, K+S) does not.
    F3 = torch.tensor(F0.copy()).cuda(); H3 = torch.tensor(H0.copy()).cuda()
    _, ll3, _ = ops.sds_sweep(x, y, F3, H3, scale, it0, seed=9, chain0=0, max_trips=48, kind=KIND[d])
    outs = []
    for kind in (KIND[d], None):
        ens = gp.chains.ChainEnsemble(x, y, F0, H0, scale, seed=9, max_trips=48, distributed=False, kind=kind)
        hyp, llk, ntr = ens.sweep(it0)
        assert hyp.shape == (B, 3) and np.all(np.isfinite(llk))
        outs.append((hyp, llk))
    assert np.array_equal(outs[0][0], H3.cpu().numpy()) and np.array_equal(outs[0][1], ll3.cpu().numpy())
    assert not np.array_equal(outs[0][1], outs[1][1])


# ---------------------------------------------------------------------------------------------- kind validation
def test_unknown_kinds_and_matern_with_wrong_P_are_rejected(gp):
    """Every entry point that takes a kind returns GPMC_EINVAL (-22) for a value outside 0..4, and for a Matern kind with
    P != 3; kinds 0 and 1 keep their meaning."""
    import torch
    lib = gp._lib.load()
    n, D = 64, 2
    x = torch.tensor(_inputs(n, D, 1)).cuda()
    g = torch.zeros((1, n), dtype=torch.float64, device='cuda')
    F = torch.zeros((1, n), dtype=torch.float64, device='cuda')
    y = torch.zeros(n, dtype=torch.float64, device='cuda')
    out = torch.zeros((1, n, n + 16), dtype=torch.float64, device='cuda')
    ws = torch.zeros(1 << 26, dtype=torch.uint8, device='cuda')
    ll = torch.zeros(4, dtype=torch.float64, device='cuda')
    gr = torch.zeros(16, dtype=torch.float64, device='cuda')
    info = torch.zeros(4, dtype=torch.int32, device='cuda')
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: t.data_ptr()
    bad = [(k, 3) for k in (-1, 5, 99)] + [(k, D + 2) for k in (2, 3, 4)] + [(k, 5) for k in (2, 3, 4)]
    for kind, P in bad:
        hyp = torch.ones((1, P), dtype=torch.float64, device='cuda')
        scale = torch.ones(P, dtype=torch.float64, device='cuda')
        calls = {
            'cov_assemble': lambda: lib.gpmc_cov_assemble(p(x), n, D, p(hyp), 1, P, kind, 0, None, p(out), n + 16, st),
            'cov_cross': lambda: lib.gpmc_cov_cross(p(x), n, p(x), n, D, p(hyp), P, kind, p(out), n + 16, st),
            'loglik_batched': lambda: lib.gpmc_loglik_batched(p(x), n, D, p(g), p(hyp), 1, P, kind, 1, p(ll), p(info),
                                                              p(ws), ws.numel(), st),
            'loglik_grad_batched': lambda: lib.gpmc_loglik_grad_batched(p(x), n, D, p(g), p(hyp), 1, P, kind, 1, p(ll), p(gr),
                                                                        p(info), p(ws), ws.numel(), st),
            'predict_batched': lambda: lib.gpmc_predict_batched(p(x), n, D, p(x), 4, p(g), p(hyp), 1, P, kind, 1, p(ll), p(gr),
                                                                p(info), p(ws), ws.numel(), st),
            'sds_sweep': lambda: lib.gpmc_sds_sweep(p(x), p(y), n, D, p(F), p(hyp), 1, P, kind, p(scale), p(scale), p(scale),
                                                    0, 0.0, 0.0, 100.0, 0, 0, None, None, None, None, 0, 8, 1, None, None,
                                                    None, p(ws), ws.numel(), st),
            'sds_run': lambda: lib.gpmc_sds_run(p(x), p(y), n, D, p(F), p(hyp), 1, P, kind, p(scale), p(scale), p(scale), 0, 1,
                                                0.0, 0.0, 100.0, 0, 0, 8, 1, None, None, None, None, 1, 1, None, p(ws),
                                                ws.numel(), st),
            'ess_sweep': lambda: lib.gpmc_ess_sweep(p(x), p(y), n, D, p(F), p(hyp), 1, P, kind, 0.0, 0.0, 100.0, 0, 0, 0,
                                                    None, None, None, None, 0, 8, 1, None, None, p(info), p(ws), ws.numel(), st),
        }
        for name, call in calls.items():
            assert call() == -22, (name, kind, P)
        hh = np.ones((1, P))
        xh = np.ascontiguousarray(x.cpu().numpy())
        assert lib.gpmc_loglik_host(xh.ctypes.data, n, D, np.zeros((1, n)).ctypes.data, hh.ctypes.data, 1, P, kind, 1,
                                    np.zeros(1).ctypes.data, np.zeros(1, dtype=np.int32).ctypes.data) == -22
        with pytest.raises(gp._lib.GpmcError):
            gp.ops.loglik_batched(x, g, hyp, kind=kind, workspace=gp.ops.Workspace())
    torch.cuda.synchronize()
    # SE kinds are unchanged: kind 0 with P = 3, kind 1 with P = D + 2, and kind=None infers them
    h3 = np.array([[2.0, 1.0, 0.5]])
    a = gp.ops.cov_assemble(x, h3, kind=0).cpu().numpy()
    assert np.array_equal(a, gp.ops.cov_assemble(x, h3).cpu().numpy())
    h4 = np.array([[2.0, 3.0, 1.0, 0.5]])
    assert np.array_equal(gp.ops.cov_assemble(x, h4, kind=1).cpu().numpy(), gp.ops.cov_assemble(x, h4).cpu().numpy())
