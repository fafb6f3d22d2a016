"""The oracle restatement against the committed golden vectors (outputs of the reference's own
``kcMCMC/sliceSample.py``, see ``oracle/make_golden.py``).  Runs anywhere, CPU only."""
import os

import numpy as np
import pytest

from conftest import golden_files, load_rows, GOLDEN
from oracle import sds_oracle as so
from oracle.make_golden import pinned_blas
from oracle.reference_loader import Tape

SDS = golden_files('sds_N*.npz')


def test_fixtures_present():
    assert len(SDS) >= 9
    for name in ('loglik_iso.npz', 'loglik_ard.npz', 'chain_N64.npz'):
        assert os.path.isfile(os.path.join(GOLDEN, name))


@pytest.mark.parametrize('path', SDS, ids=[os.path.basename(p) for p in SDS])
def test_transition_matches_reference_output(path):
    z = np.load(path)
    tape = Tape(z['z'], z['v'], z['u0'], z['U'])
    tr = so.SweepTrace()
    # the BLAS summation order of the fixture's run (OpenBLAS sets it by its thread count, whatever the host's cores)
    with pinned_blas():
        pf, ph = so.surrogate_slice_sampling(z['f'], z['x'], z['y'], z['hyp'], z['scale'], int(z['it']), tape, trace=tr)
    # same BLAS order: the restatement reproduced the literal run bit for bit when the
    # fixture was made; across CPU types allow BLAS-level rounding.
    assert tr.n_trips == int(z['ref_trips'])
    np.testing.assert_allclose(ph, z['ref_prop_hyp'], rtol=1e-13, atol=0)
    np.testing.assert_allclose(pf, z['ref_prop_f'], rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(tr.curG, z['ref_curG'], rtol=1e-11)
    np.testing.assert_allclose(tr.g, z['ref_g'], rtol=1e-13, atol=1e-13)


@pytest.mark.parametrize('path', SDS, ids=[os.path.basename(p) for p in SDS])
def test_aux_var_model_and_priors(path):
    z = np.load(path)
    K = so.cov_matrix(z['x'], z['hyp'])
    g, K_S, m, C, L = so.aux_var_model(z['f'], K, z['hyp'][2], z=z['z'])
    np.testing.assert_allclose(g, z['ref_g'], rtol=1e-13, atol=1e-13)
    np.testing.assert_allclose(np.diag(L), z['ref_diagL'], rtol=1e-12)
    np.testing.assert_allclose(m, z['ref_m'], rtol=1e-6, atol=1e-7)
    prior, grad = so.log_gamma(z['hyp'], so.PRIOR_K3, so.PRIOR_THETA3, True)
    np.testing.assert_allclose(prior, z['ref_prior'], rtol=1e-14)
    np.testing.assert_allclose(grad, z['ref_prior_grad'], rtol=1e-14)
    if 'ref_K' in z.files:
        np.testing.assert_allclose(K, z['ref_K'], rtol=1e-15, atol=0)
        np.testing.assert_allclose(L, z['ref_L'], rtol=1e-11, atol=1e-13)


def test_loglik_unit_known_answers():
    rows = load_rows(os.path.join(GOLDEN, 'loglik_iso.npz'))
    assert len(rows) >= 30
    worst = 0.0
    for r in rows:
        x = r['x'].reshape(-1, 1)
        for form, key in (('inv', 'll_inv'), ('chol', 'll_chol')):
            got = so.loglik_unit(x, r['g'], r['hyp'], form=form)
            assert abs(got - float(r[key])) <= 1e-11 * abs(float(r[key])) * max(1.0, float(r['cond']) / 1e6)
        # the reference's inv form and its own Cholesky form agree to 1e-10 while cond <= ~1e7
        gap = abs(float(r['ll_inv']) - float(r['ll_chol'])) / abs(float(r['ll_chol']))
        if float(r['cond']) < 1e7:
            assert gap < 1e-10
        worst = max(worst, gap)
        trsv = so.loglik_unit(x, r['g'], r['hyp'], form='trsv')
        assert abs(trsv - float(r['ll_chol'])) <= 1e-11 * abs(float(r['ll_chol'])) * max(1.0, float(r['cond']) / 1e6)
    assert worst < 1e-8


def test_loglik_unit_ard_known_answers():
    for r in load_rows(os.path.join(GOLDEN, 'loglik_ard.npz')):
        got = so.loglik_unit(r['x'], r['g'], r['hyp'], form='chol')
        assert abs(got - float(r['ll_chol'])) <= 1e-12 * abs(float(r['ll_chol']))


def test_chain_matches_reference_history():
    z = np.load(os.path.join(GOLDEN, 'chain_N64.npz'))
    F, H, T = so.run_chain(z['x'], z['y'], z['hyp0'], z['scale'], int(z['iters']), int(z['seed']), start_iter=int(z['start_iter']))
    assert np.array_equal(T, z['ref_trips'])
    np.testing.assert_allclose(H, z['ref_histHyp'], rtol=1e-12)
    # noise is frozen before iteration 500 (sliceSample.py:133-134) and moves afterwards
    burn = int(500 - z['start_iter'])
    assert np.all(H[2, :burn] == z['hyp0'][2]) and np.any(H[2, burn:] != z['hyp0'][2])


def test_s_diagonal_is_not_simplified():
    # sliceSample.py:184-187: S_ii differs from sn^2 in the last digits at extreme ratios (SURVEY fact 6)
    s = so.s_diagonal(np.array([1e-4]), 5.0)
    assert s[0] != 25.0 and abs(s[0] - 25.0) / 25.0 < 1e-9
    assert so.s_diagonal(np.array([100.0]), 1.2)[0] == pytest.approx(1.44, rel=1e-14)


def test_bracket_clamp_and_shrink_rules():
    # sliceSample.py:110-112: clamp at 0 BEFORE adding scale -> width is always `scale`
    hyp = np.array([1., 10., 1.2]); scale = np.array([10., 10., 5.])
    v = scale * np.array([0.9, 0.1, 0.99])
    lo = np.maximum(hyp - v, 0); hi = lo + scale
    assert lo[0] == 0 and hi[0] == 10 and lo[2] == 0 and hi[2] == 5
    assert np.all(lo <= hyp) and np.all(hyp <= hi)


ESS = golden_files('ess_N*.npz')


@pytest.mark.parametrize('path', ESS, ids=[os.path.basename(p) for p in ESS])
def test_elliptical_slice_matches_reference_output(path):
    """oracle.elliptical_slice against the outputs of the reference's own elliptical_slice (sliceSample.py:15-74) run on
    a tape; the stored nu is the Cholesky draw jitchol(K) z, which the oracle reproduces from z."""
    from oracle.reference_loader import EssTape
    z = np.load(path)
    assert len(ESS) >= 4
    pf, trips = so.elliptical_slice(z['f'], z['x'], z['y'], z['hyp'], EssTape(z['nu'], float(z['u']), z['theta']))
    assert trips == int(z['ref_trips'])
    np.testing.assert_allclose(pf, z['ref_prop_f'], rtol=1e-13, atol=1e-13)
    np.testing.assert_allclose(so.ess_nu_from_z(z['x'], z['hyp'], z['z']), z['nu'], rtol=1e-9, atol=1e-9)


def test_inf_mcmc_restatement_matches_reference_outputs():
    """oracle.inf_mcmc_unit against the reference's own inf_mcmc (sliceSample.py:234-284), one call per stored sample."""
    z = np.load(os.path.join(GOLDEN, 'infmcmc_batched_N96.npz'))
    for s in range(z['Hyp'].shape[0]):
        ym, lw, up, Fs2, _ = so.inf_mcmc_unit(z['F'][:, s], z['x'], z['y'], z['xs'], z['Hyp'][s])
        np.testing.assert_allclose(ym, z['ref_ym'][s], rtol=1e-10)
        np.testing.assert_allclose(lw, z['ref_lw'][s], rtol=1e-9)
        np.testing.assert_allclose(up, z['ref_up'][s], rtol=1e-9)
        np.testing.assert_allclose(Fs2, z['ref_Fs2'][s], rtol=1e-8, atol=1e-12)
