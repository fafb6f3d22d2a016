"""Pin the restatement to the reference file itself.  Each case's inputs, tape and outputs are stored in
``tests/golden/literal_cases.npz`` (``oracle/make_golden.py``), and the restatement must reproduce them bit for bit
(N <= 120: OpenBLAS does not split these products, so its thread count does not enter).  Where ``GPMC_REFERENCE_ROOT``
names a checkout of the original project, its own ``sliceSample.py`` runs on the same tapes as well and must return the
same bits."""
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import reference_loader as rl, sds_oracle as so, make_golden as mg

CASES = np.load(os.path.join(GOLDEN, 'literal_cases.npz'))


def _case(prefix):
    return {k[len(prefix):]: CASES[k] for k in CASES.files if k.startswith(prefix)}


@pytest.mark.parametrize('n,it,seed', mg.LITERAL_SDS_CASES)
def test_restatement_is_bit_identical_to_literal(n, it, seed):
    c = _case('sds_N%d_it%d_s%d_' % (n, it, seed))
    tape = rl.Tape(c['z'], c['v'], c['u0'], c['U'])
    tr = so.SweepTrace()
    of, oh = so.surrogate_slice_sampling(c['f'], c['x'], c['y'], c['hyp'], c['scale'], it, tape, trace=tr)
    assert tr.n_trips == int(c['trips']) and np.array_equal(oh, c['prop_hyp']) and np.array_equal(of, c['prop_f'])
    if rl.available():
        pf, ph, trips = rl.run_literal_with_tape(c['f'], c['x'], c['y'], c['hyp'], c['scale'], it, tape)
        assert trips == tr.n_trips and np.array_equal(ph, oh) and np.array_equal(pf, of)


def test_literal_module_functions():
    hyp = CASES['log_gamma_hyp']
    c, d = so.log_gamma(hyp, so.PRIOR_K3, so.PRIOR_THETA3, True)
    assert np.array_equal(c, CASES['log_gamma']) and np.array_equal(d, CASES['log_gamma_grad'])
    if rl.available():
        a, b = rl.load_literal().log_gamma(hyp, so.PRIOR_K3, so.PRIOR_THETA3, True)
        assert np.array_equal(a, c) and np.array_equal(b, d)


def test_multivariate_normal_draw_is_f_plus_sd_z():
    # sliceSample.py:194 goes through an SVD of the diagonal S; with this numpy it is f + sqrt(S_ii) z
    n = 50
    f = np.linspace(-1, 1, n)
    np.random.seed(7)
    g = np.random.multivariate_normal(f, np.diag(np.full(n, 1.44)), 1).reshape(n)
    np.random.seed(7)
    z = np.random.standard_normal(n)
    np.testing.assert_allclose(g, f + 1.2 * z, rtol=0, atol=1e-15)


@pytest.mark.parametrize('n,seed', mg.LITERAL_ESS_CASES)
def test_elliptical_slice_restatement_is_bit_identical_to_literal(n, seed):
    c = _case('ess_N%d_s%d_' % (n, seed))
    tape = rl.EssTape(c['nu'], c['u'], c['theta'])
    of, otrips = so.elliptical_slice(c['f'], c['x'], c['y'], c['hyp'], tape)
    assert otrips == int(c['trips']) and np.array_equal(of, c['prop_f'])
    if rl.available():
        pf, trips = rl.run_literal_ess_with_tape(c['f'], c['x'], c['y'], c['hyp'], tape)
        assert trips == otrips and np.array_equal(pf, of)
