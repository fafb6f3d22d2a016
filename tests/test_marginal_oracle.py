"""CPU checks of the marginal slice sampler's oracle (oracle/marginal_oracle.py): the quadrature reference of the
hyper-parameter posterior, invariance of that posterior under the restated transition, and the multi-rank plumbing of
ChainEnsemble(likelihood='gauss')."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import scipy.integrate

from oracle import marginal_oracle as mo
from oracle import sds_oracle as so

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def data(n, seed=5):
    rng = np.random.default_rng(seed)
    x = np.linspace(0, 60, n).reshape(-1, 1)
    return x, 15 * np.sin(x[:, 0] / 8) + 6 * rng.standard_normal(n) + 50


# The bracket rule hyp_min = max(hyp - v, 0) (sliceSample.py:111) is not reversible where it clips at 0: the bracket
# [0, scale] is drawn from theta with probability 1 - theta / scale, which differs between the points it holds.  The
# sampler is exact where the posterior keeps theta above scale, so these checks use priors that hold it there
# (Gamma(20, 1) on ell and sf, inverse-Gamma(20, 120) on sn; the chains never come below scale).
PRIOR = (np.array([20., 20., 20.]), np.array([1., 1., 120.]))
SCALE = np.array([3.0, 3.0, 2.0])
BOUNDS16 = ((1.5, 4.), (1.8, 4.), (0.8, 2.8))


def test_posterior_grid_1d_matches_scipy_quad():
    x, y = data(16)
    r = y - y.mean()
    pk, pth = PRIOR
    lsf, lsn = np.log(19.), np.log(6.5)
    res = mo.posterior_grid(x, y, prior=PRIOR, bounds=((1.5, 4.), (lsf, lsf), (lsn, lsn)), n=(201, 1, 1))
    ref_max = max(mo.log_posterior(x, r, np.exp([l, lsf, lsn]), pk, pth) + l for l in np.linspace(1.5, 4, 41))

    def dens(l):
        return np.exp(mo.log_posterior(x, r, np.exp([l, lsf, lsn]), pk, pth) + l - ref_max)
    Z = scipy.integrate.quad(dens, 1.5, 4., epsabs=0, epsrel=1e-12, limit=200)[0]
    mean = scipy.integrate.quad(lambda l: l * dens(l), 1.5, 4., epsabs=0, epsrel=1e-12, limit=200)[0] / Z
    var = scipy.integrate.quad(lambda l: (l - mean) ** 2 * dens(l), 1.5, 4., epsabs=0, epsrel=1e-12, limit=200)[0] / Z
    assert res['edge'] < 1e-6
    assert abs(res['mean'][0] - mean) < 1e-7 and abs(res['var'][0] - var) < 1e-7, (res, mean, var)
    assert abs(res['mean'][1] - lsf) < 1e-12 and abs(res['var'][1]) < 1e-12


def test_transition_leaves_the_posterior_invariant():
    """A long seeded oracle chain (N = 16, every prior from the start) has the moments of posterior_grid."""
    x, y = data(16)
    grid = mo.posterior_grid(x, y, prior=PRIOR, bounds=BOUNDS16, n=(33, 33, 33))
    assert grid['edge'] < 1e-4
    rng = np.random.default_rng(11)
    n_iters, P, T = 12000, 3, 64
    hh, ll, tt, exh = mo.run_chain(x, y, [20., 20., 6.], SCALE, 0, n_iters, 0, rng.uniform(size=(n_iters, P)),
                                   rng.uniform(size=n_iters), rng.uniform(size=(n_iters, T, P)), prior_k=PRIOR[0],
                                   prior_theta=PRIOR[1])
    assert exh == 0 and tt.min() >= 1 and np.all(hh.min(axis=0) > SCALE)
    logs = np.log(hh[200:])
    for d in range(3):
        se = mo.batch_means_se(logs[:, d], n_batches=40)
        assert abs(logs[:, d].mean() - grid['mean'][d]) < 4 * se, (d, logs[:, d].mean(), grid['mean'][d], se)


def test_run_chain_keeps_a_state_that_cannot_start():
    x, y = data(8)
    rng = np.random.default_rng(0)
    hh, ll, tt, exh = mo.run_chain(x, y, [np.nan, 1.0, 0.5], [1., 1., 1.], 0, 3, 0, rng.uniform(size=(3, 3)),
                                   rng.uniform(size=3), rng.uniform(size=(3, 4, 3)))
    assert exh == -1 and np.all(tt == 0) and np.all(np.isnan(ll))


def test_burn_in_freezes_the_noise():
    x, y = data(8)
    rng = np.random.default_rng(1)
    hh, _, _, _ = mo.run_chain(x, y, [0.8, 1.5, 0.5], [2., 3., 2.], 495, 10, 500, rng.uniform(size=(10, 3)),
                               rng.uniform(size=10), rng.uniform(size=(10, 64, 3)))
    assert np.all(hh[:5, 2] == 0.5) and np.any(hh[5:, 2] != 0.5)


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_two_rank_gloo_gauss_ensemble_matches_single_process():
    env = dict(os.environ, OMP_NUM_THREADS='2', OPENBLAS_NUM_THREADS='2')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
           '--master-addr', '127.0.0.1', '--master-port', str(_free_port()),
           os.path.join(ROOT, 'tests', '_gloo_marginal_worker.py')]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-4000:]
    assert 'GLOO_MARGINAL_OK' in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


def test_ensemble_rejects_an_unknown_likelihood(gp):
    with pytest.raises(ValueError):
        gp.chains.ChainEnsemble(np.zeros((4, 1)), np.zeros(4), None, np.ones((2, 3)), np.ones(3), likelihood='probit')
