"""Oracle of the library's Matern covariance kinds (GPMC_KIND_MATERN1/3/5, include/gpmc.h).

TEST INFRASTRUCTURE (see ``oracle/__init__.py``).  PARITY UNPINNED at this boundary, as for the rest of the ``kcGP``
shim: the kernel is pyGPs 1.3.4 ``cov.Matern(log_ell, d, log_sigma)`` (``pyGPs/Core/cov.py class Matern``; d = 2 nu in
{1, 3, 5}, isotropic), which the reference never calls and which is absent from this image, so the expression below is a
restatement that has not been checked against pyGPs itself.  It is written down once, in ``Matern``; the device is held to
it.  With ``ell = exp(hyp[0])``, ``sf2 = exp(2*hyp[1])``:

    u = sqrt(d) * x / ell,   t = sqrt(sqdist(u_x, u_z)),   K = sf2 * (f_d(t) * exp(-t)),
    f_1 = 1,   f_3 = 1 + t,   f_5 = 1 + t * (1 + t / 3)          (in that operation order)

The restatements of ``sds_oracle`` (SDS transition, ``inf_mcmc``, the ESS draw, the log-lik unit) and ``grad_oracle``
build their isotropic kernel as ``kcgp_shim.RBF(np.log(ell), np.log(sf))``.  ``kernel(d)`` runs them with that name bound
to the Matern kernel instead, so the Matern forms below are those restatements line for line, not copies of them.
"""
import contextlib

import numpy as np
import scipy.linalg
from scipy.spatial.distance import cdist

from . import grad_oracle as go
from . import kcgp_shim
from . import sds_oracle as so

LOG_2PI = np.log(2 * np.pi)


class Matern(object):
    """Matern kernel, isotropic, d = 2 nu in {1, 3, 5} (pyGPs 1.3.4 ``cov.Matern``, restated).  ``hyp = [log_ell,
    log_sigma]``; ``getCovMatrix(x=, z=, mode='train'|'cross'|'self_test')`` as ``kcgp_shim.RBF``."""

    def __init__(self, log_ell=0., d=3, log_sigma=0.):
        if d not in (1, 3, 5):
            raise ValueError('Matern: d must be 1, 3 or 5')
        self.d = d
        self.hyp = [log_ell, log_sigma]

    def f(self, t):
        if self.d == 1:
            return np.ones_like(t)
        if self.d == 3:
            return 1 + t
        return 1 + t * (1 + t / 3)

    def getCovMatrix(self, x=None, z=None, mode=None):
        ell = np.exp(self.hyp[0])
        sf2 = np.exp(2. * self.hyp[1])
        d = self.d

        def scaled(a):
            a = np.asarray(a, dtype=np.float64)
            return (np.sqrt(d) * (a.reshape(-1, 1) if a.ndim == 1 else a)) / ell

        if mode == 'self_test':
            A = np.zeros((z.shape[0], 1))
        elif mode == 'train':
            xs = scaled(x)
            A = np.sqrt(cdist(xs, xs, 'sqeuclidean'))
        elif mode == 'cross':
            A = np.sqrt(cdist(scaled(x), scaled(z), 'sqeuclidean'))
        else:
            raise ValueError("mode must be 'train', 'cross' or 'self_test'")
        return sf2 * (self.f(A) * np.exp(-A))


@contextlib.contextmanager
def kernel(d):
    """Inside the block, ``kcgp_shim.RBF(log_ell, log_sigma)`` -- the isotropic kernel of every ``sds_oracle`` /
    ``grad_oracle`` restatement -- is ``Matern(log_ell, d, log_sigma)``.  Not reentrant across threads."""
    if d not in (1, 3, 5):
        raise ValueError('Matern: d must be 1, 3 or 5')
    rbf = kcgp_shim.RBF
    kcgp_shim.RBF = lambda log_ell=0., log_sigma=0.: Matern(log_ell, d, log_sigma)
    try:
        yield
    finally:
        kcgp_shim.RBF = rbf


def _iso(hyp):
    hyp = np.asarray(hyp, dtype=np.float64)
    if hyp.shape[0] != 3:
        raise ValueError('the Matern kinds are isotropic: hyp = (ell, sf, sn)')
    return hyp


def cov_matrix(x, hyp, d):
    """``sds_oracle.cov_matrix`` with the Matern kernel: ``Matern(np.log(ell), d, np.log(sf)).getCovMatrix(x, 'train')``."""
    with kernel(d):
        return so.cov_matrix(x, _iso(hyp))


def loglik_unit(x, g, hyp, d, form='chol'):
    with kernel(d):
        return so.loglik_unit(x, g, _iso(hyp), form=form)


def surrogate_slice_sampling(f, x, y, hyp, scale, it, tape, d, **kw):
    with kernel(d):
        return so.surrogate_slice_sampling(f, x, y, _iso(hyp), scale, it, tape, **kw)


def ess_nu_from_z(x, hyp, z, d):
    with kernel(d):
        return so.ess_nu_from_z(x, _iso(hyp), z)


def inf_mcmc_unit(f, x, y, xs, hyp, d, **kw):
    with kernel(d):
        return so.inf_mcmc_unit(f, x, y, xs, _iso(hyp), **kw)


# ---------------------------------------------------------------------------------------------------------- gradient
def matern_g(t, d):
    """g_d(t) of dK/d ell = sf2 g_d(t) exp(-t) / ell  (g_d = t (f_d - f_d'): g_1 = t, g_3 = t^2, g_5 = t^2 (1 + t) / 3)."""
    if d == 1:
        return t
    if d == 3:
        return t * t
    return t * t * (1 + t) / 3


def contract(x, K, hyp, alpha, W, d, dtype=np.float64):
    """``grad_oracle.contract`` for the Matern kernel: dA/d ell = sf2 g_d(t) exp(-t) / ell, dA/d sf = 2 K / sf,
    dA/d sn = 2 sn I.  Returns (grad[3], mag[3]) in ``dtype``."""
    h = _iso(hyp).astype(dtype)
    x = np.asarray(x).astype(dtype)
    K = np.asarray(K).astype(dtype)
    a = np.asarray(alpha).astype(dtype)
    C = np.outer(a, a) - np.asarray(W).astype(dtype)
    u = np.sqrt(dtype(d)) * x / h[0]
    s = np.zeros_like(K)
    for c in range(x.shape[1]):
        s += (u[:, c][:, None] - u[:, c][None, :]) ** 2
    t = np.sqrt(s)
    grad, mag = np.zeros(3, dtype=dtype), np.zeros(3, dtype=dtype)
    for p, M in enumerate((h[1] ** 2 * matern_g(t, d) * np.exp(-t) / h[0], 2 * K / h[1])):
        grad[p] = (C * M).sum() / 2
        mag[p] = (np.abs(C) * np.abs(M)).sum() / 2
    grad[2] = np.trace(C) * h[2]
    mag[2] = np.abs(np.diagonal(C)).sum() * h[2]
    return grad, mag


def loglik_grad(x, g, hyp, d, form='cho', jitter=0.0):
    """(loglik, grad[3]) in FP64 with the Matern kernel, the two forms of ``grad_oracle.loglik_grad``: ``'cho'`` (alpha
    and W by ``cho_solve``) or ``'inv'`` (W = L^-T L^-1, alpha = W g)."""
    with kernel(d):
        x, K, A = go.matrix(x, _iso(hyp), jitter)
    g = np.asarray(g, dtype=np.float64)
    n = A.shape[0]
    L = np.linalg.cholesky(A)
    if form == 'cho':
        alpha = scipy.linalg.cho_solve((L, True), g)
        W = scipy.linalg.cho_solve((L, True), np.eye(n))
    else:
        Li = scipy.linalg.solve_triangular(L, np.eye(n), lower=True)
        W = Li.T @ Li
        alpha = W @ g
    z = scipy.linalg.solve_triangular(L, g, lower=True)
    ll = -(np.dot(z, z) / 2 + np.log(np.diagonal(L)).sum() + n * LOG_2PI / 2)
    return float(ll), contract(x, K, hyp, alpha, W, d)[0]
