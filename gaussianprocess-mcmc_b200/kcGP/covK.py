"""``kcGP.covK``: ``RBF(log_ell, log_sigma).getCovMatrix(x=, z=, mode=)`` (call sites ``sliceSample.py:38-39,104-105,
136-137,262-263``; pyGPs 1.3.4 ``cov.RBF`` semantics: ``sf2 * exp(-0.5 * sqdist(x/ell, z/ell))``), ``RBFard``, and
``Matern(log_ell, d, log_sigma)`` (pyGPs 1.3.4 ``cov.Matern``, restated: ``oracle/matern_oracle.py``)."""
import numpy as np

from .. import ops


class RBF(object):
    def __init__(self, log_ell=0., log_sigma=0.):
        self.hyp = [log_ell, log_sigma]

    def _natural(self):
        # the kernel works on natural-scale (ell, sf); the device applies exp(log(.)) again, as the reference's
        # covK.RBF(np.log(ll), np.log(sf)) call pattern does
        return np.array([np.exp(self.hyp[0]), np.exp(self.hyp[1]), 1.0])

    def getCovMatrix(self, x=None, z=None, mode=None):
        if mode == 'self_test':
            return np.full((np.asarray(z).shape[0], 1), np.exp(2. * self.hyp[1]))     # sf2 * exp(0)
        if mode == 'train':
            x = np.asarray(x, dtype=np.float64)
            n = x.shape[0]
            return ops.cov_assemble(x, self._natural()[None]).cpu().numpy()[0, :, :n]
        if mode == 'cross':
            return ops.cov_cross(x, z, self._natural()).cpu().numpy()
        raise ValueError("mode must be 'train', 'cross' or 'self_test'")


class RBFard(RBF):
    def __init__(self, D=None, log_ell_list=None, log_sigma=0.):
        if log_ell_list is None:
            log_ell_list = [0. for _ in range(D)]
        self.hyp = list(log_ell_list) + [log_sigma]

    def _natural(self):
        return np.array([np.exp(h) for h in self.hyp] + [1.0])


class Matern(object):
    """Matern covariance with d = 2 nu in {1, 3, 5}: ``sf2 * f_d(t) * exp(-t)``, ``t = |sqrt(d) x / ell - sqrt(d) z / ell|``,
    ``f_1 = 1``, ``f_3 = 1 + t``, ``f_5 = 1 + t (1 + t / 3)``; isotropic, ``hyp = [log_ell, log_sigma]`` as pyGPs keeps it."""
    _KINDS = {1: ops.KIND_MATERN1, 3: ops.KIND_MATERN3, 5: ops.KIND_MATERN5}

    def __init__(self, log_ell=0., d=3, log_sigma=0.):
        if d not in self._KINDS:
            raise ValueError('Matern: d must be 1, 3 or 5 (got %r)' % (d,))
        self.d = int(d)
        self.hyp = [log_ell, log_sigma]

    @property
    def kind(self):
        return self._KINDS[self.d]

    def _natural(self):
        return np.array([np.exp(self.hyp[0]), np.exp(self.hyp[1]), 1.0])

    def getCovMatrix(self, x=None, z=None, mode=None):
        if mode == 'self_test':
            return np.full((np.asarray(z).shape[0], 1), np.exp(2. * self.hyp[1]))     # sf2 * f_d(0) * exp(0)
        if mode == 'train':
            x = np.asarray(x, dtype=np.float64)
            n = x.shape[0]
            return ops.cov_assemble(x, self._natural()[None], kind=self.kind).cpu().numpy()[0, :, :n]
        if mode == 'cross':
            return ops.cov_cross(x, z, self._natural(), kind=self.kind).cpu().numpy()
        raise ValueError("mode must be 'train', 'cross' or 'self_test'")
