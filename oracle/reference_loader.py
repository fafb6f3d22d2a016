"""Load the reference's own ``kcMCMC/sliceSample.py`` UNMODIFIED as the literal oracle.

TEST INFRASTRUCTURE (see ``oracle/__init__.py``).  The original project is not
part of this repository: the loader works only where ``GPMC_REFERENCE_ROOT``
names a checkout of t-kychen/GaussianProcess-MCMC, so the literal module may not
be reached from ``-m gpu`` tests, ``smoke()`` or ``bench.py``.  The ``Tape``
classes below need no checkout.  The loader is used by ``oracle/make_golden.py``
(fixture generation) and by the CPU tests that pin :mod:`oracle.sds_oracle` to the
literal reference.

``kcMCMC/__init__.py:1`` is a Python-2 implicit relative import, so the package
cannot be imported; the module file is loaded by path instead with the ``kcGP``
shim (:mod:`oracle.kcgp_shim`) injected for ``sliceSample.py:13``.
"""
import importlib.util
import os

import numpy as np

from . import kcgp_shim

REFERENCE_ROOT = os.environ.get('GPMC_REFERENCE_ROOT', '')
_SLICE_SAMPLE = os.path.join(REFERENCE_ROOT, 'kcMCMC', 'sliceSample.py')


def available():
    return bool(REFERENCE_ROOT) and os.path.isfile(_SLICE_SAMPLE)


def load_literal(fresh=False):
    """Return the reference ``sliceSample`` module object (executed from its own file)."""
    if not available():
        raise RuntimeError('GPMC_REFERENCE_ROOT does not name a checkout of the original project (%r)' % REFERENCE_ROOT)
    kcgp_shim.install()
    name = 'gpmc_reference_sliceSample' + ('_%d' % id(object()) if fresh else '')
    spec = importlib.util.spec_from_file_location(name, _SLICE_SAMPLE)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


class Tape(object):
    """Explicit randomness for ONE ``surrogate_slice_sampling`` call.

    Draw order of the reference (``sliceSample.py``): ``z[N]`` standard normals inside
    ``aux_var_model`` (``:194``, first call only), ``v[P]`` U(0,1) for the bracket
    (``:110``), ``u0`` U(0,1) for the threshold (``:127``), then ``U[t, P]`` U(0,1) per
    shrink-loop trip ``t`` (``:132``).  Uniforms are stored on (0,1) and mapped to
    ``low + (high-low)*u`` exactly as ``numpy.random.uniform`` does.
    """

    def __init__(self, z, v, u0, U):
        self.z = np.asarray(z, dtype=np.float64)
        self.v = np.asarray(v, dtype=np.float64)
        self.u0 = float(u0)
        self.U = np.asarray(U, dtype=np.float64)

    @classmethod
    def from_seed(cls, seed, n, p=3, max_trips=64):
        rs = np.random.RandomState(seed)
        return cls(rs.standard_normal(n), rs.random_sample(p), rs.random_sample(), rs.random_sample((max_trips, p)))


class _TapeRandom(object):
    """Stand-in for ``numpy.random`` inside the literal module: replays a :class:`Tape`."""

    def __init__(self, tape):
        self.tape = tape
        self.stage = 0          # 0: expect v, 1: expect u0, 2+: trips
        self.trips = 0
        self.used_z = False

    def multivariate_normal(self, mean, cov, size):
        # sliceSample.py:194 -- cov is the diagonal S; numpy's SVD route reduces to
        # mean + sqrt(diag) * z with z in draw order (checked in make_golden.py).
        assert not self.used_z
        self.used_z = True
        sd = np.sqrt(np.diagonal(cov))
        return (np.asarray(mean) + sd * self.tape.z).reshape(1, -1)

    def uniform(self, low=0.0, high=1.0, size=None):
        if self.stage == 0:
            u = self.tape.v
        elif self.stage == 1:
            u = self.tape.u0
        else:
            if self.trips >= self.tape.U.shape[0]:
                raise RuntimeError('tape exhausted after %d trips' % self.trips)
            u = self.tape.U[self.trips]
            self.trips += 1
        self.stage += 1
        low = np.asarray(low, dtype=np.float64)
        high = np.asarray(high, dtype=np.float64)
        out = low + (high - low) * u
        return float(out) if out.ndim == 0 else out


class _NumpyProxy(object):
    """``np`` as seen by the literal module: numpy, except ``.random`` replays a tape."""

    def __init__(self, random):
        self.random = random

    def __getattr__(self, name):
        return getattr(np, name)


def run_literal_with_tape(f, x, y, hyp, scale, it, tape):
    """Run the UNMODIFIED ``surrogate_slice_sampling`` (``sliceSample.py:76-163``) on a tape.

    Returns ``(prop_f, prop_hyp, n_trips)``.  Only the module-global name ``np`` of a
    private copy of the module is rebound (to a proxy whose ``random`` replays the
    tape); not one line of the reference's code is changed.
    """
    mod = load_literal(fresh=True)
    rnd = _TapeRandom(tape)
    mod.np = _NumpyProxy(rnd)
    prop_f, prop_hyp = mod.surrogate_slice_sampling(np.array(f, dtype=np.float64), np.asarray(x, dtype=np.float64),
                                                    np.asarray(y, dtype=np.float64), np.array(hyp, dtype=np.float64),
                                                    np.asarray(scale, dtype=np.float64), iter=it)
    return np.asarray(prop_f), np.asarray(prop_hyp), rnd.trips


class EssTape(object):
    """Explicit randomness for ONE ``elliptical_slice`` call in the reference's draw order (``sliceSample.py``):
    ``nu[N]`` the ``N(0, K)`` draw of ``:41``, ``u`` U(0,1) for the slice level (``:51``), ``theta[T]`` U(0,1): the initial
    angle (``:54``) and one redraw per rejected proposal (``:74``)."""

    def __init__(self, nu, u, theta):
        self.nu = np.asarray(nu, dtype=np.float64)
        self.u = float(u)
        self.theta = np.asarray(theta, dtype=np.float64)


class _EssTapeRandom(object):
    def __init__(self, tape):
        self.tape = tape
        self.calls = 0          # uniform() calls: 0 -> u, 1 -> theta[0], k -> theta[k-1]

    def multivariate_normal(self, mean, cov, size):
        return (np.asarray(mean) + self.tape.nu).reshape(1, -1)            # :41 (mean is zero)

    def uniform(self, low=0.0, high=1.0, size=None):
        if self.calls == 0:
            u = self.tape.u
        else:
            if self.calls - 1 >= self.tape.theta.shape[0]:
                raise RuntimeError('tape exhausted after %d angles' % (self.calls - 1))
            u = self.tape.theta[self.calls - 1]
        self.calls += 1
        return float(low + (high - low) * u)


def run_literal_ess_with_tape(f, x, y, hyp, tape):
    """Run the UNMODIFIED ``elliptical_slice`` (``sliceSample.py:15-74``) on a tape.  Returns ``(prop_f, n_proposals)``."""
    mod = load_literal(fresh=True)
    rnd = _EssTapeRandom(tape)
    mod.np = _NumpyProxy(rnd)
    prop_f = mod.elliptical_slice(np.array(f, dtype=np.float64), np.asarray(x, dtype=np.float64),
                                  np.asarray(y, dtype=np.float64), np.array(hyp, dtype=np.float64))
    return np.asarray(prop_f), rnd.calls - 1
