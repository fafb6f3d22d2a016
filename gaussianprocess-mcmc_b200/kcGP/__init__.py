"""GPU-backed stand-ins for the ``kcGP`` primitives that ``kcMCMC/sliceSample.py:13`` imports
(``from kcGP import covK, likK, tools``).  The reference's ``kcGP`` is a private fork of pyGPs 1.3.4 that is not in
its tree; these classes keep the call shapes used by the reference (SURVEY 8b) and compute on the B200.
``gpK.GPR`` is the type-II maximum-likelihood regression model (pyGPs 1.3.4 ``GPR``)."""
from . import covK, likK, tools, gpK

__all__ = ['covK', 'likK', 'tools', 'gpK']
