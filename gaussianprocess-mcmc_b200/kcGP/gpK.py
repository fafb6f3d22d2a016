"""``kcGP.gpK.GPR``: GP regression with type-II maximum-likelihood hyper-parameters -- the pyGPs 1.3.4 ``GPR`` names the
reference uses (``framework.py:158,208`` ``updOpt``, ``demoRegression.py:78,110-115``, and ``plotResult.py:100``, where a
``GPR`` is the ``model`` that ``inf_mcmc(f, model)`` reads ``x, y, xs, meanfunc, covfunc, likfunc`` from).

Limited to a Gaussian likelihood (``likK.Gauss``), a zero mean and ``covK.RBF`` / ``covK.RBFard`` (what the reference
needs) or ``covK.Matern`` (d = 1, 3, 5).  The negative log marginal likelihood and its gradient come from ``ops.loglik_grad_batched``
(``gpmc_loglik_grad_batched``: assembly, Cholesky, ``A^-1`` and the gradient contraction on the device); the predictive
from ``ops.predict_batched``.  Hyper-parameters are kept on pyGPs' log scale (``covfunc.hyp``, ``log(likfunc.sn)``)."""
import numpy as np
import scipy.optimize

from .. import ops
from . import covK, likK


def _np(t):
    return t.cpu().numpy() if hasattr(t, 'cpu') else np.asarray(t)


class ZeroMean(object):
    """pyGPs ``mean.Zero``: ``getMean(x)`` is a column of zeros; no hyper-parameters."""
    hyp = []

    def getMean(self, x=None):
        return np.zeros((np.asarray(x).shape[0], 1))


class dnlZStruct(object):
    """Derivatives of ``nlZ`` with respect to the log hyper-parameters, in pyGPs' layout (``mean``, ``cov``, ``lik``)."""

    def __init__(self, cov, lik):
        self.mean = []
        self.cov = list(cov)
        self.lik = list(lik)


class GPR(object):
    def __init__(self):
        self.x = None
        self.y = None
        self.xs = None
        self.ys = None
        self.meanfunc = ZeroMean()
        self.covfunc = covK.RBF()
        self.likfunc = likK.Gauss(log_sigma=np.log(0.1))
        self.nlZ = None
        self.dnlZ = None
        self.posterior = None
        self.num_restarts = 0
        self.covRange = None
        self.likRange = None
        self.method = 'BFGS'
        self.optim_result = None
        self.hyp_samples = None

    # ------------------------------------------------------------------ model set-up (pyGPs names)
    def setData(self, x, y):
        x = np.asarray(x, dtype=np.float64)
        self.x = x.reshape(-1, 1) if x.ndim == 1 else x
        self.y = np.asarray(y, dtype=np.float64).reshape(-1, 1)

    def setPrior(self, mean=None, kernel=None):
        if mean is not None:
            raise NotImplementedError('GPR: only the zero mean is supported')
        if kernel is not None:
            if not isinstance(kernel, (covK.RBF, covK.Matern)):
                raise NotImplementedError('GPR: only covK.RBF / covK.RBFard / covK.Matern kernels are supported')
            self.covfunc = kernel

    def setNoise(self, log_sigma=np.log(0.1)):
        self.likfunc = likK.Gauss(log_sigma=log_sigma)

    def setOptimizer(self, method='BFGS', num_restarts=0, covRange=None, likRange=None):
        """Every method runs ``scipy.optimize.minimize(method='L-BFGS-B', jac=True)`` over the log hyper-parameters.
        ``num_restarts`` more runs start one after another from points drawn uniformly in ``covRange`` (one ``(lo, hi)``
        per covariance hyper-parameter) and ``likRange`` (one for ``log sn``); the best ``nlZ`` is kept."""
        self.method = method
        self.num_restarts = int(num_restarts)
        self.covRange = covRange
        self.likRange = likRange

    # ------------------------------------------------------------------ hyper-parameters
    def _kind_kw(self):
        # an RBF / RBFard row is SE iso / ARD by its width (the ops default); a Matern kernel names its kind
        kind = getattr(self.covfunc, 'kind', None)
        return {} if kind is None else {'kind': kind}

    def _log_hyp(self):
        return np.concatenate([np.asarray(self.covfunc.hyp, dtype=np.float64), [np.log(self.likfunc.sn)]])

    def _set_log_hyp(self, h):
        h = np.asarray(h, dtype=np.float64)
        self.covfunc.hyp = list(h[:-1])
        self.likfunc = likK.Gauss(log_sigma=h[-1])

    def _nlz_and_grad(self, log_hyp):
        """``nlZ`` and its gradient with respect to the log hyper-parameters (pyGPs' sign and scale)."""
        theta = np.exp(np.asarray(log_hyp, dtype=np.float64))
        ll, grad, info = ops.loglik_grad_batched(self.x, self.y.reshape(1, -1), theta[None], **self._kind_kw())
        ll, grad = float(_np(ll)[0]), _np(grad)[0]
        if int(_np(info)[0]) != 0 or not np.isfinite(ll) or not np.all(np.isfinite(grad)):
            return np.inf, np.zeros_like(theta)
        return -ll, -theta * grad

    def getPosterior(self, x=None, y=None, der=True):
        """Returns ``(nlZ, dnlZ, post)``.  ``post`` is None: the factor and ``alpha`` of the posterior stay on the device
        (``predict`` recomputes what it needs there).  ``der=False`` leaves ``dnlZ`` None."""
        if x is not None and y is not None:
            self.setData(x, y)
        nlZ, g = self._nlz_and_grad(self._log_hyp())
        self.nlZ = nlZ
        self.dnlZ = dnlZStruct(g[:-1], g[-1:]) if der else None
        self.posterior = None
        return self.nlZ, self.dnlZ, self.posterior

    def optimize(self, x=None, y=None, numIterations=40):
        if x is not None and y is not None:
            self.setData(x, y)
        starts = [self._log_hyp()]
        for _ in range(self.num_restarts):
            if self.covRange is None or self.likRange is None:
                raise ValueError('GPR.optimize: restarts need covRange and likRange (setOptimizer)')
            ranges = list(self.covRange) + list(self.likRange)
            starts.append(np.array([np.random.uniform(lo, hi) for lo, hi in ranges]))
        best = None
        for h0 in starts:
            res = scipy.optimize.minimize(self._nlz_and_grad, h0, jac=True, method='L-BFGS-B',
                                          options={'maxiter': int(numIterations)})
            if best is None or res.fun < best.fun:
                best = res
        self.optim_result = best
        self._set_log_hyp(best.x)
        return self.getPosterior()

    # ------------------------------------------------------------------ fully Bayesian hyper-parameters
    def sampleHyp(self, n_iters, n_chains=8, scale=None, burn=0, thin=1, seed=0, max_trips=64):
        """Posterior samples of the hyper-parameters instead of one type-II ML point: ``n_chains`` slice-sampling chains
        (``ops.marginal_run``: the latent f integrated out, the hyper-priors of ``sliceSample.py:124-125``, every prior
        from the first iteration) start at the current hyper-parameters and run ``n_iters`` transitions each.  The
        samples after the first ``burn`` of every chain, every ``thin``-th, are kept as natural-scale rows
        ``(ell.., sf, sn)`` in ``hyp_samples`` and returned.  ``scale``: the slice widths (default: the current theta)."""
        theta = np.exp(self._log_hyp())
        scale = theta if scale is None else np.asarray(scale, dtype=np.float64)
        import torch
        H = torch.tensor(np.tile(theta, (int(n_chains), 1))).cuda()
        hh, _, _, _ = ops.marginal_run(self.x, self.y.reshape(-1), H, scale, 0, int(n_iters), m=0.0, burn_in=0, seed=seed,
                                       max_trips=max_trips, **self._kind_kw())
        self.hyp_samples = _np(hh)[:, int(burn)::int(thin), :].reshape(-1, theta.shape[0]).copy()
        return self.hyp_samples

    # ------------------------------------------------------------------ prediction
    def predict(self, xs, ys=None, samples=None):
        """``(ym, ys2, fm, fs2, lp)`` as columns ``[M, 1]``: latent mean / variance (clamped at 0, as pyGPs does),
        ``ym = fm``, ``ys2 = fs2 + sn^2``, ``lp = log N(ys; ym, ys2)`` (``ys`` zero when omitted, as pyGPs evaluates it).

        ``samples[S, P]`` (natural-scale rows, e.g. ``hyp_samples``): the predictive of the mixture over them, from ONE
        ``ops.predict_batched`` call -- ``fm`` the mean of the per-sample means, ``fs2`` the mean of ``fs2 + fmu^2`` minus
        ``fm^2``, ``ys2 = fs2 +`` the mean of ``sn^2``."""
        xs = np.asarray(xs, dtype=np.float64)
        self.xs = xs.reshape(-1, 1) if xs.ndim == 1 else xs
        M = self.xs.shape[0]
        theta = np.exp(self._log_hyp())[None] if samples is None else np.atleast_2d(np.asarray(samples, dtype=np.float64))
        S = theta.shape[0]
        m = self.meanfunc.getMean(self.x)
        fm_rows = np.tile((self.y - m).reshape(1, -1), (S, 1))
        fmu, fs2, info = ops.predict_batched(self.x, self.xs, fm_rows, theta, **self._kind_kw())
        if np.any(_np(info) != 0):
            raise np.linalg.LinAlgError('not positive definite, even with jitter.')
        fmu = _np(fmu).reshape(S, M)
        fs2 = np.maximum(_np(fs2).reshape(S, M), 0)
        if samples is None:
            fm = self.meanfunc.getMean(self.xs) + fmu.reshape(M, 1)
            fs2 = fs2.reshape(M, 1)
            ym, ys2 = fm, fs2 + self.likfunc.sn ** 2
        else:
            mu = fmu.mean(axis=0)
            fm = self.meanfunc.getMean(self.xs) + mu.reshape(M, 1)
            fs2 = ((fs2 + fmu ** 2).mean(axis=0) - mu ** 2).reshape(M, 1)
            ym, ys2 = fm, fs2 + np.mean(theta[:, -1] ** 2)
        yy = np.zeros((M, 1)) if ys is None else np.asarray(ys, dtype=np.float64).reshape(M, 1)
        lp = -(yy - ym) ** 2 / (2 * ys2) - 0.5 * np.log(2 * np.pi * ys2)
        if ys is not None:
            self.ys = yy
        return ym, ys2, fm, fs2, lp
