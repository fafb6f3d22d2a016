"""CPU restatement (numpy/scipy, FP64) of the marginal slice sampler (``gpmc_marginal_run``), driven by tapes.

TEST INFRASTRUCTURE (see ``oracle/__init__.py``): the checker the CUDA path is compared with.  Never imported by the
product.

Under a Gaussian likelihood the latent f integrates out, and the hyper-parameter posterior is
``p(theta | y) ~ N(y - m; 0, K + S) * prod_p prior_p(theta_p)``.  One transition is the reference's hyper-rectangle slice
sampler (``sliceSample.py:110-163``) without f, g and the truncated-Gaussian term.  Everything is the existing
restatement: ``sds_oracle.loglik_unit`` (chol form) as the log-likelihood, ``log_gamma`` and ``_sum_density`` for the
density, and the bracket / shrink arithmetic of ``sds_oracle.surrogate_slice_sampling``.  For a Matern kind, run inside
``matern_oracle.kernel(d)``.
"""
import numpy as np

from . import sds_oracle as so


def loglik(x, r, hyp):
    """``log N(r; 0, K + S)`` at ``hyp``; NaN when ``jitchol`` gives up (a rejected proposal)."""
    try:
        return so.loglik_unit(x, r, hyp, form='chol')
    except (np.linalg.LinAlgError, ValueError):
        return np.nan


def density(head, hyp, G, it, burn_in, prior_k, prior_theta):
    """``head + prior[sf] + prior[ell..] + G`` (+ ``prior[sn]`` once ``it >= burn_in``): ``sliceSample.py:127-129,150-152``."""
    n_ell = hyp.shape[0] - 2
    prior, _ = so.log_gamma(hyp, prior_k, prior_theta, True)
    acc = so._sum_density(head, prior, G, n_ell)
    if it >= burn_in:
        acc += prior[-1]
    return acc


def transition(x, r, hyp, G_cur, scale, it, burn_in, v, u0, U, prior_k, prior_theta, max_trips=None):
    """One transition from ``(hyp, G_cur)`` on the tape ``v[P]``, ``u0``, ``U[T, P]``; ``r = y - m``.

    Returns ``(hyp', G', trips, exhausted)``; an exhausted transition (budget ``min(max_trips, T)`` used up) keeps
    ``(hyp, G_cur)``."""
    hyp = np.asarray(hyp, dtype=np.float64)
    scale = np.asarray(scale, dtype=np.float64)
    P = hyp.shape[0]
    vv = 0. + (scale - 0.) * np.asarray(v, dtype=np.float64)                   # :110
    hyp_min = np.maximum(hyp - vv, 0)                                          # :111
    hyp_max = hyp_min + scale                                                  # :112
    threshold = density(np.log(u0), hyp, G_cur, it, burn_in, prior_k, prior_theta)   # :127-129
    budget = U.shape[0] if max_trips is None else min(max_trips, U.shape[0])
    for trip in range(budget):                                                 # :131
        prop = hyp_min + (hyp_max - hyp_min) * U[trip]                         # :132
        if it < burn_in:
            prop[P - 1] = hyp[P - 1]                                           # :133-134
        G = loglik(x, r, prop)                                                 # :136-147
        proposal = density(0., prop, G, it, burn_in, prior_k, prior_theta)     # :149-152
        if proposal > threshold and np.isfinite(proposal):                     # :154
            return prop, G, trip + 1, False                                    # :156
        for i in range(P):                                                     # :159-163
            if prop[i] < hyp[i]:
                hyp_min[i] = prop[i]
            else:
                hyp_max[i] = prop[i]
    return hyp.copy(), G_cur, budget, True


def run_chain(x, y, hyp0, scale, it0, n_iters, burn_in, tape_v, tape_u0, tape_U, m=None, max_trips=64,
              prior_k=None, prior_theta=None):
    """One chain over ``n_iters`` transitions on tapes ``v[n_iters, P]``, ``u0[n_iters]``, ``U[n_iters, T, P]``.

    Returns ``(hist_hyp[n_iters, P], hist_loglik[n_iters], hist_trips[n_iters], exhausted)`` as ``gpmc_marginal_run``
    reports them (``exhausted = -1``: the starting log-likelihood is not finite; the state is kept with 0 trips)."""
    y = np.asarray(y, dtype=np.float64).reshape(-1)
    m = float(np.mean(y)) if m is None else m                                  # :102
    r = y - m
    hyp = np.asarray(hyp0, dtype=np.float64).copy()
    P = hyp.shape[0]
    if prior_k is None or prior_theta is None:
        prior_k, prior_theta = so.prior_constants(P - 2)
    hh = np.zeros((n_iters, P))
    ll = np.zeros(n_iters)
    tt = np.zeros(n_iters, dtype=np.int64)
    G = loglik(x, r, hyp)
    if not np.isfinite(G):
        hh[:] = hyp
        ll[:] = G
        return hh, ll, tt, -1
    exhausted = 0
    for k in range(n_iters):
        hyp, G, tt[k], ex = transition(x, r, hyp, G, scale, it0 + k, burn_in, tape_v[k], tape_u0[k], tape_U[k],
                                       prior_k, prior_theta, max_trips)
        exhausted += int(ex)
        hh[k], ll[k] = hyp, G
    return hh, ll, tt, exhausted


def log_posterior(x, r, hyp, prior_k, prior_theta):
    """Unnormalised ``log p(theta | y)`` with every prior (``burn_in = 0``): the density the sampler leaves invariant."""
    return density(0., np.asarray(hyp, dtype=np.float64), loglik(x, r, hyp), 0, 0, prior_k, prior_theta)


def posterior_grid(x, y, m=None, prior=None, kind=None, bounds=((-3., 3.),) * 3, n=(33, 33, 33)):
    """Exact marginal moments of ``(log ell, log sf, log sn)`` under ``p(theta | y)`` by quadrature on a grid of
    ``log theta`` (composite Simpson, ``n`` odd per axis, ``bounds`` in log space; ``n = 1`` fixes an axis at ``lo``).
    ``kind``: None for SE, or a Matern ``d`` (1, 3, 5).  For small N (every grid point is one ``loglik_unit``).

    Returns ``{'mean': [3], 'var': [3], 'edge': float}`` -- ``edge`` is the largest density on the grid's boundary faces
    relative to its maximum (small when the bounds hold the posterior)."""
    from contextlib import nullcontext
    from . import matern_oracle
    y = np.asarray(y, dtype=np.float64).reshape(-1)
    m = float(np.mean(y)) if m is None else m
    r = y - m
    pk, pth = so.prior_constants(1) if prior is None else prior
    axes = [np.linspace(lo, hi, k) if k > 1 else np.array([lo]) for (lo, hi), k in zip(bounds, n)]

    def simpson(k):
        if k == 1:
            return np.ones(1)
        if k % 2 == 0:
            raise ValueError('Simpson needs an odd number of points')
        w = np.ones(k)
        w[1:-1:2], w[2:-1:2] = 4., 2.
        return w
    W = [simpson(len(a)) for a in axes]
    logp = np.empty([len(a) for a in axes])
    with (matern_oracle.kernel(kind) if kind else nullcontext()):
        for idx in np.ndindex(*logp.shape):
            lt = np.array([axes[d][idx[d]] for d in range(3)])
            # density of log theta: p(theta) * theta (Jacobian)
            logp[idx] = log_posterior(x, r, np.exp(lt), pk, pth) + lt.sum()
    logp = np.where(np.isfinite(logp), logp, -np.inf)
    p = np.exp(logp - logp.max())
    w = W[0][:, None, None] * W[1][None, :, None] * W[2][None, None, :]
    Z = (w * p).sum()
    mean, var = np.zeros(3), np.zeros(3)
    for d in range(3):
        shape = [1, 1, 1]
        shape[d] = -1
        a = axes[d].reshape(shape)
        mean[d] = (w * p * a).sum() / Z
        var[d] = (w * p * (a - mean[d]) ** 2).sum() / Z
    edge = 0.0
    for d in range(3):
        if len(axes[d]) > 1:
            edge = max(edge, p.take(0, axis=d).max(), p.take(-1, axis=d).max())
    return {'mean': mean, 'var': var, 'edge': edge}


def batch_means_se(samples, n_batches=None):
    """Standard error of the mean of a ``[n_chains, n_samples]`` array: every chain is one batch when there are several
    chains (independent batches), else ``n_batches`` contiguous batches of the single chain."""
    s = np.asarray(samples, dtype=np.float64)
    if s.ndim == 2 and s.shape[0] > 1:
        b = s.mean(axis=1)
    else:
        s = s.reshape(-1)
        k = n_batches or 50
        L = s.shape[0] // k
        b = s[:k * L].reshape(k, L).mean(axis=1)
    return b.std(ddof=1) / np.sqrt(b.shape[0])
