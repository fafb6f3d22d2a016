"""Reference gradient of the GP log marginal likelihood with respect to the natural-scale hyper-parameters
``hyp = (ell.., sf, sn)`` -- the quantity ``gpmc_loglik_grad_batched`` returns (include/gpmc.h):

    loglik = -(0.5 g^T A^-1 g + 0.5 log|A| + 0.5 N log 2 pi),   A = K + S (+ jitter I),  S_ii = sn^2 (sliceSample.py:184-187)
    d loglik / d th_p = 0.5 sum_ij (alpha_i alpha_j - W_ij) dA_ij/d th_p,   alpha = A^-1 g,  W = A^-1

TEST INFRASTRUCTURE (see ``oracle/__init__.py``).  Two FP64 forms (``cho_solve`` of the Cholesky factor, and the explicit
inverse ``L^-T L^-1``) whose spread is FP64's own error on an item, and a numpy ``longdouble`` form built on
``oracle/xprec.py`` (the truth for N <= 512).  ``A`` is the FP64 matrix the device assembles (``sds_oracle.cov_matrix`` +
``s_diagonal``); the derivative factors ``dA/dtheta`` are formed in the working precision from ``x`` and ``hyp``."""
import numpy as np
import scipy.linalg

from . import sds_oracle as so
from . import xprec

LOG_2PI = np.log(2 * np.pi)


def matrix(x, hyp, jitter=0.0):
    """(x[N, D], K, A = K + S + jitter I) in FP64, as the device assembles them."""
    x = np.asarray(x, dtype=np.float64)
    if x.ndim == 1:
        x = x.reshape(-1, 1)
    hyp = np.asarray(hyp, dtype=np.float64)
    K = so.cov_matrix(x, hyp)
    A = K + np.diag(so.s_diagonal(np.diagonal(K), hyp[-1]))
    if jitter:
        A = A + jitter * np.eye(A.shape[0])
    return x, K, A


def contract(x, K, hyp, alpha, W, dtype=np.float64):
    """The gradient from alpha = A^-1 g and W = A^-1 (full symmetric), in ``dtype``; also returns the magnitude
    sum_ij |alpha_i alpha_j - W_ij| |dA_ij/dtheta_p| of each component's terms (the scale of its rounding error)."""
    hyp = np.asarray(hyp, dtype=np.float64)
    P = hyp.shape[0]
    n_ell = P - 2
    x = np.asarray(x).astype(dtype)
    K = np.asarray(K).astype(dtype)
    a = np.asarray(alpha).astype(dtype)
    W = np.asarray(W).astype(dtype)
    C = np.outer(a, a) - W
    h = hyp.astype(dtype)
    grad, mag = np.zeros(P, dtype=dtype), np.zeros(P, dtype=dtype)
    if n_ell == 1:
        d2 = np.zeros_like(K)
        for d in range(x.shape[1]):
            d2 += (x[:, d][:, None] - x[:, d][None, :]) ** 2
        dA = [K * d2 / h[0] ** 3]
    else:
        dA = [K * (x[:, d][:, None] - x[:, d][None, :]) ** 2 / h[d] ** 3 for d in range(n_ell)]
    dA.append(2 * K / h[n_ell])
    for p, M in enumerate(dA):
        grad[p] = (C * M).sum() / 2
        mag[p] = (np.abs(C) * np.abs(M)).sum() / 2
    dsn = 2 * h[n_ell + 1]
    grad[P - 1] = np.trace(C) * dsn / 2
    mag[P - 1] = np.abs(np.diagonal(C)).sum() * dsn / 2
    return grad, mag


def loglik_grad(x, g, hyp, form='cho', jitter=0.0, chol=None):
    """(loglik, grad[P]) in FP64.  ``form='cho'``: alpha and W by ``cho_solve``; ``form='inv'``: the explicit inverse
    W = L^-T L^-1, alpha = W g.  ``chol(A)`` gives the lower factor (default LAPACK's), so that callers can measure FP64's
    error over several summation orders.  Raises ``LinAlgError`` when A + jitter I is not positive definite."""
    x, K, A = matrix(x, hyp, jitter)
    g = np.asarray(g, dtype=np.float64)
    n = A.shape[0]
    L = np.linalg.cholesky(A) if chol is None else chol(A)
    if form == 'cho':
        alpha = scipy.linalg.cho_solve((L, True), g)
        W = scipy.linalg.cho_solve((L, True), np.eye(n))
    else:
        Li = scipy.linalg.solve_triangular(L, np.eye(n), lower=True)
        W = Li.T @ Li
        alpha = W @ g
    z = scipy.linalg.solve_triangular(L, g, lower=True)
    ll = -(np.dot(z, z) / 2 + np.log(np.diagonal(L)).sum() + n * LOG_2PI / 2)
    return float(ll), contract(x, K, hyp, alpha, W)[0]


def loglik_grad_xprec(x, g, hyp, jitter=0.0):
    """(loglik, grad[P], mag[P]) in numpy ``longdouble`` from the FP64 A (xprec.chol / triangular inverse); O(N^3)
    longdouble work, meant for N <= 512."""
    xprec.require()
    x, K, A = matrix(x, hyp, jitter)
    LD = xprec.LD
    L = xprec.chol(xprec.symmetric(A))
    X = xprec._tri_inv(L)                      # L^-1
    W = np.einsum('ki,kj->ij', X, X)           # A^-1 = L^-T L^-1
    gl = np.asarray(g, dtype=np.float64).astype(LD)
    alpha = W.dot(gl)
    z = X.dot(gl)
    ll = xprec.loglik_of_factor(L, z)
    grad, mag = contract(x, K, hyp, alpha, W, dtype=LD)
    return ll, grad, mag
