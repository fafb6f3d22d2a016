"""Extended-precision (numpy ``longdouble``) reference for the Cholesky factor, the forward substitution and the
log-likelihood, and backward errors of FP64 factors and solves measured against it.

TEST INFRASTRUCTURE (see ``oracle/__init__.py``).  On x86-64 ``longdouble`` is the 80-bit format (eps 2^-64 = 1.08e-19,
about 2000 times finer than FP64), so a result computed here is the exact answer of the FP64 inputs to well below FP64's
rounding; residuals of FP64 factors are formed here too, so that a backward error of one or two FP64 ulps is resolved.
Where ``longdouble`` is plain ``double`` (e.g. MSVC, some ARM ABIs) ``AVAILABLE`` is False and ``require()`` raises.

Every routine works on the lower triangle and skips the exact-zero envelope of its matrix: row i of A starts at its
first nonzero column, and Cholesky keeps that envelope exactly, so banded K+S at N = 4096 costs O(N w^2), not O(N^3).
Matrices built on the host must be symmetric (``symmetric()``): LAPACK and the device read only the lower triangle.
"""
import numpy as np

LD = np.longdouble
EPS = 2.0 ** -53                          # the unit in which backward errors are reported (FP64 unit roundoff)
AVAILABLE = bool(np.finfo(LD).eps <= 1.1e-19)
REASON = 'numpy longdouble has eps %.3g here: no extended precision on this host' % float(np.finfo(LD).eps)
NB = 64
# Entries of K far from the diagonal are subnormal, and so are the products that reproduce them: each of the n terms of
# an inner product may then lose 2^-1074 absolutely, whatever |L||L^T| is.  The componentwise errors divide by
# |L||L^T| + UNDERFLOW * n, so that such a loss counts as at most one EPS.
UNDERFLOW = 2.0 ** -1074 / EPS
LOG_2PI = np.log(2 * LD('3.14159265358979323846264338327950288'))


def require():
    if not AVAILABLE:
        raise RuntimeError(REASON)


def symmetric(A):
    """The symmetric matrix whose lower triangle is A's (what LAPACK and the device read)."""
    A = np.asarray(A)
    return np.tril(A) + np.tril(A, -1).T


def _mm(a, b):
    # einsum's plain loop is about 2.5x faster than matmul's for longdouble
    return np.einsum('ik,kj->ij', a, b)


def envelope(A):
    """First nonzero column of every row of the lower triangle of A (the diagonal when the row is zero left of it)."""
    A = np.asarray(A)
    n = A.shape[0]
    nz = np.tril(A) != 0
    nz[np.arange(n), np.arange(n)] = True
    return nz.argmax(axis=1)


def _spans(env, n):
    """Per block of NB rows: (i0, i1, k0) with k0 the smallest envelope start of the block's rows."""
    out = []
    for i0 in range(0, n, NB):
        i1 = min(n, i0 + NB)
        out.append((i0, i1, int(env[i0:i1].min())))
    return out


def chol(A):
    """Lower Cholesky factor of the FP64 matrix A (lower triangle read) in longdouble, left-looking in panels of NB
    columns.  Raises ``np.linalg.LinAlgError`` at a non-positive pivot."""
    require()
    A = np.asarray(A)
    n = A.shape[0]
    env = envelope(A)
    # last_row[c] = the last row with env <= c (the rows a panel ending at column c reaches): a running max over env
    last_row = np.full(n, -1)
    np.maximum.at(last_row, env, np.arange(n))
    last_row = np.maximum.accumulate(last_row)
    L = np.zeros((n, n), dtype=LD)
    for j in range(0, n, NB):
        e = min(n, j + NB)
        r1 = max(e, int(last_row[e - 1]) + 1)
        k0 = int(env[j:r1].min())
        P = A[j:r1, j:e].astype(LD)
        if k0 < j:
            P -= _mm(L[j:r1, k0:j], L[j:e, k0:j].T)
        for k in range(e - j):
            if k:
                P[k:, k] -= np.dot(P[k:, :k], P[k, :k])
            d = P[k, k]
            if not d > 0:
                raise np.linalg.LinAlgError('leading minor %d is not positive definite' % (j + k + 1))
            P[k, k] = np.sqrt(d)
            P[k + 1:, k] /= P[k, k]
        P[:e - j] = np.tril(P[:e - j])
        L[j:r1, j:e] = P
    return L


def trsv(L, b):
    """x with L x = b by forward substitution in longdouble (L lower, read from the lower triangle)."""
    require()
    L = np.asarray(L)
    n = L.shape[0]
    x = np.asarray(b).astype(LD).copy()
    for i0 in range(0, n, NB):
        i1 = min(n, i0 + NB)
        if i0:
            x[i0:i1] -= np.dot(L[i0:i1, :i0].astype(LD), x[:i0])
        for i in range(i0, i1):
            if i > i0:
                x[i] -= np.dot(L[i, i0:i].astype(LD), x[i0:i])
            x[i] /= LD(L[i, i])
    return x


def loglik_of_factor(L, z):
    """-(0.5 z^T z + sum log L_ii + 0.5 N log 2 pi) in longdouble for a given factor L and border row z = L^-1 g."""
    require()
    z = np.asarray(z).astype(LD)
    d = np.diagonal(np.asarray(L)).astype(LD)
    return -(np.dot(z, z) / 2 + np.log(d).sum() + z.shape[0] * LOG_2PI / 2)


def loglik(A, g):
    """log N(g; 0, A) of the FP64 matrix A (lower triangle) and vector g, in longdouble."""
    L = chol(A)
    return loglik_of_factor(L, trsv(L, g))


def _tri_inv(L):
    """Inverse of a lower-triangular longdouble matrix, by block rows."""
    n = L.shape[0]
    X = np.zeros_like(L)
    for i0 in range(0, n, NB):
        i1 = min(n, i0 + NB)
        m = i1 - i0
        D = np.zeros((m, m), dtype=LD)
        for i in range(m):                    # forward substitution on the identity
            D[i, i] = 1 / L[i0 + i, i0 + i]
            if i:
                D[i, :i] = -np.dot(L[i0 + i, i0:i0 + i], D[:i, :i]) * D[i, i]
        if i0:
            X[i0:i1, :i0] = -_mm(D, _mm(L[i0:i1, :i0], X[:i0, :i0]))
        X[i0:i1, i0:i1] = D
    return X


def r_matrix(K, S):
    """R = S - S (K+S)^-1 S (sliceSample.py:197-198 in the reduced form) in longdouble, from FP64 K and diag S."""
    require()
    S = np.asarray(S).astype(LD)
    A = np.asarray(K).astype(LD) + np.diag(S)
    n = A.shape[0]
    X = _tri_inv(chol(symmetric(A)))      # (K+S)^-1 = X^T X
    Q = np.zeros((n, n), dtype=LD)
    for i0 in range(0, n, NB):            # lower triangle of X^T X; X[k, i] = 0 for k < i
        i1 = min(n, i0 + NB)
        Q[i0:i1, :i1] = _mm(X[i0:, i0:i1].T, X[i0:, :i1])
    R = np.diag(S) - S[:, None] * Q * S[None, :]
    return symmetric(R)


def r_plus_jitter(K, S):
    """FP64 R + 1e-11 I (the matrix sliceSample.py:205 factors), formed in longdouble, symmetrized and rounded once."""
    R = r_matrix(K, S)
    return symmetric((R + LD(1e-11) * np.eye(R.shape[0], dtype=LD)).astype(np.float64))


def backward_error(A, L):
    """(componentwise, normwise) backward error of the FP64 factor L of the FP64 matrix A, in units of EPS, over the
    lower triangle: max |A - L L^T|_ij / (|L| |L^T| + UNDERFLOW n)_ij and ||A - L L^T||_F / ||A||_F.

    The residual is formed only inside A's envelope; L must be exactly zero left of it (Cholesky keeps the envelope),
    which is asserted, and then L L^T is zero there too."""
    require()
    A = np.asarray(A, dtype=np.float64)
    L = np.asarray(L, dtype=np.float64)
    n = A.shape[0]
    env = envelope(A)
    left = np.arange(n)[None, :] < env[:, None]
    assert not np.any(L[left]), 'L is nonzero left of the envelope of A'
    comp, num2, den2 = 0.0, LD(0), LD(0)
    for i0, i1, k0 in _spans(env, n):
        Lr = L[i0:i1, k0:i1]
        M = _mm(Lr.astype(LD), L[k0:i1, k0:i1].T.astype(LD))
        R = np.tril(A[i0:i1, k0:i1].astype(LD) - M, i0 - k0)
        D = np.abs(Lr) @ np.abs(L[k0:i1, k0:i1]).T + UNDERFLOW * n
        Rf = np.abs(R).astype(np.float64)
        with np.errstate(divide='ignore', invalid='ignore'):
            q = np.where(Rf == 0, 0.0, Rf / D)
        comp = max(comp, float(q.max()))
        num2 += (R * R).sum()
        Al = np.tril(A[i0:i1, k0:i1], i0 - k0).astype(LD)
        den2 += (Al * Al).sum()
    return comp / EPS, float(np.sqrt(num2 / den2)) / EPS


def solve_backward_error(L, b, z):
    """max_i |b - L z|_i / (|L| |z| + UNDERFLOW n)_i in units of EPS for the FP64 solution z of L z = b (L lower)."""
    require()
    L = np.tril(np.asarray(L, dtype=np.float64))
    z = np.asarray(z, dtype=np.float64)
    r = np.abs(np.asarray(b).astype(LD) - np.dot(L.astype(LD), z.astype(LD))).astype(np.float64)
    d = np.abs(L) @ np.abs(z) + UNDERFLOW * L.shape[0]
    with np.errstate(divide='ignore', invalid='ignore'):
        q = np.where(r == 0, 0.0, r / d)
    return float(q.max()) / EPS
