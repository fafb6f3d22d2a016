"""Accuracy of the batched Cholesky, the log-likelihood path, the batched forward substitution and the aux model against
the extended-precision reference (oracle/xprec.py), on the matrices the sampler visits: K+S at the corners of the bench
bracket (small noise, long length-scales), R + 1e-11 I of aux_var_model (cond ~1e11), a graded D A D and a
well-conditioned control.

Every accuracy check elsewhere is either against the FP64 oracle with a tolerance that grows with cond, a residual on
well-conditioned matrices, or one GPU path against another.  Here each factor's componentwise and normwise backward
error is measured in units of eps = 2^-53 and held to fixed bounds and to a few times LAPACK's on the same FP64 matrix,
and the log-likelihood is held to a few times FP64's own forward error from the longdouble truth.  B200 only; most of the
time is longdouble work on the host."""
import hashlib

import numpy as np
import pytest
import scipy.linalg

from oracle import sds_oracle as so
from oracle import xprec as xp
from test_gpu_band import _run
from test_gpu_band_compact import _band_W, _call, _compact_bytes

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not xp.AVAILABLE, reason=xp.REASON)]

# Bounds in eps = 2^-53, about 2x the worst measured on one B200 (1000 W; test A prints the worst per variant and family
# with its N and matrix): factor componentwise 19.0 (full-inverse panel factor, N=640, R of corner 11/20/0.05) and
# normwise 4.9 (graded, N=127); LAPACK on the same matrices at most 6.4 and 4.0.  The largest ratio to LAPACK, 7.2x, is
# the default path at N=128 on the R of corner 3/4/0.05: one diagonal block, so it comes from the panel factor kernels
# (DESIGN.md section 3).  Without the panel solve's refinement step the factor of R reaches 480 eps.  Border row and
# trsv componentwise 1.75.
FACTOR_COMP, FACTOR_NORM = 40.0, 12.0
VS_LAPACK = 16.0
SOLVE_COMP = 4.0

CORNERS = [(ell, sf, sn) for ell in (3.0, 11.0) for sf in (4.0, 20.0) for sn in (0.05, 0.5)]
WORST, MILD = (11.0, 20.0, 0.05), (3.0, 4.0, 0.5)
DEFAULTS = {0: 4, 1: 0, 2: 0, 3: 0, 4: 0, 9: 0}


def _tag(c):
    return '%g_%g_%g' % c


def _key(*arrays):
    h = hashlib.sha1()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def _ks(n, c):
    x = np.arange(n, dtype=np.float64).reshape(n, 1)
    K = so.cov_matrix(x, np.array(c))
    return K, so.s_diagonal(np.diagonal(K), c[2])


_families = {}


def _family(n):
    """{name: symmetric FP64 matrix} for size n; (b) from every corner up to n = 257, from two above."""
    if n not in _families:
        out = {}
        for c in CORNERS:
            K, S = _ks(n, c)
            out['a:' + _tag(c)] = xp.symmetric(K + np.diag(S))
            if n <= 257 or c in (WORST, MILD):
                out['b:' + _tag(c)] = xp.r_plus_jitter(K, S)
        rs = np.random.RandomState(n)
        M = rs.standard_normal((n, n))
        core = M @ M.T / n + np.eye(n)
        d = np.logspace(-3, 3, n)
        out['c'] = xp.symmetric(d[:, None] * core * d[None, :])
        out['d'] = xp.symmetric(core)
        _families[n] = out
    return _families[n]


_berr = {}


def _backward(A, L):
    k = _key(A, L)
    if k not in _berr:
        _berr[k] = xp.backward_error(A, L)
    return _berr[k]


def _lapack(A):
    k = _key(A, 'lapack')
    if k not in _berr:
        _berr[k] = xp.backward_error(A, scipy.linalg.cholesky(A, lower=True))
    return _berr[k]


def _potrf(gp, mats, tuning=None):
    """Factor the host matrices in one gpmc_potrf_batched call (JITTER_NONE) with the given tuning switches."""
    import torch
    n = mats[0].shape[0]
    ld = n + (n & 1)
    A = np.zeros((len(mats), n, ld))
    A[:, :, :n] = np.stack(mats)
    T = torch.tensor(A, device='cuda')
    try:
        for k, v in (tuning or {}).items():
            gp.ops.set_tuning(k, v)
        info = gp.ops.potrf_batched(T, n=n, jitter_policy=gp.JITTER_NONE).cpu().numpy()
    finally:
        for k in (tuning or {}):
            gp.ops.set_tuning(k, DEFAULTS[k])
    return T.cpu().numpy()[:, :, :n], info


# ------------------------------------------------------------------ A. factor backward error, gpmc_potrf_batched
VARIANTS = {
    'default': {},
    'panel_factor_1': {1: 1}, 'panel_factor_2': {1: 2}, 'panel_factor_3': {1: 3},
    'panel_solve_1': {4: 1},
    'tile_0': {0: 0}, 'tile_1': {0: 1}, 'tile_2': {0: 2}, 'tile_3': {0: 3}, 'tile_5': {0: 5},
    'fused_never': {9: 1}, 'fused_always': {9: 2},
    'lookahead_off': {2: 1}, 'lookahead_on': {2: 2},
    'window_256': {3: 256},
}
SIZES_A = [8, 100, 127, 128, 129, 256, 257, 640, 1000]
REPRESENTATIVE = ['a:' + _tag(WORST), 'a:' + _tag(MILD), 'b:' + _tag(WORST), 'b:' + _tag(MILD), 'c', 'd']


@pytest.mark.parametrize('variant', list(VARIANTS))
def test_factor_backward_error(gp, variant):
    worst = {}
    for n in SIZES_A:
        fam = _family(n)
        names = list(fam) if variant == 'default' else REPRESENTATIVE
        mats = [fam[k] for k in names]
        L, info = _potrf(gp, mats, VARIANTS[variant])
        assert np.all(info == 0), (n, dict(zip(names, info)))
        for b, name in enumerate(names):
            assert not np.triu(L[b], 1).any(), (n, name, 'strict upper triangle not zero')
            comp, norm = _backward(mats[b], L[b])
            lc, ln = _lapack(mats[b])
            # per family: (value, N, matrix) of the worst componentwise, normwise and ratio to LAPACK
            fam_w = worst.setdefault(name[0], [(0.0, 0, ''), (0.0, 0, ''), (0.0, 0, '')])
            for i, v in enumerate((comp, norm, max(comp / max(lc, 1.0), norm / max(ln, 1.0)))):
                fam_w[i] = max(fam_w[i], (v, n, name))
            assert comp <= FACTOR_COMP and norm <= FACTOR_NORM, (variant, n, name, comp, norm, lc, ln)
            assert comp <= VS_LAPACK * max(lc, 1.0) and norm <= VS_LAPACK * max(ln, 1.0), (variant, n, name, comp, norm, lc, ln)
    for f, (c, m, r) in sorted(worst.items()):
        print('A %-15s family %s: worst componentwise %.2f eps (N=%d %s), normwise %.2f eps (N=%d %s), %.2fx LAPACK '
              '(N=%d %s)' % ((variant, f) + c + m + r))


# ------------------------------------------------------------------ B. pivot positions
PANEL_KERNELS = {
    'potf2_reg': {}, 'potf2_full': {1: 1}, 'potf2_lite': {1: 2}, 'potf2_flow': {1: 3},
    'panel_solve_32': {4: 1}, 'fused_reg': {9: 2}, 'fused_flow': {9: 2, 1: 3},
}


@pytest.mark.parametrize('n', [257, 300, 1000])
def test_first_failed_pivot_is_reported_at_its_row(gp, n):
    ks = sorted({k for k in (0, 1, 7, 8, 63, 64, 127, 128, 129, 255, 256, n - 1) if k < n})
    mats = []
    for k in ks:
        rs = np.random.RandomState(1000 + k)
        L0 = np.eye(n) + np.tril(rs.uniform(-1.0, 1.0, (n, n)), -1) / np.sqrt(n)
        d = np.ones(n)
        d[k] = -1e-6
        A = xp.symmetric(L0 @ (d[:, None] * L0.T))
        assert scipy.linalg.lapack.dpotrf(A, lower=1)[1] == k + 1
        mats.append(A)
    for name, tuning in PANEL_KERNELS.items():
        _, info = _potrf(gp, mats, tuning)
        assert list(info) == [k + 1 for k in ks], (name, n, list(info))


@pytest.mark.parametrize('n', [256, 640])
def test_no_spurious_failures_on_r_plus_jitter(gp, n):
    # every R + 1e-11 I that LAPACK factors with a clear margin (smallest pivot^2 >= 1e3 eps max A_ii) factors on the device
    mats = []
    for c in CORNERS:
        A = xp.r_plus_jitter(*_ks(n, c))
        Lr, rinfo = scipy.linalg.lapack.dpotrf(A, lower=1)
        if rinfo == 0 and np.diag(Lr).min() ** 2 >= 1e3 * xp.EPS * np.diag(A).max():
            mats.append(A)
    assert len(mats) >= 4
    for name, tuning in PANEL_KERNELS.items():
        _, info = _potrf(gp, mats, tuning)
        assert np.all(info == 0), (name, n, list(info))


# ------------------------------------------------------------------ C. the log-likelihood path, gpmc_loglik_batched
_truth = {}


def _assembled(gp, x, h):
    """K+S of one item as gpmc_cov_assemble(add_S=True) forms it."""
    n = x.shape[0]
    k = (n, tuple(h))
    if k not in _truth:
        A = xp.symmetric(gp.ops.cov_assemble(x, h[None], add_S=True).cpu().numpy()[0, :, :n])
        _truth[k] = A
    return _truth[k]


def _blocked_chol(A, nb):
    """Left-looking FP64 Cholesky in panels of nb columns on BLAS: the same factor as LAPACK's, summed in another order.
    The panel covers only the rows and columns inside the envelope of A (what it skips is exactly zero)."""
    n = A.shape[0]
    L = np.zeros_like(A)
    env = xp.envelope(A)
    last_row = np.full(n, -1)
    np.maximum.at(last_row, env, np.arange(n))
    last_row = np.maximum.accumulate(last_row)
    for j in range(0, n, nb):
        e = min(n, j + nb)
        r1 = max(e, int(last_row[e - 1]) + 1)
        k0 = min(int(env[j:r1].min()), j)
        P = A[j:r1, j:e] - L[j:r1, k0:j] @ L[j:e, k0:j].T
        L[j:e, j:e] = scipy.linalg.cholesky(P[:e - j], lower=True)
        if e < r1:
            L[e:r1, j:e] = scipy.linalg.solve_triangular(L[j:e, j:e], P[e - j:].T, lower=True).T
    return L


FP64_ORDERS = (None, 8, 32, 128)           # LAPACK, then left-looking panels of 8, 32 and 128 columns


def _loglik_truth(A, g):
    """(longdouble truth, the FP64 log-likelihoods of LAPACK's factor and of blocked factors in FP64_ORDERS)."""
    k = _key(A, g, 'loglik')
    if k not in _truth:
        f64 = []
        for nb in FP64_ORDERS:
            L = scipy.linalg.cholesky(A, lower=True) if nb is None else _blocked_chol(A, nb)
            w = scipy.linalg.solve_triangular(L, g, lower=True)
            f64.append(-(0.5 * w @ w + np.log(np.diag(L)).sum() + 0.5 * A.shape[0] * np.log(2 * np.pi)))
        _truth[k] = (xp.loglik(A, g), f64)
    return _truth[k]


def _items(n, corners, B, seed=7):
    rs = np.random.RandomState(seed + n)
    H = np.array([corners[i % len(corners)] for i in range(B)])
    base = np.array([c[2] * rs.standard_normal(n) for c in corners])
    G = np.array([base[i % len(corners)] for i in range(B)])
    return np.arange(n, dtype=np.float64).reshape(n, 1), G, H


def _forward_errors(gp, x, G, H, ll, distinct):
    """Relative error of every item's ll against the longdouble truth; items repeat with period `distinct`.

    The bound is 8x the worst error FP64 itself makes on the batch: for each item the worst of LAPACK and three blocked
    FP64 factorizations of the same matrix.  Which rounding pattern an ill-conditioned item draws scatters its error by
    10x and more between summation orders (5e-13 to 5e-12 on one K+S at N = 129), so one order alone is not FP64's
    error; a device 10x less accurate than every FP64 order on the batch fails."""
    ref = [_loglik_truth(_assembled(gp, x, H[b]), G[b]) for b in range(distinct)]
    dev = np.array([float(abs((ll[b] - ref[b % distinct][0]) / ref[b % distinct][0])) for b in range(len(ll))])
    fp64 = np.array([max(float(abs((f - truth) / truth)) for f in f64) for truth, f64 in ref])
    bound = max(8 * fp64.max(), 1e-14)
    assert dev.max() <= bound, (int(dev.argmax()), dev.max(), fp64.max())
    return dev.max(), fp64.max()


C_SHAPES = [
    (127, 8), (128, 8), (129, 16), (257, 8),     # look-ahead (few matrices), no window
    (257, 160),                                  # plain left-looking
    (641, 8), (1000, 8),                         # windows of 512 + look-ahead
    (641, 200), (1000, 160),                     # plain left-looking
]


@pytest.mark.parametrize('n,B', C_SHAPES)
def test_loglik_factor_border_row_and_value(gp, n, B):
    x, G, H = _items(n, CORNERS, B)
    res = {}
    for env, band in ((0, 0), (1, 0), (1, 1)):
        out = _run(gp, x, G, H, dense=not env, band=bool(band))
        assert np.all(out['info'] == 0)
        w = [0.0] * 4
        for b in range(len(CORNERS)):
            A = _assembled(gp, x, H[b])
            L, z, ll = out['L'][b], out['z'][b], out['ll'][b]
            comp, norm = _backward(A, L)
            lc, ln = _lapack(A)
            assert comp <= FACTOR_COMP and norm <= FACTOR_NORM, (env, band, b, comp, norm)
            assert comp <= VS_LAPACK * max(lc, 1.0) and norm <= VS_LAPACK * max(ln, 1.0), (env, band, b, comp, norm, lc, ln)
            sb = xp.solve_backward_error(L, G[b], z)
            assert sb <= SOLVE_COMP, (env, band, b, sb)
            # the quadratic form and log-determinant reduction on their own: the value of the factor the device holds
            zl, dl = z.astype(xp.LD), np.log(np.diagonal(L).astype(xp.LD))
            scale = float(np.dot(zl, zl) / 2 + np.abs(dl).sum() + n * xp.LOG_2PI / 2)
            red = float(abs(ll - xp.loglik_of_factor(L, z))) / (n * xp.EPS * scale)
            assert red <= 1.0, (env, band, b, red)
            w = [max(w[0], comp), max(w[1], norm), max(w[2], sb), max(w[3], red)]
        fwd, lap = _forward_errors(gp, x, G, H, out['ll'], len(CORNERS))
        res[(env, band)] = out
        print('C n=%d B=%d env=%d band=%d: factor %.2f / %.2f eps, border row %.2f eps, reduction %.3f N eps, '
              'forward %.2e (worst FP64 order %.2e)' % (n, B, env, band, w[0], w[1], w[2], w[3], fwd, lap))
    # copies of an item anywhere in the batch are factored alike
    for b in range(len(CORNERS), B):
        assert res[(1, 1)]['ll'][b] == res[(1, 1)]['ll'][b % len(CORNERS)]


N_BIG = 4096
BIG_CORNERS = [(3.0, 4.0, 0.5), (3.0, 20.0, 0.05), (11.0, 4.0, 0.5), (11.0, 20.0, 0.05)]


def test_loglik_n4096_banded_residual(gp):
    # one wave, windows + look-ahead; the residual is formed inside the band of K+S only
    x, G, H = _items(N_BIG, BIG_CORNERS, 8)
    out = _run(gp, x, G, H)
    assert np.all(out['info'] == 0)
    for b in range(len(BIG_CORNERS)):
        A = _assembled(gp, x, H[b])
        assert xp.envelope(A).max() > 0
        comp, norm = _backward(A, out['L'][b])
        sb = xp.solve_backward_error(out['L'][b], G[b], out['z'][b])
        print('C n=4096 %s: factor %.2f / %.2f eps, border row %.2f eps' % (_tag(tuple(H[b])), comp, norm, sb))
        assert comp <= FACTOR_COMP and norm <= FACTOR_NORM and sb <= SOLVE_COMP
    fwd, lap = _forward_errors(gp, x, G, H, out['ll'], len(BIG_CORNERS))
    print('C n=4096 one wave: forward %.2e (worst FP64 order %.2e)' % (fwd, lap))


@pytest.mark.parametrize('compact', [1, 0])
def test_loglik_n4096_compact_waves_forward_error(gp, compact):
    # waves of 80 items run the plain left-looking schedule on compact rows (key 17 on) or the dense layout in many waves
    B, wave = 160, 80
    x, G, H = _items(N_BIG, BIG_CORNERS, B)
    W = _band_W(x, H)
    ll, info, (Wg, waves) = _call(gp, x, G, H, _compact_bytes(N_BIG, B, wave, W), compact=bool(compact))
    assert np.all(info == 0)
    assert (Wg, waves) == ((W, 2) if compact else (0, waves)) and waves > 1
    fwd, lap = _forward_errors(gp, x, G, H, ll, len(BIG_CORNERS))
    print('C n=4096 B=%d compact=%d (%d waves): forward %.2e (worst FP64 order %.2e)' % (B, compact, waves, fwd, lap))


# ------------------------------------------------------------------ D. gpmc_trsv_lower_batched
@pytest.mark.parametrize('n', [256, 1024])
def test_trsv_on_ill_conditioned_factor(gp, n):
    A = xp.r_plus_jitter(*_ks(n, WORST))
    L = scipy.linalg.cholesky(A, lower=True)
    rs = np.random.RandomState(n)
    rhs = rs.standard_normal((6, n)) * np.logspace(-3, 3, 6)[:, None]
    z, quad = gp.ops.trsv_lower(L, rhs, want_lognormal=True)
    z, quad = z.cpu().numpy(), quad.cpu().numpy()
    worst = 0.0
    for b in range(len(rhs)):
        sb = xp.solve_backward_error(L, rhs[b], z[b])
        worst = max(worst, sb)
        assert sb <= SOLVE_COMP, (b, sb)
        zl, dl = z[b].astype(xp.LD), np.log(np.diagonal(L).astype(xp.LD))
        scale = float(np.dot(zl, zl) / 2 + np.abs(dl).sum() + n * xp.LOG_2PI / 2)
        assert abs(quad[b] - xp.loglik_of_factor(L, z[b])) <= n * xp.EPS * scale
    print('D n=%d cond(L) %.1e: solve backward error %.2f eps' % (n, np.linalg.cond(L), worst))


# ------------------------------------------------------------------ E. gpmc_aux_var_model
@pytest.mark.parametrize('n', [256, 640])
@pytest.mark.parametrize('corner', [WORST, MILD])
def test_aux_var_model_against_true_r(gp, n, corner):
    K, S = _ks(n, corner)
    g = np.sqrt(S) * np.random.RandomState(n).standard_normal(n)
    L, m, C, info = gp.ops.aux_var_model_device(K, S, g)
    L, m, C, info = L.cpu().numpy(), m.cpu().numpy(), C.cpu().numpy(), info.cpu().numpy()
    assert np.all(info == 0)
    comp, norm = _backward(xp.symmetric(K + np.diag(S)), L)
    assert comp <= FACTOR_COMP and norm <= FACTOR_NORM, (comp, norm)
    R = xp.r_matrix(K, S)
    m_true = np.dot(R, g.astype(xp.LD) / S.astype(xp.LD))
    jit = xp.LD(1e-11) * np.eye(n, dtype=xp.LD)

    def r_err(Cf):
        Cl = Cf.astype(xp.LD)
        return float(np.linalg.norm((xp._mm(Cl, Cl.T) - jit - R).astype(np.float64)) / np.linalg.norm(R.astype(np.float64)))

    def m_err(mf):
        return float(np.linalg.norm((mf - m_true).astype(np.float64)) / np.linalg.norm(m_true.astype(np.float64)))

    _, _, m_or, C_or, _ = so.aux_var_model(None, K, corner[2], g=g, r_form='reduced')
    dr, orr = r_err(C), r_err(C_or)
    dm, orm = m_err(m), m_err(m_or)
    print('E n=%d %s: L %.2f / %.2f eps; R rel err %.2e (oracle %.2e); m rel err %.2e (oracle %.2e)'
          % (n, _tag(corner), comp, norm, dr, orr, dm, orm))
    assert dr <= 8 * orr + 1e-15
    assert dm <= 8 * orm + 1e-15
