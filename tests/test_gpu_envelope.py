"""Envelope skips of the batched log-likelihood (gpmc_set_tuning(14, .)): bit-identical to the dense path.

The assembly records, per 64-row block of K+S, the first column holding a nonzero; the update GEMM and the panel solve
skip the products that envelope shows to be exact zeros.  Every case runs with the skips on and forced off and requires
equal loglik, info, factor L and border row z = L^-1 g.  B200 only."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ENV_ROWS = 64


def _layout(N, B):
    """Byte offsets of the matrices and the envelope in gpmc_loglik_batched's workspace for a wave of all B items
    (capi.cu: loglik_layout and the carving of the workspace)."""
    a = lambda v: (v + 255) // 256 * 256
    ld = (N + 15) // 16 * 16
    fixed = a(B * 8) + a(B * 4) + 256 + a(32 * ld * 8)
    mat = (N + 1) * ld * 8
    return ld, fixed, fixed + B * mat + B * 128 * 128 * 8


def _run(gp, x, G, H, on):
    """loglik, info, the factored matrices (lower triangle + border row) and the envelope of one envelope mode."""
    import torch
    gp.ops.set_tuning(14, 1 if on else 0)
    try:
        ws = gp.ops.Workspace()
        B, N = G.shape
        ll, info = gp.ops.loglik_batched(x, G, H, workspace=ws, max_wave=B)
        torch.cuda.synchronize()
        ld, off_mat, off_env = _layout(N, B)
        buf = ws.buf.cpu().numpy()
        mats = buf[off_mat:off_mat + B * (N + 1) * ld * 8].view(np.float64).reshape(B, N + 1, ld)
        L = np.tril(mats[:, :N, :N])
        z = mats[:, N, :N].copy()
        nblk = (N + ENV_ROWS - 1) // ENV_ROWS
        env = buf[off_env:off_env + B * nblk * 4].view(np.int32).reshape(B, nblk).copy() if on else None
        return ll.cpu().numpy(), info.cpu().numpy(), L, z, env
    finally:
        gp.ops.set_tuning(14, 1)


def _host_envelope(gp, x, H):
    """First column holding a nonzero in each 64-row block of the lower triangle of K+S as the device assembles it."""
    A = gp.ops.cov_assemble(x, H, add_S=True, lower_only=True).cpu().numpy()
    N = A.shape[1]
    nz = np.tril(A[:, :, :N] != 0)
    nblk = (N + ENV_ROWS - 1) // ENV_ROWS
    env = np.full((A.shape[0], nblk), np.iinfo(np.int32).max, dtype=np.int64)
    for r in range(nblk):
        blk = nz[:, r * ENV_ROWS:(r + 1) * ENV_ROWS, :].any(axis=1)
        has = blk.any(axis=1)
        env[has, r] = blk[has].argmax(axis=1)
    return env


def _check(gp, x, G, H, expect_skips=True, fused=False):
    ll1, info1, L1, z1, env = _run(gp, x, G, H, True)
    ll0, info0, L0, z0, _ = _run(gp, x, G, H, False)
    assert np.array_equal(info1, info0)
    ok = info0 == 0
    assert np.array_equal(ll1[ok], ll0[ok])
    assert np.array_equal(np.isnan(ll1), np.isnan(ll0))
    assert np.array_equal(L1[ok], L0[ok])
    assert np.array_equal(z1[ok], z0[ok])
    if fused:                  # fused panel launches: the log-lik path records no envelope and factors densely
        return None
    host = _host_envelope(gp, x, H)
    assert np.array_equal(env, host)
    if expect_skips:           # the case exercises the skips: some row block is zero in a whole 128-column block column
        assert (env[ok] >= 128).any()
    return env


def _batch(gp, n, B, ell=None, seed=2000):
    G, H = gp.synthetic.loglik_batch(B, n, seed=seed)
    if ell is not None:
        H[:, 0] = ell
    return np.arange(n, dtype=np.float64).reshape(n, 1), G, H


@pytest.mark.parametrize('n,B', [
    (1000, 160),      # plain left-looking schedule, many matrices per launch
    (4096, 8),        # windows + look-ahead streams, split in-window updates
    (3000, 2),        # windowed, ragged last block column
    (2500, 1),        # single matrix
    (512, 700),       # fused panel factor + solve launches: dense either way
    (777, 96),        # band edges and the matrix edge off the 64 / 128 grid
])
def test_envelope_matches_dense(gp, n, B):
    x, G, H = _batch(gp, n, B)
    _check(gp, x, G, H, expect_skips=n >= 700, fused=n < 640)


@pytest.mark.parametrize('ell', [0.05, 1.7, 13.3, 29.0])
def test_envelope_band_widths(gp, ell):
    # ell = 0.05: K+S is tridiagonal (exp(-200) is a normal double, exp(-800) underflows), every block's envelope is the
    # row above it; larger ell: band edges at about 38.6 ell rows, off the 64-row grid
    x, G, H = _batch(gp, 1100, 24, ell=ell, seed=2100)
    env = _check(gp, x, G, H, expect_skips=ell < 20)
    if ell == 0.05:
        assert np.array_equal(env, np.tile(np.maximum(np.arange(env.shape[1]) * ENV_ROWS - 1, 0), (env.shape[0], 1)))


def test_envelope_ard_is_dense(gp):
    # ARD D=4 over a small box: no entry underflows, so the envelope is 0 everywhere and nothing is skipped
    rs = np.random.RandomState(7)
    n, B = 700, 48
    x = rs.uniform(0.0, 3.0, size=(n, 4))
    H = np.column_stack([rs.uniform(1.0, 4.0, size=(B, 4)), rs.uniform(1.0, 3.0, size=B), rs.uniform(0.3, 1.0, size=B)])
    G = rs.standard_normal((B, n))
    env = _check(gp, x, G, H, expect_skips=False)
    assert (env == 0).all()


def test_envelope_jitter_ladder_and_failures(gp):
    # sn = 1e-9 and long length-scales: K+S is numerically singular, the plain attempt fails and the jitter ladder
    # re-assembles those items (recomputing their envelope); sf = 0 gives NaN on the diagonal: not PD
    n, B = 900, 12
    x, G, H = _batch(gp, n, B, seed=2200)
    H[0::3, 2] = 1e-9
    H[0::3, 0] = [6.0, 9.0, 12.0, 4.0]
    H[1, 1] = 0.0
    _, info, _, _, _ = _run(gp, x, G, H, True)
    assert (info != 0).any()
    _check(gp, x, G, H, expect_skips=False)
