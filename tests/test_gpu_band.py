"""Band-only assembly and launches of the batched log-likelihood (gpmc_set_tuning(15, .)): bit-identical to the dense path.

A bound taken before the assembly gives, per item and 64-row block, the first 64-column tile that can hold a nonzero of
K+S.  Only the band right of it is assembled, the update GEMM and the panel solve launch only the band's rows, and the
region left of the band is cleared inline in the assembly (gpmc_set_tuning(16, 2)), on a side stream (16, 1) or not at
all (16, 0).  Every band run starts from a workspace filled with NaN: an element read outside the band would reach the
outputs.  B200 only."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ENV_ROWS = 64


def _layout(N, B):
    """Byte offsets of the matrices, the envelope and the band starts w in gpmc_loglik_batched's workspace for a wave of B
    items (capi.cu: loglik_layout and the carving of the workspace)."""
    a = lambda v: (v + 255) // 256 * 256
    ld = (N + 15) // 16 * 16
    nblk = (N + ENV_ROWS - 1) // ENV_ROWS
    fixed = a(B * 8) + a(B * 4) + 256 + a(32 * ld * 8)
    off_env = fixed + B * (N + 1) * ld * 8 + B * 128 * 128 * 8
    return ld, nblk, fixed, off_env, off_env + B * nblk * 4


def _run(gp, x, G, H, dense=False, band=True, clear=2, wave=None, poison=True):
    """loglik, info and -- for a single wave -- the factored lower triangle, the border row, the envelope and w."""
    import torch
    lib = gp._lib.load()
    B, N = G.shape
    wave = B if wave is None else wave
    gp.ops.set_tuning(14, 0 if dense else 1)
    gp.ops.set_tuning(15, 1 if band else 0)
    gp.ops.set_tuning(16, clear)
    try:
        ws = gp.ops.Workspace()
        nbytes = lib.gpmc_workspace_bytes(gp._lib.OP_LOGLIK, N, np.asarray(x).shape[1], min(B, wave))
        ws.buf = torch.full((nbytes,), 0xFF if poison else 0, dtype=torch.uint8, device='cuda')
        ll, info = gp.ops.loglik_batched(x, G, H, workspace=ws, max_wave=wave)
        torch.cuda.synchronize()
        out = {'ll': ll.cpu().numpy(), 'info': info.cpu().numpy()}
        if wave >= B:
            ld, nblk, off_mat, off_env, off_w = _layout(N, B)
            buf = ws.buf.cpu().numpy()
            mats = buf[off_mat:off_mat + B * (N + 1) * ld * 8].view(np.float64).reshape(B, N + 1, ld)
            out['L'] = np.tril(mats[:, :N, :N])
            out['z'] = mats[:, N, :N].copy()
            out['env'] = buf[off_env:off_env + B * nblk * 4].view(np.int32).reshape(B, nblk).astype(np.int64)
            out['w'] = buf[off_w:off_w + B * nblk * 4].view(np.int32).reshape(B, nblk).astype(np.int64)
        return out
    finally:
        gp.ops.set_tuning(14, 1)
        gp.ops.set_tuning(15, 1)
        gp.ops.set_tuning(16, 2)


def _in_band(w, N):
    """[B, N, N] mask of the elements the band assembly writes (lower triangle from 64 w[r] on)."""
    cols = np.arange(N)
    first = np.repeat(w * ENV_ROWS, ENV_ROWS, axis=1)[:, :N]
    return (cols[None, None, :] >= first[:, :, None]) & (cols[None, None, :] <= cols[None, :, None])


def _same(a, b):
    """Bitwise equality of float arrays (NaN == NaN in the same places)."""
    return np.array_equal(np.asarray(a).view(np.int64), np.asarray(b).view(np.int64))


def _check(gp, x, G, H, clear=2, wave=None):
    ref = _run(gp, x, G, H, dense=True, poison=False, wave=wave)
    got = _run(gp, x, G, H, clear=clear, wave=wave)
    assert np.array_equal(got['info'], ref['info'])
    assert _same(got['ll'], ref['ll'])
    if 'L' not in got:
        return got
    ok = ref['info'] == 0
    assert _same(got['z'][ok], ref['z'][ok])
    if clear:
        assert _same(got['L'][ok], ref['L'][ok])
    else:
        # nothing cleared: left of the band the poison stays; inside it the factor is the dense one
        m = _in_band(got['w'], G.shape[1])[ok]
        assert _same(got['L'][ok][m], ref['L'][ok][m])
    # every nonzero lies in the band
    env = got['env']
    assert (got['w'] * ENV_ROWS <= env).all()
    return got


def _batch(gp, n, B, ell=None, seed=2000):
    G, H = gp.synthetic.loglik_batch(B, n, seed=seed)
    if ell is not None:
        H[:, 0] = ell
    return np.arange(n, dtype=np.float64).reshape(n, 1), G, H


@pytest.mark.parametrize('clear', [2, 1, 0])
def test_band_poisoned_workspace_matches_dense(gp, clear):
    x, G, H = _batch(gp, 2048, 48, seed=2300)
    got = _check(gp, x, G, H, clear=clear)
    assert (got['w'] > 0).any()                 # the case leaves part of the triangle out of the band


@pytest.mark.parametrize('n,B', [
    (1000, 160),      # plain left-looking schedule, many matrices per launch
    (4096, 8),        # windows + look-ahead streams, split in-window updates
    (3000, 2),        # windowed, ragged last block column
    (2500, 1),        # single matrix
    (777, 96),        # band edges and the matrix edge off the 64 / 128 grid
])
def test_band_schedules(gp, n, B):
    x, G, H = _batch(gp, n, B)
    _check(gp, x, G, H)


def _cases(gp):
    rs = np.random.RandomState(11)
    out = {'bench': _batch(gp, 4096, 16, seed=2400)}
    for ell in (0.05, 29.0):
        out['ell_%g' % ell] = _batch(gp, 1100, 8, ell=ell, seed=2500)
    x, G, H = _batch(gp, 1100, 8, seed=2600)
    out['shuffled'] = (x[rs.permutation(x.shape[0])], G, H)
    n, B = 900, 8
    xa = np.column_stack([np.arange(n, dtype=np.float64), rs.uniform(0.0, 3.0, size=(n, 3))])
    Ha = np.column_stack([rs.uniform(0.5, 4.0, size=(B, 4)), rs.uniform(1.0, 3.0, size=B), rs.uniform(0.3, 1.0, size=B)])
    out['ard4'] = (xa, rs.standard_normal((B, n)), Ha)
    x, G, H = _batch(gp, 1100, 8, seed=2700)
    H[1, 1] = 0.0                               # sf = 0
    H[2, 0] = np.nan                            # a NaN length-scale
    H[3, 0] = 1e3                               # one dense item among narrow ones
    out['odd_items'] = (x, G, H)
    return out


@pytest.mark.parametrize('case', ['bench', 'ell_0.05', 'ell_29', 'shuffled', 'ard4', 'odd_items'])
def test_band_bound_is_conservative(gp, case):
    x, G, H = _cases(gp)[case]
    got = _check(gp, x, G, H)
    # against the envelope of a full assembly too (the band run's envelope comes from the band tiles alone)
    full = _run(gp, x, G, H, band=False, poison=False)
    assert np.array_equal(got['env'], full['env'])
    assert (got['w'] * ENV_ROWS <= full['env']).all()
    if case == 'odd_items':
        assert (got['w'][[1, 2, 3]] == 0).all()


def test_band_jitter_ladder_and_failures(gp):
    # the ladder re-assembles the failing items inside the same band; sf = 0 gives NaN on the diagonal: not PD
    n, B = 900, 12
    x, G, H = _batch(gp, n, B, seed=2200)
    H[0::3, 2] = 1e-9
    H[0::3, 0] = [6.0, 9.0, 12.0, 4.0]
    H[1, 1] = 0.0
    got = _check(gp, x, G, H)
    assert (got['info'] != 0).any()
    _check(gp, x, G, H, clear=1)                # the side-stream clear runs before the failed attempt's kernels


def test_band_several_waves(gp):
    # a wide wave (long length-scales) followed by narrow ones: each wave sizes its own launches, and the clear of one wave
    # finishes before the next one assembles into the same buffers
    n, B = 1500, 30
    x, G, H = _batch(gp, n, B, seed=2800)
    H[:10, 0] = np.linspace(20.0, 30.0, 10)
    H[10:, 0] = np.linspace(0.1, 2.0, 20)
    _check(gp, x, G, H, wave=10)
    _check(gp, x, G, H, wave=7)


@pytest.mark.parametrize('key,value', [(0, 0), (0, 5), (4, 1)])
def test_band_off_with_kernels_that_read_whole_rows(gp, key, value):
    # the cp.async / persistent tile kernels and the 32-column panel solve do not start at the envelope: the band must not
    # be used with them (it would leave elements they read unwritten); results stay those of the dense path
    x, G, H = _batch(gp, 1000, 24, seed=2900)
    gp.ops.set_tuning(key, value)
    try:
        got = _run(gp, x, G, H)
        ref = _run(gp, x, G, H, dense=True, poison=False)
    finally:
        gp.ops.set_tuning(key, 4 if key == 0 else 0)
    assert np.array_equal(got['info'], ref['info'])
    assert np.allclose(got['ll'], ref['ll'], rtol=1e-12, atol=0.0)
