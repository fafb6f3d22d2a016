"""Compact band storage of the batched log-likelihood (gpmc_set_tuning(17, .)): bit-identical to the dense path.

When the dense layout would need several waves, gpmc_loglik_batched bounds the band of every item of the call and, if
rows W = 128 + 64 * (widest band) columns wide need fewer waves that run the plain left-looking schedule, stores only
those columns of each row (the border row in an array of its own).  Every run here hands the library exactly the bytes
it is given, filled with NaN, between two guard regions that must stay untouched; results are compared bit for bit with
the dense path run in one wave on a workspace large enough for the whole batch.  B200 only."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ENV_ROWS, NB = 64, 128
GUARD = 1 << 20


def _a(v):
    return (v + 255) // 256 * 256


def _band_W(x, H):
    """Row width of the compact layout, from the band bound of cov_assemble.cu (1-D x, isotropic kernel)."""
    x = np.asarray(x, dtype=np.float64)[:, 0]
    N = x.shape[0]
    nblk = (N + ENV_ROWS - 1) // ENV_ROWS
    bl = np.array([x[r * ENV_ROWS:(r + 1) * ENV_ROWS].min() for r in range(nblk)])
    bh = np.array([x[r * ENV_ROWS:(r + 1) * ENV_ROWS].max() for r in range(nblk)])
    width = 0
    for h in H:
        ell, sf2 = np.exp(np.log(h[0])), np.exp(2.0 * np.log(h[1]))
        if not (np.isfinite(sf2) and sf2 > 0 and np.isfinite(ell) and ell > 0 and np.isfinite(x).all()):
            width = nblk - 1
            continue
        thr = 760.0 + max(0.0, np.log(sf2))
        lo = np.arange(nblk)
        for r in range(nblk):
            for c in range(r):
                g = max(0.0, bl[r] / ell - bh[c] / ell, bl[c] / ell - bh[r] / ell)
                if not (0.5 * (g * g) * (1.0 - 1e-9) > thr):
                    lo[r] = c
                    break
        w = np.array([min(lo[max(r - 1, 0)], lo[r], lo[min(r + 1, nblk - 1)]) // (NB // ENV_ROWS) * (NB // ENV_ROWS)
                      for r in range(nblk)])
        width = max(width, int((np.arange(nblk) - w).max()))
    return (NB + ENV_ROWS * width + 15) // 16 * 16


def _compact_bytes(N, B, wave, W):
    """Workspace bytes that hold waves of `wave` items in the compact layout of width W (capi.cu's carving)."""
    ld = (N + 15) // 16 * 16
    nblk = (N + ENV_ROWS - 1) // ENV_ROWS
    fixed = _a(B * 8) + _a(B * 4) + 256 + _a(32 * ld * 8)
    return fixed + 2 * _a(B * nblk * 4) + 256 + wave * (N * W * 8 + ld * 8 + NB * NB * 8)


def _call(gp, x, G, H, nbytes, compact=True):
    """loglik, info and (band_W, waves) of one gpmc_loglik_batched call on a NaN-filled workspace of exactly nbytes."""
    import torch
    lib = gp._lib.load()
    xd = torch.tensor(np.asarray(x, dtype=np.float64)).cuda()
    Gd, Hd = torch.tensor(G).cuda(), torch.tensor(H).cuda()
    B, N = G.shape
    D, P = xd.shape[1], Hd.shape[1]
    raw = torch.full((nbytes + 2 * GUARD,), 0xA5, dtype=torch.uint8, device='cuda')
    raw[GUARD:GUARD + nbytes] = 0xFF                   # NaN
    ll = torch.empty(B, dtype=torch.float64, device='cuda')
    info = torch.empty(B, dtype=torch.int32, device='cuda')
    gp.ops.set_tuning(17, 1 if compact else 0)
    try:
        rc = lib.gpmc_loglik_batched(xd.data_ptr(), N, D, Gd.data_ptr(), Hd.data_ptr(), B, P, gp.ops.kind_of(D, P),
                                     gp.ops.JITTER_PYGPS, ll.data_ptr(), info.data_ptr(), raw.data_ptr() + GUARD, nbytes,
                                     ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
        gp._lib.check(rc, 'gpmc_loglik_batched')
        torch.cuda.synchronize()
        W, waves = ctypes.c_int(-1), ctypes.c_int(-1)
        gp._lib.check(lib.gpmc_loglik_layout(ctypes.byref(W), ctypes.byref(waves)), 'gpmc_loglik_layout')
    finally:
        gp.ops.set_tuning(17, 1)
    assert bool((raw[:GUARD] == 0xA5).all().item()), 'bytes BEFORE the workspace were written'
    assert bool((raw[GUARD + nbytes:] == 0xA5).all().item()), 'bytes AFTER the workspace were written'
    return ll.cpu().numpy(), info.cpu().numpy(), (W.value, waves.value)


def _reference(gp, x, G, H):
    lib = gp._lib.load()
    B, N = G.shape
    ll, info, (W, waves) = _call(gp, x, G, H, lib.gpmc_workspace_bytes(gp._lib.OP_LOGLIK, N, np.asarray(x).shape[1], B),
                                 compact=False)
    assert (W, waves) == (0, 1)
    return ll, info


def _same(a, b):
    return np.array_equal(np.asarray(a).view(np.int64), np.asarray(b).view(np.int64))


def _dense_waves(gp, N, D, B, nbytes):
    lib = gp._lib.load()
    one = lib.gpmc_workspace_bytes(gp._lib.OP_LOGLIK, N, D, 1)
    per = lib.gpmc_workspace_bytes(gp._lib.OP_LOGLIK, N, D, 2) - one
    wave = min(B, (nbytes - (one - per)) // per)
    return -(-B // wave)


def _check_compact(gp, x, G, H, wave):
    """Compact run in waves of `wave` items against the one-wave dense reference."""
    B, N = G.shape
    W = _band_W(x, H)
    nbytes = _compact_bytes(N, B, wave, W)
    ref_ll, ref_info = _reference(gp, x, G, H)
    ll, info, layout = _call(gp, x, G, H, nbytes)
    assert layout == (W, -(-B // wave)), (layout, W)
    assert layout[1] < _dense_waves(gp, N, 1, B, nbytes)
    assert np.array_equal(info, ref_info)
    assert _same(ll, ref_ll)
    return info


def _batch(gp, n, B, seed):
    G, H = gp.synthetic.loglik_batch(B, n, seed=seed)
    return np.arange(n, dtype=np.float64).reshape(n, 1), G, H


@pytest.mark.parametrize('n,B,wave', [
    (4096, 96, 96),       # the bench shape: one compact wave where the dense layout needs several
    (1000, 160, 160),     # matrix edge off the 128 grid
    (777, 200, 200),      # band edges and the matrix edge off the 64 / 128 grid
    (1000, 400, 200),     # the compact layout needs several waves too
])
def test_compact_matches_dense(gp, n, B, wave):
    x, G, H = _batch(gp, n, B, seed=3000 + n)
    _check_compact(gp, x, G, H, wave)


def test_compact_jitter_ladder(gp):
    # failing first attempts are re-assembled in place through the item map, inside the same compact rows
    x, G, H = _batch(gp, 1000, 160, seed=3100)
    H[0::7, 2] = 1e-9
    H[0::7, 0] = np.linspace(4.0, 12.0, len(H[0::7]))
    _check_compact(gp, x, G, H, 160)


def _check_dense_fallback(gp, x, G, H, nbytes):
    # the call runs exactly the dense path of the same workspace (its waves, and with them its schedules)
    B, N = G.shape
    ll, info, (W, waves) = _call(gp, x, G, H, nbytes)
    ref_ll, ref_info, ref_layout = _call(gp, x, G, H, nbytes, compact=False)
    assert (W, waves) == ref_layout == (0, _dense_waves(gp, N, np.asarray(x).shape[1], B, nbytes))
    assert waves > 1
    assert np.array_equal(info, ref_info)
    assert _same(ll, ref_ll)
    return info


def test_wide_items_fall_back_to_dense(gp):
    # one item whose band is the whole triangle (NaN length-scale, sf = 0, a huge length-scale) makes W = ld: dense
    n, B = 1000, 160
    for col, v in ((0, np.nan), (1, 0.0), (0, 1e3)):
        x, G, H = _batch(gp, n, B, seed=3200)
        H[5, col] = v
        info = _check_dense_fallback(gp, x, G, H, _compact_bytes(n, B, B, 704))
        assert info[5] != 0 or col == 0


def test_ard_stays_dense(gp):
    # inputs scattered in every dimension: no tile of K+S is certainly zero, the band is the whole triangle
    rs = np.random.RandomState(12)
    n, B = 1000, 160
    x = rs.uniform(0.0, 3.0, size=(n, 3))
    H = np.column_stack([rs.uniform(0.5, 4.0, size=(B, 3)), rs.uniform(1.0, 3.0, size=B), rs.uniform(0.3, 1.0, size=B)])
    G = rs.standard_normal((B, n))
    _check_dense_fallback(gp, x, G, H, _compact_bytes(n, B, B, 704))


def test_key17_off_is_the_dense_path(gp):
    x, G, H = _batch(gp, 1000, 160, seed=3300)
    nbytes = _compact_bytes(1000, 160, 160, _band_W(x, H))
    ref_ll, ref_info = _reference(gp, x, G, H)
    ll, info, (W, waves) = _call(gp, x, G, H, nbytes, compact=False)
    assert W == 0 and waves == _dense_waves(gp, 1000, 1, 160, nbytes) > 1
    assert np.array_equal(info, ref_info)
    assert _same(ll, ref_ll)
