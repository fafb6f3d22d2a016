"""Fused panel launches of the compact band layout: the panel factor and the band-limited panel solve of a block column in
one launch per chain (default), or in two launches (gpmc_set_tuning(9, 1)).  Both are bit-identical to the dense path run
in one wave.  B200 only."""
import numpy as np
import pytest

from test_gpu_band_compact import NB, _band_W, _batch, _call, _check_compact, _compact_bytes

pytestmark = pytest.mark.gpu


# The compact layout runs the panel factor and the panel solve of a block column in one launch (one CTA per chain) unless
# gpmc_set_tuning(9, 1) forbids fused panels; both must give the dense path's bits.
def _with_key9(gp, value, fn):
    gp.ops.set_tuning(9, value)
    try:
        return fn()
    finally:
        gp.ops.set_tuning(9, 0)


@pytest.mark.parametrize('key9', [0, 1])
@pytest.mark.parametrize('n,B,wave', [(4096, 96, 96), (1000, 160, 160), (777, 200, 200), (1000, 400, 200)])
def test_compact_fused_and_separate_panels_match_dense(gp, key9, n, B, wave):
    x, G, H = _batch(gp, n, B, seed=3000 + n)
    _with_key9(gp, key9, lambda: _check_compact(gp, x, G, H, wave))


@pytest.mark.parametrize('key9', [0, 1])
def test_compact_fused_and_separate_panels_jitter_ladder(gp, key9):
    x, G, H = _batch(gp, 1000, 160, seed=3100)
    H[0::7, 2] = 1e-9
    H[0::7, 0] = np.linspace(4.0, 12.0, len(H[0::7]))
    _with_key9(gp, key9, lambda: _check_compact(gp, x, G, H, 160))


@pytest.mark.parametrize('key9', [0, 1])
def test_compact_sub_block_skip_off_grid(gp, key9):
    # short length-scales start the envelope of a row block deep inside the block column (the fused solve starts its chain
    # at the first 8-column sub-block that can hold a nonzero), mixed with longer ones that widen the band; the band's last
    # row block and the matrix edge (777) are off the 64 grid
    x, G, H = _batch(gp, 777, 200, seed=3400)
    H[:, 0] = np.where(np.arange(200) % 3 == 0, np.linspace(0.3, 1.5, 200), np.linspace(2.0, 8.0, 200))
    info = _with_key9(gp, key9, lambda: _check_compact(gp, x, G, H, 200))
    assert np.all(info == 0)


def test_compact_default_makes_no_panel_trsm_launch(gp):
    x, G, H = _batch(gp, 1000, 160, seed=3500)
    nbytes = _compact_bytes(1000, 160, 160, _band_W(x, H))
    gp.ops.profile(True)
    try:
        _, info, (W, waves) = _call(gp, x, G, H, nbytes)
        prof = gp.ops.profile_read()
    finally:
        gp.ops.profile(False)
    assert W > 0 and waves == 1 and np.all(info == 0)
    assert prof['panel_trsm'][1] == 0, prof
    assert prof['potf2'][1] == -(-1000 // NB), prof
