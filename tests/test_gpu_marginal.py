"""gpmc_marginal_run (slice sampling of the hyper-parameters with f integrated out) against oracle/marginal_oracle.py:
tape parity, Philox determinism, the posterior, failure handling, argument checks and the Python layers above it."""
import ctypes

import numpy as np
import pytest

from oracle import marginal_oracle as mo
from oracle import matern_oracle
from oracle import sds_oracle as so

pytestmark = pytest.mark.gpu


def tapes(B, n_iters, P, T, seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(size=(B, n_iters, P)), rng.uniform(size=(B, n_iters)), rng.uniform(size=(B, n_iters, T, P))


def run(gp, x, y, H0, scale, it0, n_iters, **kw):
    import torch
    H = torch.tensor(np.ascontiguousarray(H0, dtype=np.float64)).cuda()
    hh, ll, tt, ex = gp.ops.marginal_run(x, y, H, scale, it0, n_iters, **kw)
    return hh.cpu().numpy(), ll.cpu().numpy(), tt.cpu().numpy(), ex.cpu().numpy(), H.cpu().numpy()


def oracle_chains(x, y, H0, scale, it0, n_iters, burn_in, tape, d=None, **kw):
    from contextlib import nullcontext
    out = []
    with (matern_oracle.kernel(d) if d else nullcontext()):
        for b in range(H0.shape[0]):
            out.append(mo.run_chain(x, y, H0[b], scale, it0, n_iters, burn_in, tape.v[b], tape.u0[b], tape.U[b], **kw))
    return out


def assert_parity(x, y, dev, ref, d=None):
    hh, ll, tt, ex, H = dev
    r = y - np.mean(y)
    for b, (rh, rl, rt, re) in enumerate(ref):
        assert np.array_equal(hh[b], rh), (b, np.flatnonzero((hh[b] != rh).any(axis=1))[:3])
        assert np.array_equal(tt[b], rt) and ex[b] == re, (b, tt[b], rt, ex[b], re)
        assert np.array_equal(H[b], rh[-1])
        rel = np.abs(ll[b] - rl) / np.abs(rl)
        for k in np.flatnonzero(~(rel <= 1e-10)):
            # DESIGN.md section 4: 1e-10 relative where cond(K + S) <= 1e6
            with (matern_oracle.kernel(d) if d else __import__('contextlib').nullcontext()):
                K = so.cov_matrix(x, rh[k])
            KS = K + np.diag(so.s_diagonal(np.diagonal(K), rh[k][-1]))
            assert np.linalg.cond(KS) > 1e6, (b, k, ll[b][k], rl[k])


CASES = [('se', 64, 8, None, 1), ('se', 200, 16, None, 1), ('se', 455, 32, None, 1), ('ard', 200, 8, None, 3),
         ('matern1', 200, 8, 1, 1), ('matern3', 200, 8, 3, 1), ('matern5', 200, 8, 5, 1)]


@pytest.mark.parametrize('name,n,B,d,D', CASES, ids=[c[0] + '_N%d' % c[1] for c in CASES])
def test_tape_parity_with_the_oracle_chain(gp, name, n, B, d, D):
    """40 transitions from iteration 480 across burn_in = 500: theta and trips exact, G to the DESIGN section 4 policy."""
    if D == 1:
        x, y = gp.synthetic.ih45_series(n)
    else:
        x, y = gp.synthetic.ard_inputs(n, d=D)
    _, H0 = gp.synthetic.chain_states(B, n, n_ell=D)
    H0 = np.ascontiguousarray(H0)
    P = D + 2
    scale = np.array([10.0] * D + [10.0, 5.0])
    tape = gp.ops.MarginalTape(*tapes(B, 40, P, 64, seed=n + 7 * P))
    kind = {None: None, 1: 2, 3: 3, 5: 4}[d]
    dev = run(gp, x, y, H0, scale, 480, 40, burn_in=500, tape=tape, kind=kind)
    ref = oracle_chains(x, y, H0, scale, 480, 40, 500, tape, d=d)
    assert_parity(x, y, dev, ref, d=d)
    assert np.all(dev[0][:, :20, -1] == H0[:, None, -1])              # noise frozen before iteration 500


def _shared_inputs(gp, n, B):
    x, y = gp.synthetic.ih45_series(n)
    _, H0 = gp.synthetic.chain_states(B, n)
    return x, y, H0, np.array(gp.synthetic.SCALE)


def test_philox_calls_compose_bit_for_bit(gp):
    import torch
    n, B = 64, 64
    x, y, H0, scale = _shared_inputs(gp, n, B)
    # precondition: at this N an item's log-likelihood does not depend on the batch it is evaluated in
    _, Hb = gp.synthetic.chain_states(1000, n)
    r = torch.tensor(np.tile(y - y.mean(), (1000, 1))).cuda()
    big, _ = gp.ops.loglik_batched(x, r, Hb)
    for j in (0, 17, 999):
        one, _ = gp.ops.loglik_batched(x, r[j:j + 1], Hb[j:j + 1])
        assert one.item() == big[j].item(), j
    K = 6
    full = run(gp, x, y, H0, scale, 600, K, seed=9)
    H = H0.copy()
    for k in range(K):
        step = run(gp, x, y, H, scale, 600 + k, 1, seed=9)
        assert np.array_equal(step[0][:, 0], full[0][:, k]) and np.array_equal(step[1][:, 0], full[1][:, k])
        assert np.array_equal(step[2][:, 0], full[2][:, k])
        H = step[4]
    assert np.array_equal(H, full[4])
    lo = run(gp, x, y, H0[:B // 2], scale, 600, K, seed=9, chain0=0)
    hi = run(gp, x, y, H0[B // 2:], scale, 600, K, seed=9, chain0=B // 2)
    for i in range(4):
        assert np.array_equal(np.concatenate([lo[i], hi[i]]), full[i]), i


def test_bench_shape_repeats_bit_for_bit_in_the_compact_layout(gp):
    import torch
    n, B = 4096, 1024
    _, y = gp.synthetic.ih45_series(n)
    x = np.arange(n, dtype=np.float64).reshape(n, 1)
    _, H0 = gp.synthetic.loglik_batch(B, n)
    scale = np.array(gp.synthetic.SCALE)
    lib = gp._lib.load()
    outs = []
    for _ in range(2):
        # one trip per transition: every round evaluates all 1024 chains, the last one included
        outs.append(run(gp, x, y, H0, scale, 600, 2, seed=5, max_trips=1))
        W, waves = ctypes.c_int(-1), ctypes.c_int(-1)
        lib.gpmc_loglik_layout(ctypes.byref(W), ctypes.byref(waves))
        assert W.value > 0, (W.value, waves.value)
        act, _ = gp.ops.marginal_rounds()
        assert list(act) == [B, B, B]
    for a, b in zip(outs[0], outs[1]):
        assert np.array_equal(a, b)
    a = run(gp, x, y, H0[:256], scale, 600, 1, seed=5)
    b = run(gp, x, y, H0[:256], scale, 600, 1, seed=5)
    for u, v in zip(a, b):
        assert np.array_equal(u, v)


# the bracket rule hyp_min = max(hyp - v, 0) is exact only where it does not clip (tests/test_marginal_oracle.py): priors
# that keep theta above scale
PRIOR = (np.array([20., 20., 20.]), np.array([1., 1., 120.]))
SCALE = np.array([3.0, 3.0, 2.0])


def posterior_data(n, seed=5):
    rng = np.random.default_rng(seed)
    x = np.linspace(0, 60, n).reshape(-1, 1)
    return x, 15 * np.sin(x[:, 0] / 8) + 6 * rng.standard_normal(n) + 50


@pytest.mark.parametrize('d', [None, 3], ids=['se', 'matern3'])
def test_posterior_moments_match_quadrature(gp, d):
    x, y = posterior_data(64)
    grid = mo.posterior_grid(x, y, prior=PRIOR, kind=d, bounds=((1.9, 3.9), (1.9, 4.2), (1.15, 2.3)), n=(41, 41, 41))
    assert grid['edge'] < 1e-4
    B = 2048
    H0 = np.tile([20., 20., 6.], (B, 1))
    hh, ll, tt, ex, _ = run(gp, x, y, H0, SCALE, 0, 300, burn_in=0, seed=21, prior_k=PRIOR[0], prior_theta=PRIOR[1],
                            kind=None if d is None else 3)
    assert np.all(ex == 0) and np.all(hh.min(axis=(0, 1)) > SCALE)
    logs = np.log(hh[:, 50:, :])
    for j in range(3):
        se = mo.batch_means_se(logs[:, :, j])
        assert abs(logs[:, :, j].mean() - grid['mean'][j]) < 4 * se, (j, logs[:, :, j].mean(), grid['mean'][j], se)


def test_failed_factorisation_is_a_rejected_proposal_that_shrinks(gp):
    n = 64
    x, y = gp.synthetic.ih45_series(n)
    H0 = np.array([[1.0, 10.0, 1.2], [2.0, 9.0, 1.5]])
    scale = np.array(gp.synthetic.SCALE)
    v, u0, U = tapes(2, 3, 3, 64, seed=4)
    v[0, 0, 0] = 0.9                      # bracket of ell clipped at 0 ...
    U[0, 0, 0, 0] = 0.0                   # ... and the first proposal at ell = 0: x / ell is not finite
    tape = gp.ops.MarginalTape(v, u0, U)
    dev = run(gp, x, y, H0, scale, 0, 3, burn_in=0, tape=tape)
    ref = oracle_chains(x, y, H0, scale, 0, 3, 0, tape)
    assert_parity(x, y, dev, ref)
    lo = np.maximum(H0[0] - scale * v[0, 0], 0)
    bad = lo + scale * U[0, 0, 0]
    assert bad[0] == 0.0
    G, info = gp.ops.loglik_batched(x, (y - y.mean())[None], bad[None])
    assert int(info.item()) != 0 and np.isnan(G.item())        # the ladder could not rescue it
    assert dev[2][0, 0] >= 2                                     # rejected: the transition went on in a shrunk bracket


def test_non_finite_start_and_exhausted_budget(gp):
    n, B = 64, 12
    x, y = gp.synthetic.ih45_series(n)
    _, H0 = gp.synthetic.chain_states(B, n)
    H0[3] = [np.nan, 5.0, 1.0]
    scale = np.array(gp.synthetic.SCALE)
    tape = gp.ops.MarginalTape(*tapes(B, 10, 3, 64, seed=8))
    dev = run(gp, x, y, H0, scale, 600, 10, tape=tape, max_trips=1)
    ref = oracle_chains(x, y, H0, scale, 600, 10, 500, tape, max_trips=1)
    hh, ll, tt, ex, H = dev
    assert ex[3] == -1 and np.all(tt[3] == 0) and np.all(np.isnan(ll[3]))
    assert np.array_equal(hh[3], np.tile(H0[3], (10, 1)), equal_nan=True)
    good = [b for b in range(B) if b != 3]
    assert_parity(x, y, tuple(a[good] for a in dev), [ref[b] for b in good])
    assert ex[good].sum() > 0                                    # the budget of one trip ran out somewhere
    kept = (tt[good] == 1) & np.all(hh[good] == np.concatenate([H0[good][:, None], hh[good][:, :-1]], axis=1), axis=2)
    assert kept.sum() >= ex[good].sum()


def test_argument_checks(gp):
    import torch
    lib = gp._lib.load()
    x = torch.zeros((8, 1), dtype=torch.float64, device='cuda')
    y = torch.zeros(8, dtype=torch.float64, device='cuda')
    h = torch.ones((2, 3), dtype=torch.float64, device='cuda')
    p3 = torch.ones(3, dtype=torch.float64, device='cuda')
    ws = torch.empty(lib.gpmc_workspace_bytes(gp._lib.OP_MARGINAL, 8, 1, 2), dtype=torch.uint8, device='cuda')
    t = torch.full((2, 1, 3), 0.5, dtype=torch.float64, device='cuda')

    def call(B=2, P=3, kind=0, n_iters=1, it0=0, burn_in=0, max_trips=8, jp=1, tv=None, tu=None, tU=None, T=0, N=8):
        return lib.gpmc_marginal_run(x.data_ptr(), N, 1, y.data_ptr(), 0.0, h.data_ptr(), B, P, kind, p3.data_ptr(),
                                     p3.data_ptr(), p3.data_ptr(), it0, n_iters, burn_in, 1, 0, tv, tu, tU, T, max_trips, jp,
                                     None, None, None, None, ws.data_ptr(), ws.numel(), None)
    E = -22
    assert call(kind=7) == E and call(kind=1, P=5) == E and call(P=4) == E and call(kind=2, P=4) == E
    assert call(n_iters=-1) == E and call(it0=-1) == E and call(burn_in=-1) == E and call(max_trips=0) == E
    assert call(jp=5) == E and call(N=0) == E and call(B=-1) == E
    assert call(tv=t.data_ptr()) == E and call(tv=t.data_ptr(), tu=t.data_ptr(), tU=t.data_ptr(), T=0) == E
    assert call(T=3) == E
    assert call(B=0) == 0 and call(n_iters=0) == 0
    torch.cuda.synchronize()
    hh, ll, tt, ex = gp.ops.marginal_run(x, y, h[:0], p3, 0, 4)
    assert hh.shape == (0, 4, 3)
    hh, ll, tt, ex = gp.ops.marginal_run(x, y, h, p3, 0, 0)
    assert hh.shape == (2, 0, 3) and np.array_equal(h.cpu().numpy(), np.ones((2, 3)))


def test_chain_ensemble_gauss_equals_marginal_run(gp):
    n, B = 64, 10
    x, y, H0, scale = _shared_inputs(gp, n, B)
    ens = gp.chains.ChainEnsemble(x, y, None, H0, scale, seed=13, likelihood='gauss', burn_in=500)
    hist, ll, trips = ens.run(8, start_iter=495)
    hh, l2, t2, ex, _ = run(gp, x, y, H0, scale, 495, 8, seed=13, burn_in=500)
    assert np.array_equal(hist, np.transpose(hh, (0, 2, 1))) and np.array_equal(ll, l2) and np.array_equal(trips, t2)
    ens2 = gp.chains.ChainEnsemble(x, y, None, H0, scale, seed=13, likelihood='gauss', burn_in=500)
    h1, l1, t1 = ens2.sweep(495)
    assert np.array_equal(h1, hh[:, 0]) and np.array_equal(l1, l2[:, 0]) and np.array_equal(t1, t2[:, 0])


@pytest.mark.parametrize('d', [None, 3], ids=['se', 'matern3'])
def test_gpr_sample_hyp_and_mixture_predict(gp, d):
    from gpmc_b200.kcGP import covK, gpK
    x, y = posterior_data(48)
    xs = np.linspace(-5, 65, 23).reshape(-1, 1)
    model = gpK.GPR()
    model.setData(x, y)
    if d is not None:
        model.setPrior(kernel=covK.Matern(np.log(15.), d, np.log(20.)))
    else:
        model.setPrior(kernel=covK.RBF(np.log(15.), np.log(20.)))
    model.setNoise(np.log(6.))
    S = model.sampleHyp(30, n_chains=4, scale=[5., 5., 2.], burn=10, thin=4, seed=3)
    assert S.shape == (4 * 5, 3) and np.all(np.isfinite(S))
    ym, ys2, fm, fs2, lp = model.predict(xs, samples=S)
    from contextlib import nullcontext
    mus, vs = [], []
    with (matern_oracle.kernel(d) if d else nullcontext()):
        for h in S:
            _, _, _, Fs2, Fmu = so.inf_mcmc_unit(y, x, y, xs, h)
            mus.append(Fmu[:, 0])
            vs.append(Fs2[:, 0])
    mus, vs = np.array(mus), np.array(vs)
    mu = mus.mean(axis=0)
    var = (vs + mus ** 2).mean(axis=0) - mu ** 2
    assert np.allclose(fm[:, 0], mu, rtol=1e-9, atol=1e-9 * np.abs(mu).max())
    assert np.allclose(fs2[:, 0], var, rtol=1e-9, atol=1e-9 * var.max())
    assert np.allclose(ys2[:, 0], var + np.mean(S[:, -1] ** 2), rtol=1e-9, atol=1e-9 * var.max())
