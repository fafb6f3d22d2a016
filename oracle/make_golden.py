"""Generate ``tests/golden/*.npz`` by running the reference's own ``kcMCMC/sliceSample.py``.

TEST INFRASTRUCTURE (see ``oracle/__init__.py``).  Needs a checkout of the original project:
``GPMC_REFERENCE_ROOT=<checkout> python -m oracle.make_golden``.  The tests read only the
committed fixtures; neither this script nor the original project is needed to run them.
``python -m oracle.make_golden literal-cases`` writes ``literal_cases.npz`` alone and runs
without a checkout; its ``source`` entry then says that the restatement made it.

Each ``sds_N*.npz`` holds the inputs of one ``surrogate_slice_sampling`` call, the explicit
randomness (tape), and what the UNMODIFIED reference returned for it, plus literal
``aux_var_model`` / ``log_gamma`` outputs at the starting point.  ``loglik_*.npz`` hold
known-answer log-marginal values (``sliceSample.py:147`` form and ``:145-146`` form).
``chain_N64.npz`` is a 40-iteration chain of the literal sampler across the burn-in switch.
"""
import os
import sys

import numpy as np

from . import kcgp_shim, reference_loader as rl, sds_oracle as so

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(os.path.dirname(HERE), 'tests', 'golden')
# OpenBLAS threads the fixtures are made with.  OpenBLAS splits a product by its thread count, and f' of the
# ill-conditioned SDS fixtures follows that summation order (up to 5e-4 absolute at N = 200 and 512 between 1 and 8
# threads), so the tests replay the restatement with the same count.
BLAS_THREADS = 8


def pinned_blas():
    """Context in which OpenBLAS runs BLAS_THREADS threads, whatever the host's cores (needs threadpoolctl)."""
    import threadpoolctl
    return threadpoolctl.threadpool_limits(limits=BLAS_THREADS)


def _series(n, seed=124, hyp=(5.0, 4.0, 2.5)):
    # demoRegression.py:117-136 recipe (sf 20 -> 4, clipped to the likelihood's support)
    rs = np.random.RandomState(seed)
    x = np.arange(0, n, dtype=np.float64).reshape(n, 1)
    K = kcgp_shim.RBF(np.log(hyp[0]), np.log(hyp[1])).getCovMatrix(x=x, mode='train')
    L = kcgp_shim.jitchol(K + hyp[2] ** 2 * np.eye(n))
    y = np.clip(np.dot(L, rs.normal(size=(n,))) + 91.1538461538, 0., 100.)
    return x, y


def sds_case(n, it, seed, hyp0, f_mode):
    x, y = _series(n)
    hyp = np.asarray(hyp0, dtype=np.float64)
    scale = np.asarray([10., 10., 5.])
    if f_mode == 'zero':
        f = np.zeros(n)                                  # framework.py:64
    else:
        # a mid-chain state: three restated transitions from the framework.py:63-64 start
        histF, histHyp, _ = so.run_chain(x, y, hyp, scale, 3, 9000 + seed, start_iter=it)
        f, hyp = histF[:, -1].copy(), histHyp[:, -1].copy()
    tape = rl.Tape.from_seed(seed, n, p=3, max_trips=64)
    prop_f, prop_hyp, trips = rl.run_literal_with_tape(f, x, y, hyp, scale, it, tape)

    # literal pieces at the starting point (module functions called directly)
    mod = rl.load_literal(fresh=True)
    rnd = rl._TapeRandom(tape)
    mod.np = rl._NumpyProxy(rnd)
    K = kcgp_shim.RBF(np.log(hyp[0]), np.log(hyp[1])).getCovMatrix(x=x, mode='train')
    g, K_S, m, C, L = mod.aux_var_model(f, K, hyp[2])
    ita = np.linalg.solve(C, f - m)
    curG = -(np.dot(np.dot(g.T, np.linalg.inv(K_S)), g) / 2. + np.log(np.diag(L.T)).sum() + g.shape[0] * np.log(2 * np.pi) / 2.)
    prior, grad = mod.log_gamma(hyp, np.asarray([1., 3., 3.]), np.asarray([1., 1.5, 3.]), True)

    # restatement trace (per-trip values); equality with the literal result is asserted here too
    tr = so.SweepTrace()
    of, oh = so.surrogate_slice_sampling(f, x, y, hyp, scale, it, tape, trace=tr)
    assert np.array_equal(of, prop_f) and np.array_equal(oh, prop_hyp) and tr.n_trips == trips, \
        'restatement diverged from the literal reference (n=%d it=%d seed=%d)' % (n, it, seed)
    out = dict(x=x, y=y, f=f, hyp=hyp, scale=scale, it=it, z=tape.z, v=tape.v, u0=tape.u0, U=tape.U[:trips + 2],
               ref_prop_f=prop_f, ref_prop_hyp=prop_hyp, ref_trips=trips,
               ref_g=g, ref_m=m, ref_ita=ita, ref_diagL=np.diag(L).copy(), ref_diagC=np.diag(C).copy(),
               ref_curG=curG, ref_prior=prior, ref_prior_grad=grad,
               trace_cur_llk=tr.cur_llk, trace_threshold=tr.threshold,
               trace_prop_hyp=np.asarray(tr.prop_hyp), trace_propG=np.asarray(tr.propG),
               trace_propG_chol=np.asarray(tr.propG_chol), trace_prop_llk=np.asarray(tr.prop_llk),
               trace_proposal=np.asarray(tr.proposal), cond_KS=np.linalg.cond(K_S))
    if n <= 64:
        out.update(ref_K=K, ref_L=L, ref_C=C)
    return out


def loglik_cases():
    """Known answers for the metric's unit over the prior-supported range, incl. a cond ~1e8 case."""
    rows = []
    rs = np.random.RandomState(2024)
    for n in (8, 64, 200, 512, 1000):
        x = np.arange(0, n, dtype=np.float64).reshape(n, 1)
        for hyp in ([1., 10., 1.2], [0.35, 2.0, 0.2], [5., 4., 2.5], [7.8868277, 9.69728866, 1.2],
                    [12.5, 18., 0.05], [0.01, 0.02, 4.9], [3.3, 25., 0.004]):
            hyp = np.asarray(hyp)
            g = hyp[2] * rs.standard_normal(n) + rs.standard_normal(n)
            K = so.cov_matrix(x, hyp)
            K_S = K + np.diag(so.s_diagonal(np.diagonal(K), hyp[2]))
            try:
                L, info = __import__('scipy').linalg.lapack.dpotrf(K_S, lower=1)
                if info != 0:
                    continue                      # keep only cases that need no jitter
                L = np.tril(L)
                rows.append(dict(n=n, x=x[:, 0], hyp=hyp, g=g,
                                 ll_inv=float(so.log_marginal_inv_form(g, K_S, L)),
                                 ll_chol=float(so.log_marginal_chol_form(g, L)),
                                 cond=float(np.linalg.cond(K_S)),
                                 logdet_half=float(np.log(np.diag(L)).sum())))
            except np.linalg.LinAlgError:
                continue
    return rows


def ard_cases():
    rows = []
    rs = np.random.RandomState(77)
    for n, d in ((32, 2), (128, 4), (512, 4)):
        x = rs.uniform(0., 10., size=(n, d))
        for _ in range(3):
            hyp = np.concatenate([rs.uniform(0.5, 6., size=d), [rs.uniform(1., 12.)], [rs.uniform(0.3, 3.)]])
            g = hyp[-1] * rs.standard_normal(n)
            K = so.cov_matrix(x, hyp)
            K_S = K + np.diag(so.s_diagonal(np.diagonal(K), hyp[-1]))
            L = kcgp_shim.jitchol(K_S)
            rows.append(dict(n=n, d=d, x=x, hyp=hyp, g=g, ll_inv=float(so.log_marginal_inv_form(g, K_S, L)),
                             ll_chol=float(so.log_marginal_chol_form(g, L)), cond=float(np.linalg.cond(K_S))))
    return rows


def chain_case(n=64, iters=40, start_iter=480, seed=500):
    """Literal sampler run as ``framework.py:68-75`` does, across the ``iter == 500`` switch."""
    x, y = _series(n)
    hyp = np.asarray([1., 10., 1.2])
    scale = np.asarray([10., 10., 5.])
    f = np.zeros(n)
    histF = np.zeros((n, iters))
    histHyp = np.zeros((3, iters))
    trips = np.zeros(iters, dtype=np.int64)
    for i in range(iters):
        tape = rl.Tape.from_seed(seed + i, n, p=3, max_trips=64)
        f, hyp, t = rl.run_literal_with_tape(f, x, y, hyp, scale, start_iter + i, tape)
        histF[:, i], histHyp[:, i], trips[i] = f, hyp, t
    oF, oH, oT = so.run_chain(x, y, [1., 10., 1.2], scale, iters, seed, start_iter=start_iter)
    assert np.array_equal(oF, histF) and np.array_equal(oH, histHyp) and np.array_equal(oT, trips)
    return dict(x=x, y=y, hyp0=np.asarray([1., 10., 1.2]), scale=scale, iters=iters, start_iter=start_iter, seed=seed,
                ref_histF=histF, ref_histHyp=histHyp, ref_trips=trips)


class _ZeroMean(object):
    def getMean(self, x):
        return np.zeros((x.shape[0], 1))


def infmcmc_case(n=64, ns=17, n_samples=5, seed=808):
    """The reference's own ``inf_mcmc`` (``sliceSample.py:234-284``) under the shim, on a small synthetic model."""
    import types
    x, y = _series(n)
    rs = np.random.RandomState(seed)
    xs = np.sort(rs.uniform(0, n, size=(ns, 1)), axis=0)
    hyp = np.asarray([4.2, 3.1, 1.7])
    f = (y - y.mean())[:, None] * 0.6 + 0.3 * rs.standard_normal((n, n_samples))
    model = types.SimpleNamespace(x=x, y=y.reshape(-1, 1), xs=xs, meanfunc=_ZeroMean(),
                                  covfunc=kcgp_shim.RBF(np.log(hyp[0]), np.log(hyp[1])),
                                  likfunc=kcgp_shim.TruncatedGauss2(upper=100 - y.mean(), lower=0 - y.mean(), log_sigma=np.log(hyp[2])))
    mod = rl.load_literal(fresh=True)
    ym, lw, up, Fs2 = mod.inf_mcmc(f, model)
    return dict(x=x, y=y, xs=xs, hyp=hyp, f=f, ref_ym=ym, ref_lw=lw, ref_up=up, ref_Fs2=Fs2)


def infmcmc_batched_case(n=96, ns=13, S=6, seed=909):
    """The reference's ``inf_mcmc`` called once per stored sample, each with its own (ll, sf, sn) -- the loop of
    ``framework.py:223-243`` -- as the fixture for the batched device path."""
    import types
    x, y = _series(n)
    rs = np.random.RandomState(seed)
    xs = np.sort(rs.uniform(0, n, size=(ns, 1)), axis=0)
    Hyp = np.column_stack([rs.uniform(1.5, 7., S), rs.uniform(2., 9., S), rs.uniform(0.6, 2.8, S)])
    F = (y - y.mean())[:, None] * rs.uniform(0.4, 0.9, S)[None, :] + 0.3 * rs.standard_normal((n, S))
    mod = rl.load_literal(fresh=True)
    out = [[], [], [], []]
    for s in range(S):
        model = types.SimpleNamespace(x=x, y=y.reshape(-1, 1), xs=xs, meanfunc=_ZeroMean(),
                                      covfunc=kcgp_shim.RBF(np.log(Hyp[s, 0]), np.log(Hyp[s, 1])),
                                      likfunc=kcgp_shim.TruncatedGauss2(upper=100 - y.mean(), lower=0 - y.mean(), log_sigma=np.log(Hyp[s, 2])))
        res = mod.inf_mcmc(F[:, s:s + 1], model)
        uni = so.inf_mcmc_unit(F[:, s], x, y, xs, Hyp[s])
        for k in range(4):
            assert np.array_equal(res[k], uni[k]), 'restated inf_mcmc differs from the literal one'
            out[k].append(res[k])
    return dict(x=x, y=y, xs=xs, Hyp=Hyp, F=F, ref_ym=np.stack(out[0]), ref_lw=np.stack(out[1]), ref_up=np.stack(out[2]),
                ref_Fs2=np.stack(out[3]))


def ess_case(n, seed, hyp, f_scale):
    """The reference's ``elliptical_slice`` (``sliceSample.py:15-74``) run UNMODIFIED on a tape; ``nu`` is the Cholesky
    draw ``jitchol(K) z`` (``z`` is stored too, so the device's own draw can be checked against it)."""
    x, y = _series(n)
    rs = np.random.RandomState(seed)
    hyp = np.asarray(hyp, dtype=np.float64)
    f = f_scale * (y - y.mean()) + 0.2 * rs.standard_normal(n)
    z = rs.standard_normal(n)
    nu = so.ess_nu_from_z(x, hyp, z)
    tape = rl.EssTape(nu, rs.random_sample(), rs.random_sample(64))
    pf, trips = rl.run_literal_ess_with_tape(f, x, y, hyp, tape)
    of, otrips = so.elliptical_slice(f, x, y, hyp, tape)
    assert np.array_equal(pf, of) and trips == otrips, 'restated elliptical_slice differs from the literal one'
    cond_K = float(np.linalg.cond(so.cov_matrix(x, np.concatenate([hyp[:-1], [1.0]]))))
    return dict(x=x, y=y, hyp=hyp, f=f, z=z, nu=nu, u=tape.u, theta=tape.theta, ref_prop_f=pf, ref_trips=trips, cond_K=cond_K)


# the cases of tests/test_oracle_vs_reference.py, stored in literal_cases.npz
LITERAL_SDS_CASES = [(24, 0, 1), (24, 777, 2), (96, 499, 3), (96, 500, 4)]
LITERAL_ESS_CASES = [(40, 5), (120, 6)]
LOG_GAMMA_HYP = [0.7, 3.0, 1.9]


def literal_cases():
    """Inputs, tapes and outputs of the cases of ``tests/test_oracle_vs_reference.py``.  The outputs are computed by the
    restatement; where the reference is present, its own functions run on the same tapes and must return the same bits.
    ``source`` records which of the two produced the stored values."""
    lit = rl.available()
    mod = rl.load_literal() if lit else None
    out = {'source': 'restatement, asserted bit-identical to kcMCMC/sliceSample.py' if lit else 'oracle/sds_oracle.py restatement'}
    for n, it, seed in LITERAL_SDS_CASES:
        x, y = _series(n)
        f, hyp, scale = np.zeros(n), np.array([1., 10., 1.2]), np.array([10., 10., 5.])
        tape = rl.Tape.from_seed(seed, n)
        tr = so.SweepTrace()
        of, oh = so.surrogate_slice_sampling(f, x, y, hyp, scale, it, tape, trace=tr)
        if lit:
            pf, ph, trips = rl.run_literal_with_tape(f, x, y, hyp, scale, it, tape)
            assert trips == tr.n_trips and np.array_equal(ph, oh) and np.array_equal(pf, of)
        k = 'sds_N%d_it%d_s%d_' % (n, it, seed)
        out.update({k + 'x': x, k + 'y': y, k + 'f': f, k + 'hyp': hyp, k + 'scale': scale, k + 'z': tape.z, k + 'v': tape.v,
                    k + 'u0': tape.u0, k + 'U': tape.U[:tr.n_trips + 2], k + 'prop_f': of, k + 'prop_hyp': oh,
                    k + 'trips': tr.n_trips})
    for n, seed in LITERAL_ESS_CASES:
        x, y = _series(n)
        rs = np.random.RandomState(seed)
        hyp = np.array([4., 5., 1.8])
        f = 0.7 * (y - y.mean())
        tape = rl.EssTape(so.ess_nu_from_z(x, hyp, rs.standard_normal(n)), rs.random_sample(), rs.random_sample(64))
        of, trips = so.elliptical_slice(f, x, y, hyp, tape)
        if lit:
            pf, ltrips = rl.run_literal_ess_with_tape(f, x, y, hyp, tape)
            assert ltrips == trips and np.array_equal(pf, of)
        k = 'ess_N%d_s%d_' % (n, seed)
        out.update({k + 'x': x, k + 'y': y, k + 'f': f, k + 'hyp': hyp, k + 'nu': tape.nu, k + 'u': tape.u,
                    k + 'theta': tape.theta, k + 'prop_f': of, k + 'trips': trips})
    hyp = np.array(LOG_GAMMA_HYP)
    a, b = so.log_gamma(hyp, so.PRIOR_K3, so.PRIOR_THETA3, True)
    if lit:
        c, d = mod.log_gamma(hyp, so.PRIOR_K3, so.PRIOR_THETA3, True)
        assert np.array_equal(a, c) and np.array_equal(b, d)
    out.update(log_gamma_hyp=hyp, log_gamma=a, log_gamma_grad=b)
    return out


def write_literal_cases():
    np.savez_compressed(os.path.join(GOLDEN, 'literal_cases.npz'), **literal_cases())
    print('literal_cases written')


def main():
    if not rl.available():
        sys.exit('set GPMC_REFERENCE_ROOT to a checkout of the original project: fixtures are made by running its sliceSample.py')
    os.makedirs(GOLDEN, exist_ok=True)
    cases = [(8, 0, 11, [1., 10., 1.2], 'zero'), (8, 700, 12, [0.35, 2.0, 0.2], 'mid'),
             (64, 0, 21, [1., 10., 1.2], 'zero'), (64, 650, 22, [0.35, 2.0, 0.2], 'mid'), (64, 499, 23, [3., 6., 2.], 'mid'),
             (200, 0, 2, [1., 10., 1.2], 'zero'), (200, 600, 31, [1., 10., 1.2], 'mid'),
             (512, 10, 41, [1., 10., 1.2], 'zero'), (512, 900, 42, [4., 5., 2.2], 'mid')]
    for n, it, seed, hyp0, fm in cases:
        out = sds_case(n, it, seed, hyp0, fm)
        path = os.path.join(GOLDEN, 'sds_N%d_it%d_s%d.npz' % (n, it, seed))
        np.savez_compressed(path, **out)
        print('%s trips=%d prop_hyp=%s cond=%.2e' % (os.path.basename(path), out['ref_trips'], out['ref_prop_hyp'], out['cond_KS']))
    rows = loglik_cases()
    np.savez_compressed(os.path.join(GOLDEN, 'loglik_iso.npz'), n_cases=len(rows),
                        **{'%s_%d' % (k, i): v for i, r in enumerate(rows) for k, v in r.items()})
    print('loglik_iso: %d cases, cond range %.1e..%.1e, max |inv-chol| rel %.1e' % (
        len(rows), min(r['cond'] for r in rows), max(r['cond'] for r in rows),
        max(abs(r['ll_inv'] - r['ll_chol']) / abs(r['ll_chol']) for r in rows)))
    rows = ard_cases()
    np.savez_compressed(os.path.join(GOLDEN, 'loglik_ard.npz'), n_cases=len(rows),
                        **{'%s_%d' % (k, i): v for i, r in enumerate(rows) for k, v in r.items()})
    print('loglik_ard: %d cases' % len(rows))
    np.savez_compressed(os.path.join(GOLDEN, 'infmcmc_N64.npz'), **infmcmc_case())
    print('infmcmc_N64 written')
    np.savez_compressed(os.path.join(GOLDEN, 'infmcmc_batched_N96.npz'), **infmcmc_batched_case())
    print('infmcmc_batched_N96 written')
    for n, seed, hyp, fs in ((64, 61, [3., 5., 1.5], 0.8), (200, 62, [5., 4., 2.5], 0.6), (200, 63, [1., 10., 1.2], 0.0), (455, 64, [8., 3., 2.0], 0.9),
                             (200, 65, [0.35, 2.0, 0.2], 0.7)):
        out = ess_case(n, seed, hyp, fs)
        np.savez_compressed(os.path.join(GOLDEN, 'ess_N%d_s%d.npz' % (n, seed)), **out)
        print('ess_N%d_s%d: %d proposals' % (n, seed, out['ref_trips']))
    ch = chain_case()
    np.savez_compressed(os.path.join(GOLDEN, 'chain_N64.npz'), **ch)
    print('chain_N64: trips mean %.2f max %d; final hyp %s' % (ch['ref_trips'].mean(), ch['ref_trips'].max(), ch['ref_histHyp'][:, -1]))
    write_literal_cases()


if __name__ == '__main__':
    with pinned_blas():
        write_literal_cases() if sys.argv[1:] == ['literal-cases'] else main()
