"""Device time of the marginal slice sampler (gpmc_marginal_run) beside the log-likelihood unit it is built on.

    python tools/marginal_timing.py [--reps 3] [--iters 4] [--out profiles/r08_marginal.json]

Per shape: one call of n_iters transitions of every chain (Philox, iteration 600, burn-in 500 passed), timed with CUDA
events after a warm-up call, alternated rep by rep with ONE standalone gpmc_loglik_batched call of the same number of items
(the chains' starting theta, y - mean(y) as every right-hand side).  Reported: ms per iteration of all chains, mean trips
per transition, rounds per iteration, log-likelihood evaluations per second inside the sampler, and the share of the
sampler's time spent in tail rounds (rounds that evaluate fewer than 1/8 of the chains; host wall time per round, each
round ends in a synchronisation).  Also one surrogate-data slice-sampling transition (gpmc_sds_run, 256 chains) at N = 4096
for the per-transition comparison, and the card and its power limit.

Shapes: N = 4096 x 1024 SE with the bench's inputs (synthetic.loglik_batch, x = 0 .. N-1, y from synthetic.ih45_series);
N = 512 ARD D = 4 x 4096 (synthetic.ard_inputs); N = 4096 Matern 3 x 256 at ell / 10 (short enough for the compact layout).
"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import gpmc_b200 as gp
import torch
from grad_timing import card


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1), out


def layout():
    lib = gp._lib.load()
    W, waves = ctypes.c_int(-1), ctypes.c_int(-1)
    lib.gpmc_loglik_layout(ctypes.byref(W), ctypes.byref(waves))
    return {'band_W': W.value, 'waves': waves.value}


def case(name, x, y, H0, scale, kind, n_iters, reps):
    B, P = H0.shape
    xd, yd = torch.tensor(x).cuda(), torch.tensor(y).cuda()
    H0d = torch.tensor(H0).cuda()
    ws_s, ws_l = gp.ops.Workspace(), gp.ops.Workspace()
    r = torch.tensor(np.tile(y - y.mean(), (B, 1))).cuda()
    state = {}

    def sampler():
        H = H0d.clone()
        state['out'] = gp.ops.marginal_run(xd, yd, H, scale, 600, n_iters, seed=11, kind=kind, workspace=ws_s)
        return state['out']

    def unit():
        return gp.ops.loglik_batched(xd, r, H0d, workspace=ws_l, kind=kind)

    timed(sampler)
    timed(unit)
    rec = {'case': name, 'n': x.shape[0], 'chains': B, 'P': P, 'kind': kind, 'n_iters': n_iters, 'sampler_ms': [], 'unit_ms': []}
    for _ in range(reps):
        rec['sampler_ms'].append(timed(sampler)[0])
        act, ms = gp.ops.marginal_rounds()
        sampler_layout = layout()
        rec['unit_ms'].append(timed(unit)[0])
    hh, ll, tt, ex = state['out']
    tt = tt.cpu().numpy()
    evals = int(act.sum())
    med = float(np.median(rec['sampler_ms']))
    tail = act < max(1, B // 8)
    rec.update({
        'sampler_ms_median': med,
        'ms_per_iteration': med / n_iters,
        'mean_trips': float(tt.mean()),
        'rounds': int(act.shape[0]),
        'rounds_per_iteration': float((act.shape[0] - 1) / n_iters),
        'evals': evals,
        'evals_per_s_in_sampler': evals / (med / 1e3),
        'unit_ms_median': float(np.median(rec['unit_ms'])),
        'unit_evals_per_s': B / (float(np.median(rec['unit_ms'])) / 1e3),
        'tail_rounds': int(tail.sum()),
        'tail_share_of_time': float(ms[tail].sum() / ms.sum()),
        'round_active': act.tolist(),
        'round_ms': ms.tolist(),
        'exhausted': int((ex.cpu().numpy() != 0).sum()),
        'last_round_layout': sampler_layout,
        'unit_layout': layout(),
    })
    print(json.dumps({k: rec[k] for k in ('case', 'ms_per_iteration', 'mean_trips', 'rounds_per_iteration',
                                          'evals_per_s_in_sampler', 'unit_ms_median', 'tail_share_of_time')}), flush=True)
    del ws_s, ws_l
    torch.cuda.empty_cache()
    return rec


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--iters', type=int, default=4)
    ap.add_argument('--out', default=os.path.join('profiles', 'r08_marginal.json'))
    a = ap.parse_args(argv)
    rec = {'card': card(), 'reps': a.reps, 'cases': []}
    scale3 = np.array(gp.synthetic.SCALE)

    n = 4096
    x = np.arange(n, dtype=np.float64).reshape(n, 1)
    _, y = gp.synthetic.ih45_series(n)
    _, H = gp.synthetic.loglik_batch(1024, n)
    rec['cases'].append(case('se_4096x1024_bench', x, y, H, scale3, None, a.iters, a.reps))

    n, D = 512, 4
    x, y = gp.synthetic.ard_inputs(n, d=D)
    _, H = gp.synthetic.loglik_batch(4096, n, n_ell=D)
    rec['cases'].append(case('ard4_512x4096', x, y, H, np.array([10.] * D + [10., 5.]), None, a.iters, a.reps))

    n = 4096
    x = np.arange(n, dtype=np.float64).reshape(n, 1)
    _, y = gp.synthetic.ih45_series(n)
    _, H = gp.synthetic.loglik_batch(256, n)
    H[:, 0] *= 0.1
    rec['cases'].append(case('matern3_4096x256_short_ell', x, y, H, np.array([1.0, 10.0, 5.0]), 3, a.iters, a.reps))

    # the surrogate-data slice sampler: one transition of 256 chains at the same N (per-transition comparison)
    xs, ys = gp.synthetic.ih45_series(n)
    F0, H0 = gp.synthetic.chain_states(256, n)
    xd, yd = torch.tensor(xs).cuda(), torch.tensor(ys).cuda()
    ws = gp.ops.Workspace()

    def sds():
        F, Hh = torch.tensor(F0).cuda(), torch.tensor(H0).cuda()
        return gp.ops.sds_run(xd, yd, F, Hh, scale3, 600, 1, seed=3, workspace=ws)
    timed(sds)
    ms = [timed(sds)[0] for _ in range(max(1, a.reps - 1))]
    rec['sds_run_4096x256_one_transition'] = {'ms': ms, 'ms_median': float(np.median(ms)),
                                              'note': 'each call includes the H2D copy of the 256 x 4096 start state'}
    print(json.dumps({'sds_run_ms': float(np.median(ms))}), flush=True)
    rec['note'] = ('CUDA events around one call; sampler and standalone unit alternated rep by rep after one warm-up each; '
                   'round_ms is host wall time per round (each round ends in a stream synchronisation)')
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec['card']))


if __name__ == '__main__':
    main()
