"""Device time of the Matern kinds (d = 1, 3, 5) beside the squared exponential on the same inputs, per call: CUDA events,
one warm-up call of each arm, the arms alternated rep by rep.  Also the per-class kernel split of each arm (gpmc_profile_read,
a separate pass), the layout and wave count of every log-likelihood call (gpmc_loglik_layout), and the card and its power
limit.

    python tools/matern_timing.py [--reps 3] [--out profiles/r07_matern.json]

Cases (x = 0, 1, .., N-1; g and (ell, sf, sn) from synthetic.loglik_batch, the bench's bracket):
  loglik  N = 4096 x 1024 at the bench's bracket and at a short-ell bracket (ell / 10: the band is narrow enough for the
          compact layout), N = 512 x 4096 at the bench's bracket;
  grad    N = 4096 x 256;
  sds     one surrogate-data slice-sampling transition (Philox, iteration 600) of 256 chains at N = 4096.
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import gpmc_b200 as gp
import torch
from grad_timing import card, class_split, time_call

KINDS = [('se', None), ('matern1', 2), ('matern3', 3), ('matern5', 4)]


def layout():
    import ctypes
    lib = gp._lib.load()
    W, waves = ctypes.c_int(-1), ctypes.c_int(-1)
    gp._lib.check(lib.gpmc_loglik_layout(ctypes.byref(W), ctypes.byref(waves)), 'gpmc_loglik_layout')
    return {'band_W': W.value, 'waves': waves.value}


def run_case(name, arms, reps):
    """arms: {kind name: (callable, after-call info fn or None)}; returns the case record."""
    out = {'case': name, 'arms': {}}
    for k, (fn, info) in arms.items():
        time_call(fn)
        out['arms'][k] = {'ms_reps': []}
        if info:
            out['arms'][k].update(info())
    for _ in range(reps):
        for k, (fn, _) in arms.items():
            out['arms'][k]['ms_reps'].append(time_call(fn)[0])
    for k, (fn, _) in arms.items():
        a = out['arms'][k]
        a['ms'] = float(np.median(a['ms_reps']))
        a['kernel_ms'] = class_split(fn)
    base = out['arms']['se']['ms']
    for k in out['arms']:
        out['arms'][k]['ratio_to_se'] = out['arms'][k]['ms'] / base
    print(json.dumps({'case': name, **{k: round(v['ms'], 3) for k, v in out['arms'].items()}}), flush=True)
    return out


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--out', default=os.path.join('profiles', 'r07_matern.json'))
    a = ap.parse_args(argv)
    rec = {'card': card(), 'reps': a.reps, 'cases': []}

    def loglik_case(name, n, B, ell_scale):
        x = torch.tensor(np.arange(n, dtype=np.float64).reshape(n, 1)).cuda()
        G, H = gp.synthetic.loglik_batch(B, n)
        H[:, 0] *= ell_scale
        Gd, Hd = torch.tensor(G).cuda(), torch.tensor(H).cuda()
        arms = {}
        for k, kind in KINDS:
            ws = gp.ops.Workspace()
            fn = (lambda ws=ws, kind=kind: gp.ops.loglik_batched(x, Gd, Hd, workspace=ws, kind=kind))

            def info(fn=fn):
                ll, inf = fn()
                torch.cuda.synchronize()
                return dict(layout(), failed_items=int((inf.cpu().numpy() != 0).sum()))
            arms[k] = (fn, info)
        c = run_case(name, arms, a.reps)
        c.update({'n': n, 'batch': B, 'ell_range': [float(H[:, 0].min()), float(H[:, 0].max())]})
        rec['cases'].append(c)
        del arms
        torch.cuda.empty_cache()

    loglik_case('loglik_4096x1024_bench_bracket', 4096, 1024, 1.0)
    loglik_case('loglik_4096x1024_short_ell', 4096, 1024, 0.1)
    loglik_case('loglik_512x4096_bench_bracket', 512, 4096, 1.0)

    n, B = 4096, 256
    x = torch.tensor(np.arange(n, dtype=np.float64).reshape(n, 1)).cuda()
    G, H = gp.synthetic.loglik_batch(B, n)
    Gd, Hd = torch.tensor(G).cuda(), torch.tensor(H).cuda()
    arms = {}
    for k, kind in KINDS:
        ws = gp.ops.Workspace()
        arms[k] = ((lambda ws=ws, kind=kind: gp.ops.loglik_grad_batched(x, Gd, Hd, workspace=ws, kind=kind)), None)
    c = run_case('grad_4096x256', arms, a.reps)
    c.update({'n': n, 'batch': B})
    rec['cases'].append(c)
    del arms
    torch.cuda.empty_cache()

    xs, y = gp.synthetic.ih45_series(n)
    F0, H0 = gp.synthetic.chain_states(B, n)
    scale = np.array(gp.synthetic.SCALE)
    xd, yd = torch.tensor(xs).cuda(), torch.tensor(y).cuda()
    arms, state = {}, {}
    for k, kind in KINDS:
        ws = gp.ops.Workspace()

        def fn(ws=ws, kind=kind, k=k):
            # every call starts from the same state, so each rep times the same transition
            F, Hh = torch.tensor(F0).cuda(), torch.tensor(H0).cuda()
            nt, ll, st = gp.ops.sds_sweep(xd, yd, F, Hh, scale, 600, seed=3, max_trips=64, workspace=ws, kind=kind)
            state[k] = (nt, st)
            return nt

        def info(k=k):
            nt, st = state[k]
            return {'trips_total': int(nt.sum().item()), 'exhausted': int((st != 0).sum().item())}
        arms[k] = (fn, info)
    c = run_case('sds_transition_4096x256', arms, max(1, a.reps - 1))
    c.update({'n': n, 'batch': B, 'note': 'each call includes the H2D copy of the 256 x 4096 start state (about 8 MB)'})
    rec['cases'].append(c)

    rec['note'] = ('per-call device time, CUDA events around one call, median of the reps, arms alternated rep by rep; '
                   'kernel_ms from a separate pass with event pairs around every launch; band_W = 0 is the dense layout')
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec['card']))


if __name__ == '__main__':
    main()
