"""Device time of one log-likelihood gradient call (ops.loglik_grad_batched) against one log-likelihood call
(ops.loglik_batched) on the same inputs (synthetic.loglik_batch), per call: CUDA events, one warm-up call of each arm, the
arms alternated rep by rep.  Also the per-class kernel split of each arm (gpmc_profile_read, a separate pass), the flop
count of the gradient path, whether the two calls' loglik are bitwise equal, and the card and its power limit.

    python tools/grad_timing.py [--reps 3] [--out profiles/r05_loglik_grad.json]

Flop per item of the gradient path: Cholesky N^3/3 (nominal, as bench.py counts it; the band makes the real count smaller),
the triangular inverse U = L^-T N^3/3, and W = U U^T as launched: 128 x 64 tiles of each 128-row block row from the band
bound's first column on, each contracting from its first row to N (2 * 128 * 64 * (N - 128 R) per tile).
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gpmc_b200 as gp
import torch

CASES = [(4096, 256, 1), (4096, 1024, 1), (2048, 64, 1), (512, 4096, 4)]
NB, TILE_N, ENV_ROWS = 128, 64, 64


def card():
    out = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader,nounits', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(',')
        out.update({'smi_name': q[0].strip(), 'power_limit_w': float(q[1]), 'sm_max_mhz': float(q[2])})
    except Exception as e:          # the measurement stands without it, but says so
        out['power_limit_w'] = None
        out['power_query_error'] = repr(e)
    return out


def band_width(x, h):
    """The band bound of cov_assemble.cu for one item: max over 64-row blocks r of r - w[r] (64-column tiles)."""
    n, D = x.shape
    nblk = (n + ENV_ROWS - 1) // ENV_ROWS
    n_ell = len(h) - 2
    ell = np.exp(np.log(h[:n_ell]))
    sf2 = np.exp(2 * np.log(h[n_ell]))
    thr = 760.0 + max(0.0, np.log(sf2))
    lo_b = np.array([x[r * ENV_ROWS:(r + 1) * ENV_ROWS].min(axis=0) for r in range(nblk)])
    hi_b = np.array([x[r * ENV_ROWS:(r + 1) * ENV_ROWS].max(axis=0) for r in range(nblk)])
    e = ell if n_ell > 1 else np.full(D, ell[0])
    lo = np.arange(nblk)
    for r in range(nblk):
        gap = np.maximum(0.0, np.maximum(lo_b[r] / e - hi_b[:r] / e, lo_b[:r] / e - hi_b[r] / e))
        maybe = np.flatnonzero(~(0.5 * (gap ** 2).sum(axis=1) * (1 - 1e-9) > thr))
        lo[r] = maybe[0] if len(maybe) else r
    w = lo.copy()
    w[1:] = np.minimum(w[1:], lo[:-1])
    w[:-1] = np.minimum(w[:-1], lo[1:])
    w = w // (NB // ENV_ROWS) * (NB // ENV_ROWS)
    return int((np.arange(nblk) - w).max())


def flops(n, width):
    nrb = (n + NB - 1) // NB
    syrk = 0.0
    for R in range(nrb):
        c0 = 0 if width < 0 or 2 * (nrb - 1) - width <= 0 else max(0, 2 * R - width) * ENV_ROWS
        cols = min(n, R * NB + NB) - c0
        syrk += 2.0 * min(NB, n - R * NB) * ((cols + TILE_N - 1) // TILE_N) * TILE_N * (n - R * NB)
    return {'cholesky_nominal': n ** 3 / 3.0, 'inverse': n ** 3 / 3.0, 'w_syrk_launched': syrk,
            'w_syrk_dense_lower': 2.0 * sum(min(NB, n - R * NB) * min(n, R * NB + NB) * (n - R * NB) for R in range(nrb))}


def time_call(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def class_split(fn):
    gp.ops.profile(True)
    fn()
    torch.cuda.synchronize()
    prof = gp.ops.profile_read()
    gp.ops.profile(False)
    return {k: round(v[0], 3) for k, v in prof.items() if v[0] > 0}


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--out', default=os.path.join('profiles', 'r05_loglik_grad.json'))
    a = ap.parse_args(argv)
    rec = {'card': card(), 'reps': a.reps, 'cases': []}
    for n, B, D in CASES:
        x = np.arange(n, dtype=np.float64).reshape(n, 1) if D == 1 else gp.synthetic.ard_inputs(n, D)[0]
        G, H = gp.synthetic.loglik_batch(B, n, n_ell=D)
        xd, Gd, Hd = torch.tensor(x).cuda(), torch.tensor(G).cuda(), torch.tensor(H).cuda()
        ws_l, ws_g = gp.ops.Workspace(), gp.ops.Workspace()
        arm_l = lambda: gp.ops.loglik_batched(xd, Gd, Hd, workspace=ws_l)
        arm_g = lambda: gp.ops.loglik_grad_batched(xd, Gd, Hd, workspace=ws_g)
        _, (ll_l, info_l) = time_call(arm_l)
        _, (ll_g, grad, info_g) = time_call(arm_g)
        t_l, t_g = [], []
        for _ in range(a.reps):
            t_l.append(time_call(arm_l)[0])
            t_g.append(time_call(arm_g)[0])
        per_item = gp._lib.load().gpmc_workspace_bytes(gp._lib.OP_LOGLIK_GRAD, n, D, 1)
        wave = max(1, min(B, ws_g.buf.numel() // per_item))
        widths = [max(band_width(x, h) for h in H[s0:s0 + wave]) for s0 in range(0, B, wave)]
        fl = flops(n, max(widths))
        ok = (info_l.cpu().numpy() == 0) & (info_g.cpu().numpy() == 0)
        ll_l, ll_g = ll_l.cpu().numpy(), ll_g.cpu().numpy()
        ms_l, ms_g = float(np.median(t_l)), float(np.median(t_g))
        flop_item = fl['cholesky_nominal'] + fl['inverse'] + fl['w_syrk_launched']
        case = {'n': n, 'batch': B, 'ard_dims': D if D > 1 else 0, 'loglik_ms': ms_l, 'grad_ms': ms_g, 'ratio': ms_g / ms_l,
                'loglik_ms_reps': t_l, 'grad_ms_reps': t_g, 'grad_evals_per_s': B / (ms_g * 1e-3),
                'band_width_tiles_per_wave': widths, 'flop_per_item': fl,
                'grad_tflops': B * flop_item / (ms_g * 1e-3) / 1e12,
                'failed_items': int((~ok).sum()), 'grad_finite': bool(np.isfinite(grad.cpu().numpy()[ok]).all()),
                'loglik_bitwise_equal': bool(np.array_equal(ll_l[ok], ll_g[ok])),
                'loglik_max_rel_diff': float(np.max(np.abs(ll_l[ok] - ll_g[ok]) / np.abs(ll_l[ok]))) if ok.any() else None,
                'kernel_ms_loglik': class_split(arm_l), 'kernel_ms_grad': class_split(arm_g)}
        rec['cases'].append(case)
        print(json.dumps({k: case[k] for k in ('n', 'batch', 'ard_dims', 'loglik_ms', 'grad_ms', 'ratio', 'grad_tflops')}), flush=True)
        del ws_l, ws_g
        torch.cuda.empty_cache()
    rec['note'] = ('per-call device time, CUDA events around one call, median of the reps, arms alternated; kernel_ms_* from a '
                   'separate pass with event pairs around every launch; grad_tflops counts flop_per_item (nominal Cholesky + '
                   'inverse + W as launched) over the gradient call\'s time')
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec['card']))


if __name__ == '__main__':
    main()
