"""Envelope skips on vs. forced off (gpmc_set_tuning(14, .)) on the bench.py workload: per-class kernel ms per step, the
update GEMM's executed vs. dense tile-K work, and launched vs. working CTAs of the update GEMM and the panel solve.

The work counts replay the plain left-looking schedule of sequences.cu (the one the bench workload runs: N=4096, waves of
several hundred matrices) on envelopes the device wrote: every (item, block column j, 128x64 output tile) of the update
GEMM contracts over K = 128 j densely, and from floor16 of the tile's envelope on with the skips; a panel-solve CTA works
when one of its 64-row blocks has a nonzero left of column 128 (j + 1).  A second run with ell = 0.05 (diagonal K+S: every
update tile and almost every solve CTA is empty) gives the cost of an empty CTA.

    python tools/envelope_ab.py [--n 4096] [--chains 1024] [--steps 3] [--out DIR]
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gpmc_b200 as gp
import torch

NB, TBM, TBN, TBK, ENV_ROWS = 128, 128, 64, 16, 64


def envelopes(x, G, H, wave=128):
    """The envelopes the device writes, read back from gpmc_loglik_batched's workspace, wave by wave
    (layout as in tests/test_gpu_envelope.py)."""
    n = G.shape[1]
    a = lambda v: (v + 255) // 256 * 256
    ld = (n + 15) // 16 * 16
    nblk = (n + ENV_ROWS - 1) // ENV_ROWS
    out = []
    gp.ops.set_tuning(14, 1)
    for s0 in range(0, G.shape[0], wave):
        g, h = G[s0:s0 + wave], H[s0:s0 + wave]
        B = g.shape[0]
        ws = gp.ops.Workspace()
        gp.ops.loglik_batched(x, g, h, workspace=ws, max_wave=B)
        off = a(B * 8) + a(B * 4) + 256 + a(32 * ld * 8) + B * (n + 1) * ld * 8 + B * NB * NB * 8
        out.append(ws.buf[off:off + B * nblk * 4].cpu().numpy().view(np.int32).reshape(B, nblk).astype(np.int64))
    return np.concatenate(out)


def work_counts(env, n, wave):
    """Update GEMM: (dense, executed) K chunks summed over tiles, (launched, working) CTAs; panel solve: (launched,
    working) CTAs -- per factorisation of every item, for waves of `wave` matrices."""
    B, nblk = env.shape
    big = np.iinfo(np.int64).max // 4

    def first_col(r0, r1):                          # env over rows r0 .. r1-1 (all < n here), per item
        return env[:, r0 // ENV_ROWS:(r1 - 1) // ENV_ROWS + 1].min(axis=1)

    g_dense = g_exec = g_launch = g_work = 0
    t_launch = t_work = 0
    nt = (n + NB - 1) // NB
    for j in range(1, nt):
        j0 = j * NB
        rows = n - j0
        kb = [first_col(j0 + TBN * tn, min(n, j0 + TBN * tn + TBN)) for tn in range(NB // TBN) if j0 + TBN * tn < n]
        for tm in range((rows + TBM - 1) // TBM):
            ka = first_col(j0 + tm * TBM, min(n, j0 + tm * TBM + TBM))
            for k_b in kb:
                kenv = np.maximum(ka, k_b)
                koff = np.maximum(0, (np.minimum(kenv, big) // TBK) * TBK)
                chunks = np.maximum(0, j0 - koff) // TBK
                g_dense += B * (j0 // TBK)
                g_exec += int(chunks.sum())
                g_launch += B
                g_work += int((chunks > 0).sum())
        # panel solve of block column j - 1 (rows below its diagonal block; the border row rides in the last block)
        c0 = j0 - NB
        srows = n - (c0 + NB)
        if srows <= 0:
            continue
        sblk = srows // ENV_ROWS if srows % ENV_ROWS == 0 else (srows + ENV_ROWS - 1) // ENV_ROWS
        per = 4 if sblk * wave >= 16 * 296 else (2 if sblk * wave >= 8 * 296 else 1)
        grid = (sblk + per - 1) // per
        empty = np.stack([first_col(c0 + NB + rb * ENV_ROWS, min(n, c0 + NB + rb * ENV_ROWS + ENV_ROWS)) >= c0 + NB
                          if rb < sblk - 1 else np.zeros(B, bool) for rb in range(sblk)], axis=1)
        for cta in range(grid):
            t_launch += B
            t_work += int((~empty[:, cta::grid].all(axis=1)).sum())
    return {'gemm_k_chunks_dense': g_dense, 'gemm_k_chunks_executed': g_exec,
            'gemm_k_work_fraction': g_exec / g_dense if g_dense else None,
            'gemm_ctas_launched': g_launch, 'gemm_ctas_working': g_work,
            'trsm_ctas_launched': t_launch, 'trsm_ctas_working': t_work}


def per_step_ms(x, G, H, on, steps):
    gp.ops.set_tuning(14, 1 if on else 0)
    try:
        for _ in range(2):
            ll, info = gp.ops.loglik_batched(x, G, H)
        torch.cuda.synchronize()
        gp.ops.profile(True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            ll, info = gp.ops.loglik_batched(x, G, H)
        e1.record()
        torch.cuda.synchronize()
        prof = gp.ops.profile_read()
        gp.ops.profile(False)
        return e0.elapsed_time(e1) / steps, {k: v[0] / steps for k, v in prof.items() if v[1] > 0}, ll.cpu().numpy(), info.cpu().numpy()
    finally:
        gp.ops.set_tuning(14, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n', type=int, default=4096)
    ap.add_argument('--chains', type=int, default=1024)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    n, B = a.n, a.chains
    x = np.arange(n, dtype=np.float64).reshape(n, 1)
    G, H = gp.synthetic.loglik_batch(B, n)
    lib = gp._lib.load()
    ws_bytes = lib.gpmc_workspace_bytes(gp._lib.OP_LOGLIK, n, 1, B)
    per_item = lib.gpmc_workspace_bytes(gp._lib.OP_LOGLIK, n, 1, 2) - lib.gpmc_workspace_bytes(gp._lib.OP_LOGLIK, n, 1, 1)
    wave = min(B, ws_bytes // per_item)
    env = envelopes(x, G, H)
    counts = work_counts(env, n, wave)
    rows = []
    for label, Hs in (('bench', H), ('diagonal_ell_0.05', np.column_stack([np.full(B, 0.05), H[:, 1:]]))):
        res = {}
        for on in (False, True):
            ms, cls, ll, info = per_step_ms(x, G, Hs, on, a.steps)
            res['on' if on else 'off'] = {'ms_per_step': ms, 'kernel_ms_per_step': cls, 'll': ll, 'info': info}
        same = bool(np.array_equal(res['on']['ll'], res['off']['ll']) and np.array_equal(res['on']['info'], res['off']['info']))
        row = {'case': label, 'n': n, 'chains': B, 'wave': int(wave), 'outputs_bitwise_equal': same}
        for k in ('off', 'on'):
            row[k] = {'ms_per_step': res[k]['ms_per_step'], 'kernel_ms_per_step': res[k]['kernel_ms_per_step']}
        if label == 'bench':
            row['work'] = counts
        else:
            # every update tile is empty: gemm ms over launched CTAs is what one empty CTA costs the step
            c = work_counts(np.tile(np.arange(env.shape[1]) * ENV_ROWS, (B, 1)), n, wave)
            km = res['on']['kernel_ms_per_step']
            row['empty_cta_us'] = {'gemm_update': 1e3 * km.get('gemm_update', 0.0) / c['gemm_ctas_launched'],
                                   'panel_trsm': 1e3 * km.get('panel_trsm', 0.0) / c['trsm_ctas_launched']}
            row['work'] = c
        rows.append(row)
        print(json.dumps(row))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'envelope_ab.json'), 'w') as f:
            json.dump(rows, f, indent=1)


if __name__ == '__main__':
    main()
