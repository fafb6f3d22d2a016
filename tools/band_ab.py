"""Band-only assembly and launches on vs. off (gpmc_set_tuning(15, .)) on the bench.py workload, in the dense layout with
the region left of the band cleared inline in the assembly (gpmc_set_tuning(16, 2)) or on a side stream (16, 1), and in
the compact band layout (gpmc_set_tuning(17, 1), default: only the band's columns are stored, all chains in fewer waves)
with the panel factor and solve of a block column in one launch (default) or in two (gpmc_set_tuning(9, 1)):
ms per step, per class kernel ms and launches per step, waves and row width W of each arm, launched vs. working CTAs of
the assembly, the update GEMM and the panel solve, a bitwise comparison of loglik and info with the envelope-only run and
between the two compact arms, and the name and power limit of the card.

The CTA counts replay the plain left-looking schedule of sequences.cu (the one the bench workload runs) on the envelopes,
band starts w and wave bands the device wrote (read back from gpmc_loglik_batched's workspace, wave by wave).  A CTA
works when it does more than leave: an assembly CTA when its tile is in the band, an update-GEMM CTA when its contraction
is not empty, a panel-solve CTA when one of its row blocks has a nonzero left of the block column's end (or carries the
border row).

    python tools/band_ab.py [--n 4096] [--chains 1024] [--steps 3] [--out DIR]
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


def band_data(x, G, H, wave):
    """Per wave: (envelope [B, nblk], w [B, nblk], band of the launches, band width of the assembly)."""
    n = G.shape[1]
    a = lambda v: (v + 255) // 256 * 256
    ld = (n + 15) // 16 * 16
    nblk = (n + ENV_ROWS - 1) // ENV_ROWS
    out = []
    for s0 in range(0, G.shape[0], wave):
        g, h = G[s0:s0 + wave], H[s0:s0 + wave]
        B = g.shape[0]
        ws = gp.ops.Workspace()
        gp.ops.loglik_batched(x, g, h, workspace=ws, max_wave=B)
        buf = ws.buf.cpu().numpy()
        band = buf[a(B * 8) + a(B * 4):a(B * 8) + a(B * 4) + 8].view(np.int32)
        off_env = a(B * 8) + a(B * 4) + 256 + a(32 * ld * 8) + B * (n + 1) * ld * 8 + B * NB * NB * 8
        env = buf[off_env:off_env + B * nblk * 4].view(np.int32).reshape(B, nblk).astype(np.int64)
        w = buf[off_env + B * nblk * 4:off_env + 2 * B * nblk * 4].view(np.int32).reshape(B, nblk).astype(np.int64)
        out.append((env, w, int(band[0]), int(band[1])))
    return out


def work_counts(waves, n, band_on):
    """Launched and working CTAs per factorisation of every item (summed over waves)."""
    big = np.iinfo(np.int64).max // 4
    c = dict.fromkeys(('asm_launched', 'asm_working', 'gemm_launched', 'gemm_working', 'trsm_launched', 'trsm_working'), 0)
    nt = (n + NB - 1) // NB
    nblk = (n + ENV_ROWS - 1) // ENV_ROWS
    for env, w, band, width in waves:
        B = env.shape[0]

        def first_col(r0, r1):
            return env[:, r0 // ENV_ROWS:(r1 - 1) // ENV_ROWS + 1].min(axis=1)

        if band_on:
            c['asm_launched'] += B * nblk * (min(width, nblk - 1) + 1)
            c['asm_working'] += int((np.arange(nblk)[None, :] - w + 1).sum())
        else:
            c['asm_launched'] += B * nblk * (nblk + 1) // 2
            c['asm_working'] += B * nblk * (nblk + 1) // 2
        for j in range(1, nt):
            j0 = j * NB
            rows = n - j0
            if band_on:
                rows = min(rows, NB + band * ENV_ROWS)
            kb = [first_col(j0 + TBN * tn, min(n, j0 + TBN * tn + TBN)) for tn in range(NB // TBN) if j0 + TBN * tn < n]
            for tm in range((rows + TBM - 1) // TBM):
                ka = first_col(j0 + tm * TBM, min(n, j0 + tm * TBM + TBM))
                for k_b in kb:
                    kenv = np.maximum(ka, k_b)
                    koff = np.maximum(0, (np.minimum(kenv, big) // TBK) * TBK)
                    c['gemm_launched'] += B
                    c['gemm_working'] += int((koff < j0).sum())
            # panel solve of block column j - 1 (rows below its diagonal block and the border row)
            c0 = j0 - NB
            srows = n + 1 - (c0 + NB)
            if srows <= 1:
                continue
            sblk = (srows - 1) // ENV_ROWS if (srows - 1) % ENV_ROWS == 0 else (srows + ENV_ROWS - 1) // ENV_ROWS
            blocks = list(range(sblk))
            if band_on and band < sblk - 1:
                blocks = list(range(band)) + [sblk - 1]
            per = 4 if len(blocks) * B >= 16 * 296 else (2 if len(blocks) * B >= 8 * 296 else 1)
            grid = (len(blocks) + per - 1) // per
            empty = np.stack([first_col(c0 + NB + rb * ENV_ROWS, min(n, c0 + NB + rb * ENV_ROWS + ENV_ROWS)) >= c0 + NB
                              if rb < sblk - 1 else np.zeros(B, bool) for rb in blocks], axis=1)
            for cta in range(grid):
                c['trsm_launched'] += B
                c['trsm_working'] += int((~empty[:, cta::grid].all(axis=1)).sum())
    return c


def layout():
    """(row width W of the compact layout or 0 for dense, waves) of the last call"""
    import ctypes
    W, waves = ctypes.c_int(-1), ctypes.c_int(-1)
    gp._lib.load().gpmc_loglik_layout(ctypes.byref(W), ctypes.byref(waves))
    return W.value, waves.value


def per_step_ms(x, G, H, band, clear, compact, fuse_off, steps):
    gp.ops.set_tuning(15, band)
    gp.ops.set_tuning(16, clear)
    gp.ops.set_tuning(17, compact)
    gp.ops.set_tuning(9, fuse_off)
    try:
        for _ in range(2):
            ll, info = gp.ops.loglik_batched(x, G, H)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            ll, info = gp.ops.loglik_batched(x, G, H)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        lay = layout()
        gp.ops.profile(True)                    # per-class times in a run of their own (the events slow the host)
        for _ in range(steps):
            gp.ops.loglik_batched(x, G, H)
        prof = gp.ops.profile_read()
        gp.ops.profile(False)
        return (ms, {k: v[0] / steps for k, v in prof.items() if v[1] > 0}, {k: v[1] / steps for k, v in prof.items() if v[1] > 0},
                ll.cpu().numpy(), info.cpu().numpy(), lay)
    finally:
        gp.ops.set_tuning(15, 1)
        gp.ops.set_tuning(16, 2)
        gp.ops.set_tuning(17, 1)
        gp.ops.set_tuning(9, 0)


def card():
    """name and power limit of the card, read next to the measurement"""
    import subprocess
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ''
    return q or torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n', type=int, default=4096)
    ap.add_argument('--chains', type=int, default=1024)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--rounds', type=int, default=2, help='alternations of the three arms')
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    n, B = a.n, a.chains
    x = np.arange(n, dtype=np.float64).reshape(n, 1)
    G, H = gp.synthetic.loglik_batch(B, n)
    lib = gp._lib.load()
    ws_bytes = lib.gpmc_workspace_bytes(gp._lib.OP_LOGLIK, n, 1, B)
    per_item = lib.gpmc_workspace_bytes(gp._lib.OP_LOGLIK, n, 1, 2) - lib.gpmc_workspace_bytes(gp._lib.OP_LOGLIK, n, 1, 1)
    wave = min(B, ws_bytes // per_item)
    gp.ops.set_tuning(17, 0)                    # the dense layout's workspace contents, wave by wave
    try:
        waves = band_data(x, G, H, wave)
    finally:
        gp.ops.set_tuning(17, 1)
    # the compact layout factors every chain in one wave (when it fits) with the call's widest band
    one = [(np.concatenate([w[0] for w in waves]), np.concatenate([w[1] for w in waves]),
            max(w[2] for w in waves), max(w[3] for w in waves))]
    # (label, band, clear, compact, fused panels forbidden)
    arms = (('band_off', 0, 1, 0, 1), ('band_on_side_clear', 1, 1, 0, 1), ('band_on_inline_clear', 1, 2, 0, 1),
            ('band_compact', 1, 2, 1, 1), ('band_compact_fused', 1, 2, 1, 0))
    res = {k[0]: [] for k in arms}
    outs = {}
    for _ in range(a.rounds):
        for label, band, clear, compact, fuse_off in arms:
            ms, cls, nl, ll, info, lay = per_step_ms(x, G, H, band, clear, compact, fuse_off, a.steps)
            res[label].append({'ms_per_step': ms, 'kernel_ms_per_step': cls, 'launches_per_step': nl, 'band_W': lay[0],
                               'waves': lay[1]})
            outs[label] = (ll, info)
    gp.ops.set_tuning(14, 0)
    try:
        ll_d, info_d = gp.ops.loglik_batched(x, G, H)
        dense = (ll_d.cpu().numpy(), info_d.cpu().numpy())
    finally:
        gp.ops.set_tuning(14, 1)
    same = lambda p, q: bool(np.array_equal(p[0].view(np.int64), q[0].view(np.int64)) and np.array_equal(p[1], q[1]))
    row = {'card': card(), 'n': n, 'chains': B, 'wave': int(wave), 'steps': a.steps,
           'wave_bands': [{'launch_band_blocks': w[2], 'assembly_band_tiles': w[3]} for w in waves],
           'work_band_off': work_counts(waves, n, False), 'work_band_on': work_counts(waves, n, True),
           'work_band_compact': work_counts(one, n, True),
           'outputs_bitwise_equal_to_band_off': {k[0]: same(outs[k[0]], outs['band_off']) for k in arms},
           'compact_fused_bitwise_equal_to_compact': same(outs['band_compact_fused'], outs['band_compact']),
           'band_off_bitwise_equal_to_dense': same(outs['band_off'], dense),
           'arms': res}
    print(json.dumps(row))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'band_ab.json'), 'w') as f:
            json.dump(row, f, indent=1)


if __name__ == '__main__':
    main()
