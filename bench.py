#!/usr/bin/env python
"""bench.py -- GP log-lik evals/sec (N=4096, batched chains) on N B200s, with the Cholesky's fraction of FP64 peak.

One "step" = one pass of the hot path over one batch: every chain of this rank evaluates one
log-marginal likelihood  log N(g_c; 0, K(theta_c) + S(theta_c))  (assemble K+S, Cholesky, forward
substitution, quadratic form, log-det; SURVEY 8a rows a2+a4+a5) and, with more than one rank, the
per-chain results are all-gathered once (the "one all-gather of samples per sweep" of SURVEY 8e).

  python bench.py [--gpus N] [--steps K] [--warmup W]              our CUDA path
  python bench.py --impl reference [...]                            the reference's CPU path (oracle port)
  python bench.py --dump-outputs DIR [...]                          also write the last timed step's outputs as DIR/*.npy
                                                                    (CUDA path only; refused with --impl reference)

Prints ONE JSON line (rank 0).  `value` is timed with the inputs resident in HBM; `e2e` goes through
the C-ABI host-buffer call (pinned H2D of x/g/theta and D2H of loglik/info inside the timed region).
Besides the headline (BASELINE config 5 shard) the line carries `configs`: one sub-record per other
BASELINE config shape (log-lik unit at C2/C3/C4) and per device-resident SDS sweep (whole
`surrogate_slice_sampling` transitions, sliceSample.py:76-163, at C2, C3 and a C5 shard), each with
its own timing, roofline fraction and a GPU-vs-oracle check on sampled items.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'GP log-lik evals/sec (N=4096, batched chains)'
UNIT = 'evals/s'


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--nobs', dest='n', type=int, default=4096, help='observations per chain (BASELINE: 4096)')
    ap.add_argument('--chains-per-gpu', type=int, default=1024, help='BASELINE config 5: 8192 chains over 8 GPUs')
    ap.add_argument('--cpu-sample', type=int, default=4, help='evals in the bounded CPU sample')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-peaks', action='store_true')
    ap.add_argument('--no-configs', action='store_true', help='skip the sub-records of the other BASELINE configs / SDS sweeps')
    ap.add_argument('--only-configs', default=None, help='comma list of sub-record names to run (e.g. C3_loglik,C3_sds)')
    ap.add_argument('--gemm-cfg', type=int, default=None, help='experiment: DMMA tile kernel variant (0: 8 warps, 1: 16 warps)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step returned (loglik, info) as DIR/<name>.npy, for comparing two builds')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs needs --impl b200')
    return args


def workload_config(n, B, world):
    """`config` of the JSON line: IDENTICAL (keys and values) for the CUDA arm and the reference arm."""
    return {'workload': 'BASELINE config 5 (8xB200 chain-parallel: N=4096, 8192 chains sharded by GPU): N=%d, %d chains '
                        'per GPU, one log-lik eval per chain per step, SE+noise kernel on a unit-spaced 1-D grid '
                        '(IH45-shaped)' % (n, B),
            'n': n, 'chains_per_gpu': B, 'evals_per_step': world * B, 'kernel': 'SE iso + noise',
            'l2': 'per-step working set %d matrices x %.0f MiB >> 126 MB L2 (no flush needed)' % (B, n * n * 8 / 2 ** 20),
            'collective': 'one all_gather of loglik per step' if world > 1 else 'none (single rank)'}


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU every 200 ms while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.nv = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, 'nvmlClocksEventReasonHwSlowdown', 0x8): 'hw_slowdown',
            getattr(nv, 'nvmlClocksEventReasonHwThermalSlowdown', 0x40): 'hw_thermal_slowdown',
            getattr(nv, 'nvmlClocksEventReasonSwThermalSlowdown', 0x20): 'sw_thermal_slowdown',
            getattr(nv, 'nvmlClocksEventReasonSwPowerCap', 0x4): 'sw_power_cap',
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        import numpy as np
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {'sm_mhz': med, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons), 'samples': len(self.samples)}


# ------------------------------------------------------------------------------------ CPU (oracle)
def set_blas_threads():
    """The CPU arm uses every host core.  torchrun exports OMP_NUM_THREADS=1 when nproc > 1, which numpy's OpenBLAS
    honours, so the thread count is set explicitly BEFORE numpy is imported and the EFFECTIVE count is what gets
    reported (threadpoolctl)."""
    cores = os.cpu_count() or 1
    for k in ('OPENBLAS_NUM_THREADS', 'OMP_NUM_THREADS', 'MKL_NUM_THREADS'):
        os.environ[k] = str(cores)
    return cores


def effective_blas_threads():
    try:
        import threadpoolctl
        import numpy  # noqa: F401  (loads the BLAS so that threadpoolctl can see it)
        import scipy.linalg  # noqa: F401
        pools = [p for p in threadpoolctl.threadpool_info() if p.get('user_api') == 'blas']
        if pools:
            return int(max(p.get('num_threads', 1) for p in pools))
    except Exception:
        pass
    return int(os.environ.get('OPENBLAS_NUM_THREADS', os.cpu_count() or 1))


def cpu_unit_evals_per_s(n, sample, form, ard=0, first=0):
    """Time the oracle's restatement of the unit on the host cores (OpenBLAS threads = all cores)."""
    import numpy as np
    from oracle import sds_oracle as so
    import gpmc_b200 as gp
    if ard:
        x, _ = gp.synthetic.ard_inputs(n, ard)
        n_ell = ard
    else:
        x = np.arange(n, dtype=np.float64).reshape(n, 1)
        n_ell = 1
    G, H = gp.synthetic.loglik_batch(sample, n, n_ell=n_ell, first_chain=first)
    so.loglik_unit(x[:256], G[0, :256], H[0], form=form)        # warm the BLAS threads
    t0 = time.perf_counter()
    vals = [so.loglik_unit(x, G[i], H[i], form=form) for i in range(sample)]
    dt = time.perf_counter() - t0
    return sample / dt, dt, vals


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path.  The reference is pure
    Python with its kcGP primitives missing, so the arm is the oracle port (oracle/sds_oracle.py),
    in the form the reference writes it: dense inv for the quadratic form (sliceSample.py:147)."""
    if rank != 0:
        return
    threads = effective_blas_threads()
    sample = max(1, min(2, 12 // max(1, args.steps)))      # ~5 s per eval at N=4096 on 8 cores
    for _ in range(min(args.warmup, 1)):
        cpu_unit_evals_per_s(args.n, 1, 'inv')
    t0 = time.perf_counter()
    total = 0
    for _ in range(args.steps):
        cpu_unit_evals_per_s(args.n, sample, 'inv')
        total += sample
    dt = time.perf_counter() - t0
    v = total / dt
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': 1e3 * dt / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': workload_config(args.n, args.chains_per_gpu, max(1, args.gpus)),
        'cpu_baseline': {'value': v, 'unit': UNIT, 'cores': threads, 'kind': 'port',
                         'host_cpus': os.cpu_count(),
                         'sample': 'each timed step is a bounded sample of the workload: %d steps x %d evals at N=%d, one '
                                   'chain after another on the host (the reference has no multi-chain mode, '
                                   'framework.py:68-75), in the form the reference writes: sliceSample.py:136-137,183-190,'
                                   '196,147 (dense inv); numpy/scipy OpenBLAS, %d threads in effect (threadpoolctl; set '
                                   'explicitly, torchrun\'s OMP_NUM_THREADS=1 overridden)' % (args.steps, sample, args.n, threads)},
        'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------- GPU path
def measured_peaks(torch, gp):
    """FP64 peaks measured in this run: cuBLAS DGEMM 8192^3 (the practical dense-FP64 ceiling) and the
    register-resident DMMA / DFMA issue rates of our own probes."""
    out = {}
    n = 8192
    a = torch.randn((n, n), dtype=torch.float64, device='cuda')
    b = torch.randn((n, n), dtype=torch.float64, device='cuda')
    c = torch.empty_like(a)
    for _ in range(2):
        torch.matmul(a, b, out=c)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b, out=c)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    out['cublas_dgemm_8192_tflops'] = 2.0 * n ** 3 / (best * 1e-3) / 1e12
    del a, b, c
    torch.cuda.empty_cache()
    out['dmma_issue_tflops'] = gp.ops.fp64_peak('dmma', 8192)[0]
    out['dfma_issue_tflops'] = gp.ops.fp64_peak('dfma', 8192)[0]
    return out


def committed_traffic(n, nb):
    """DRAM bytes per eval of the update kernel from the committed ncu summary of the CURRENT kernel
    (profiles/r02_traffic.json, written by tools/ncu_traffic.py from an `ncu --set full` capture); None if absent."""
    try:
        d = json.load(open(os.path.join(ROOT, 'profiles', 'r02_traffic.json')))
        for row in d.get('update_kernel', []):
            if row.get('n') == n and row.get('panel_width') == nb:
                return row.get('dram_bytes_per_eval'), d.get('source')
    except Exception:
        pass
    return None, None


def hbm_peak_gbs():
    try:
        return json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json'))).get('hbm_gbs'), 'MEASURED_PEAKS.json'
    except Exception:
        return 6650.0, 'fallback of B200_PROFILING.md (MEASURED_PEAKS.json absent)'


def chol_kernel_ms(prof):
    return prof['gemm_update'][0] + prof['potf2'][0] + prof['panel_trsm'][0] + prof.get('fused_small', (0.0, 0))[0]


def sub_loglik(gp, torch, np, name, n, B, ard, reps, peak_tf, n_check, what):
    """Log-lik unit at one BASELINE config shape: timing (CUDA events), Cholesky roofline fraction (N^3/3 flop per eval
    over the wall time of the pass AND over the Cholesky launches alone), GPU vs oracle on `n_check` sampled items."""
    from oracle import sds_oracle as so
    if ard:
        x, _ = gp.synthetic.ard_inputs(n, ard)
        n_ell = ard
    else:
        x = np.arange(n, dtype=np.float64).reshape(n, 1)
        n_ell = 1
    G, H = gp.synthetic.loglik_batch(B, n, n_ell=n_ell)
    xd, Gd, Hd = torch.tensor(x).cuda(), torch.tensor(G).cuda(), torch.tensor(H).cuda()
    for _ in range(3):
        ll, info = gp.ops.loglik_batched(xd, Gd, Hd)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        ll, info = gp.ops.loglik_batched(xd, Gd, Hd)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    # per-class kernel times from a separate pass: the event pairs around every launch cost 3-4 % on the look-ahead
    # schedules (hundreds of launches on three streams), so they stay out of the timed region
    preps = max(1, min(reps, 3))
    gp.ops.profile(True)
    for _ in range(preps):
        gp.ops.loglik_batched(xd, Gd, Hd)
    torch.cuda.synchronize()
    prof = gp.ops.profile_read()
    gp.ops.profile(False)
    launches = int(sum(v[1] for v in prof.values()))
    flops = B * n ** 3 / 3.0
    ll_h = ll.cpu().numpy()
    idx = np.unique(np.linspace(0, B - 1, min(B, n_check)).astype(int))
    t0 = time.perf_counter()
    ref = np.array([so.loglik_unit(x, G[i], H[i], form='chol') for i in idx])
    cpu_dt = time.perf_counter() - t0
    rel = float(np.max(np.abs(ll_h[idx] - ref) / np.abs(ref)))
    tf_pass = flops / (ms * 1e-3) / 1e12
    rec = {'name': name, 'kind': 'loglik', 'workload': what, 'n': n, 'batch': B, 'ard_dims': ard, 'reps': reps,
           'ms_per_pass': ms, 'evals_per_s': B / (ms * 1e-3), 'failed_items': int((info != 0).sum().item()),
           'roofline': {'bound': 'tensor', 'unit': 'TFLOP/s', 'flop_per_eval': n ** 3 / 3.0,
                        'achieved': tf_pass, 'peak': peak_tf, 'frac': tf_pass / peak_tf if peak_tf else None,
                        'what': 'N^3/3 flop per eval over the WALL time of the whole pass (assembly, reductions, launch gaps included)'},
           'kernel_ms': {k: round(v[0] / preps, 4) for k, v in prof.items() if v[0] > 0},
           'kernel_ms_note': 'from a separate pass with CUDA event pairs around every launch (not the timed passes)',
           'gpu_launches_per_pass': launches // preps,
           'gpu_vs_oracle_max_rel_err': rel, 'oracle_items': [int(i) for i in idx],
           'cpu_oracle_s_per_eval': cpu_dt / len(idx)}
    del xd, Gd, Hd
    return rec


def sub_sds(gp, torch, np, name, n, B, ard, sweeps, start_iter, peak_tf, n_check, what, dist=None, world=1, rank=0, run_mode=False):
    """Device-resident SDS sweeps (whole surrogate_slice_sampling transitions for B chains PER RANK through
    ChainEnsemble): chain-sweeps/s, trips, 4/3 N^3 flop per auxiliary-model evaluation against the DGEMM rate,
    per-rank busy time (trip-count imbalance) and a tape-driven comparison with the oracle on sampled chains."""
    from oracle import sds_oracle as so
    from oracle.reference_loader import Tape
    if ard:
        x, y = gp.synthetic.ard_inputs(n, ard)
        n_ell = ard
    else:
        x, y = gp.synthetic.ih45_series(n)
        n_ell = 1
    P = n_ell + 2
    scale = np.array([gp.synthetic.SCALE[0]] * n_ell + list(gp.synthetic.SCALE[1:]))
    F0, H0 = gp.synthetic.chain_states(B, n, n_ell=n_ell, first_chain=rank * B)

    def one_pass(profile):
        """The same sweeps from the same state and seeds (identical work); with `profile` every launch is bracketed by a
        CUDA event pair -- thousands of them, so the per-class kernel times come from a pass of their own, not the timed one."""
        ens = gp.chains.ChainEnsemble(x, y, F0, H0, scale, seed=1, max_trips=64, sharded_input=True,
                                      distributed=(world > 1))
        ens.sweep(start_iter)                                   # warm-up: allocations, lazy module load, NCCL
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        if profile:
            gp.ops.profile(True)
        busy, trips = [], []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if run_mode:
            # the whole caller loop in ONE device call (gpmc_sds_run): chains advance on their own, one all-gather at the end
            _, _, ntg = ens.run(sweeps, start_iter=start_iter + 1)
            busy.append(ens.last_busy_ms)
            trips = [ntg[:, i] for i in range(sweeps)]
        else:
            for i in range(sweeps):
                Hg, llg, ntg = ens.sweep(start_iter + 1 + i)    # gathered over ranks
                busy.append(ens.last_busy_ms)
                trips.append(ntg)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        prof = gp.ops.profile_read() if profile else None
        if profile:
            gp.ops.profile(False)
        return ms, busy, trips, prof, ens

    ms, busy, trips, _, ens = one_pass(False)
    exhausted_total = int(ens.exhausted_total)
    del ens
    _, _, trips_p, prof, ens = one_pass(True)
    # (same state and seeds; launch sizes follow the polled status words, so schedules -- and the last bits -- may differ)
    repeat_ok = bool(all(np.array_equal(a_, b_) for a_, b_ in zip(trips, trips_p)))
    del ens
    busy_local = float(np.sum(busy))
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        tb = torch.zeros(world, dtype=torch.float64, device='cuda')
        tb[rank] = busy_local
        dist.all_reduce(tb)
        busy_ranks = [float(v) for v in tb.cpu().tolist()]
    else:
        busy_ranks = [busy_local]
    trips = np.stack(trips)                                 # [sweeps, world*B]
    evals = int((trips + 1).sum())                          # aux-model evaluations: one at theta + one per trip
    flops = evals * (4.0 / 3.0) * n ** 3
    tf = flops / (ms * 1e-3) / 1e12
    rec = {'name': name, 'kind': 'sds_run' if run_mode else 'sds_sweep', 'workload': what, 'n': n, 'chains_per_gpu': B, 'chains': world * B,
           'ard_dims': ard, 'sweeps': sweeps, 'start_iter': start_iter + 1,
           's_per_sweep': ms * 1e-3 / sweeps, 'chain_sweeps_per_s': world * B * sweeps / (ms * 1e-3),
           'mean_trips': float(trips.mean()), 'max_trips': int(trips.max()), 'aux_evals': evals,
           'exhausted_chains': exhausted_total,
           'roofline': {'bound': 'tensor', 'unit': 'TFLOP/s', 'flop_per_aux_eval': (4.0 / 3.0) * n ** 3,
                        'achieved': tf, 'peak': peak_tf * world if peak_tf else None,
                        'frac': tf / (peak_tf * world) if peak_tf else None,
                        'what': '4/3 N^3 flop per auxiliary-model evaluation (chol(K+S), U = L^-T, R = S - S U U^T S, chol(R)) '
                                'over the WALL time of the sweeps (control kernels, host round trips, idle tails included)'},
           'busy_ms_per_rank': busy_ranks,
           'imbalance_max_over_mean': (max(busy_ranks) / (sum(busy_ranks) / len(busy_ranks))) if min(busy_ranks) > 0 else None,
           'kernel_ms_rank0': {k: round(v[0], 3) for k, v in prof.items() if v[0] > 0},
           'kernel_ms_note': 'from a repeat of the same sweeps with CUDA event pairs around every launch (not the timed pass)',
           'profiled_pass_same_trip_counts': repeat_ok,
           'gpu_launches_rank0': int(sum(v[1] for v in prof.values()))}
    # ---- parity on sampled chains: tape-driven transition on the device vs the tape-driven oracle (reduced R form, the
    # one the device evaluates): theta' and trip counts exact, log N(g) to 1e-10
    if rank == 0 and n_check > 0:
        F0c, H0c = gp.synthetic.chain_states(n_check, n, n_ell=n_ell, first_chain=7)
        tapes = [Tape.from_seed(4242 + c, n, p=P, max_trips=64) for c in range(n_check)]
        Fd = torch.tensor(F0c).cuda()
        Hd = torch.tensor(H0c).cuda()
        tp = gp.ops.Tape(np.stack([t.z for t in tapes]), np.stack([t.v for t in tapes]), [float(t.u0) for t in tapes],
                         np.stack([t.U for t in tapes]))
        nt, ll, st = gp.ops.sds_sweep(x, y, Fd, Hd, scale, start_iter, tape=tp)
        nt, ll, Hn, Fn = nt.cpu().numpy(), ll.cpu().numpy(), Hd.cpu().numpy(), Fd.cpu().numpy()
        worst_h = worst_ll = worst_f = 0.0
        trips_equal = True
        t0 = time.perf_counter()
        for c in range(n_check):
            tr = so.SweepTrace()
            of, oh = so.surrogate_slice_sampling(F0c[c], x, y, H0c[c], scale, start_iter, tapes[c], trace=tr, r_form='reduced')
            trips_equal = trips_equal and (int(nt[c]) == tr.n_trips)
            worst_h = max(worst_h, float(np.max(np.abs(Hn[c] - oh) / np.abs(oh))))
            worst_ll = max(worst_ll, abs(ll[c] - tr.propG[-1]) / abs(tr.propG[-1]))
            worst_f = max(worst_f, float(np.abs(Fn[c] - of).max()))
        rec['gpu_vs_oracle'] = {'chains': n_check, 'trips_equal': bool(trips_equal), 'theta_max_rel_err': worst_h,
                                'loglik_max_rel_err': float(worst_ll), 'f_max_abs_err': worst_f,
                                'cpu_oracle_s_per_transition': (time.perf_counter() - t0) / n_check,
                                'how': 'tape-driven transition (explicit draws in the reference order) on the device vs oracle/sds_oracle.py'}
    return rec


def sub_predict(gp, torch, np, n=455, S=100, M=40, reps=5, n_check=3):
    """SURVEY row f2: `inf_mcmc` (sliceSample.py:234-284) for S stored samples in ONE device pass (gpmc_predict_batched) --
    the call crossValid.execute makes per fold (framework.py:223-243), IH45-sized series -- against the oracle's per-sample
    restatement timed on the host."""
    from oracle import sds_oracle as so
    rs = np.random.RandomState(77)
    x, y = gp.synthetic.ih45_series(n)
    xs = np.sort(rs.uniform(0, n, size=(M, 1)), axis=0)
    Hyp = np.column_stack([rs.uniform(1.5, 7., S), rs.uniform(2., 9., S), rs.uniform(0.6, 2.8, S)])
    F = (y - y.mean())[:, None] * 0.7 + 0.3 * rs.standard_normal((n, S))
    Ft = np.ascontiguousarray(F.T)
    xd, xsd = torch.tensor(np.asarray(x, dtype=np.float64).reshape(n, -1)).cuda(), torch.tensor(xs).cuda()
    Fd, Hd = torch.tensor(Ft).cuda(), torch.tensor(Hyp).cuda()
    for _ in range(2):
        fmu, fs2, info = gp.ops.predict_batched(xd, xsd, Fd, Hd)
    torch.cuda.synchronize()
    # (the call reads a status word back, so it is sensitive to host load -- e.g. BLAS threads still spinning after the CPU
    #  baseline leg: every call is timed on its own and the median reported, the minimum beside it)
    per_call = []
    for _ in range(max(reps, 9)):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fmu, fs2, info = gp.ops.predict_batched(xd, xsd, Fd, Hd)
        e1.record()
        torch.cuda.synchronize()
        per_call.append(e0.elapsed_time(e1))
    ms = float(np.median(per_call))
    fmu_h, fs2_h = fmu.cpu().numpy(), fs2.cpu().numpy()
    worst_mu = worst_s2 = 0.0
    t0 = time.perf_counter()
    for s_ in range(n_check):
        _, _, _, Fs2, Fmu = so.inf_mcmc_unit(F[:, s_], x, y, xs, Hyp[s_])
        worst_mu = max(worst_mu, float(np.max(np.abs(fmu_h[s_] - Fmu[:, 0]) / np.maximum(np.abs(Fmu[:, 0]), 1e-9))))
        worst_s2 = max(worst_s2, float(np.max(np.abs(np.maximum(fs2_h[s_], 0) - Fs2[:, 0]) / np.maximum(np.abs(Fs2[:, 0]), 1e-10))))
    cpu = (time.perf_counter() - t0) / n_check
    return {'name': 'F2_predict', 'kind': 'predict', 'workload': 'SURVEY row f2: inf_mcmc for %d stored samples x %d test points at N=%d in one '
            'gpmc_predict_batched call (right-hand sides as border rows of the factorisation)' % (S, M, n),
            'n': n, 'samples': S, 'test_points': M, 'reps': len(per_call), 'ms_per_call': ms, 'ms_per_call_min': float(min(per_call)),
            'samples_per_s': S / (ms * 1e-3),
            'failed_items': int((info != 0).sum().item()),
            'gpu_vs_oracle': {'samples': n_check, 'fmu_max_rel_err': worst_mu, 'fs2_max_rel_err': worst_s2, 'cpu_oracle_s_per_sample': cpu}}


def sub_ess(gp, torch, np, n=455, B=1024, updates=9, n_check=2):
    """SURVEY row f4: `elliptical_slice` (sliceSample.py:15-74) as a device path (gpmc_ess_sweep: nu = chol(K) z and the
    whole bracket loop per chain), B chains with their own hyper-parameters; tape-driven check against the oracle."""
    from oracle import sds_oracle as so
    from oracle.reference_loader import EssTape
    rs = np.random.RandomState(78)
    x, y = gp.synthetic.ih45_series(n)
    Hyp = np.column_stack([rs.uniform(2., 6., B), rs.uniform(3., 8., B), rs.uniform(0.8, 2.5, B)])
    F0 = np.tile(0.7 * (y - y.mean()), (B, 1))
    F, Hd = torch.tensor(F0).cuda(), torch.tensor(Hyp).cuda()
    gp.ops.ess_sweep(x, y, F, Hd, it=0, seed=5)
    torch.cuda.synchronize()
    trips = 0.0
    per_update = []
    for it in range(updates):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        nt, st, info = gp.ops.ess_sweep(x, y, F, Hd, it=1 + it, seed=5)
        e1.record()
        torch.cuda.synchronize()
        per_update.append(e0.elapsed_time(e1))
        trips += float(nt.double().mean().item())
    ms = float(np.median(per_update))
    # tape-driven: the N(0, K) draw nu on the tape, decisions and f' against the oracle
    worst = 0.0
    trips_equal = True
    t0 = time.perf_counter()
    for c in range(n_check):
        r2 = np.random.RandomState(900 + c)
        nu = so.ess_nu_from_z(x, Hyp[c], r2.standard_normal(n))
        u, th = r2.random_sample(), r2.random_sample(64)
        of, ot = so.elliptical_slice(F0[c], x, y, Hyp[c], EssTape(nu, u, th))
        Fc = torch.tensor(F0[c][None].copy()).cuda()
        ntc, stc, _ = gp.ops.ess_sweep(x, y, Fc, Hyp[c][None], tape=gp.ops.EssTape([float(u)], th[None], nu=nu[None]), max_trips=64)
        trips_equal = trips_equal and int(ntc.item()) == ot
        worst = max(worst, float(np.abs(Fc.cpu().numpy()[0] - of).max()))
    cpu = (time.perf_counter() - t0) / n_check
    return {'name': 'F4_ess', 'kind': 'ess', 'workload': 'SURVEY row f4: elliptical_slice updates of f for %d chains at N=%d on the device '
            '(gpmc_ess_sweep)' % (B, n), 'n': n, 'chains': B, 'updates': updates, 'ms_per_update': ms, 'ms_per_update_min': float(min(per_update)),
            'chain_updates_per_s': B / (ms * 1e-3), 'mean_proposals_per_update': trips / updates,
            'gpu_vs_oracle': {'chains': n_check, 'trips_equal': bool(trips_equal), 'f_max_abs_err': worst,
                              'cpu_oracle_s_per_update_incl_draw': cpu, 'how': 'nu, u, theta on a tape in the reference order'}}


def sub_c1(gp, np, iters=30, cpu_iters=20, literal=False):
    """BASELINE config 1 (demoRegression.py: N=200, one chain): the reference's caller loop (demoRegression.py:23-30) on
    the drop-in `kcMCMC.sliceSample.surrogate_slice_sampling`, host arrays in / out, global numpy stream seeded like the
    reference (seed 124, hyp0 = [0.35, 2.0, 0.2]); the CPU oracle consumes the same stream beside it."""
    from oracle import sds_oracle as so
    from oracle.reference_loader import Tape
    n = 200
    x, y = gp.synthetic.ih45_series(n)
    scale = np.array([10., 10., 5.])
    sds = gp.kcMCMC.sliceSample
    if literal:
        gp.ops.set_tuning(8, 1)
    try:
        np.random.seed(124)
        f, h = np.zeros(n), np.array([0.35, 2.0, 0.2])
        sds.surrogate_slice_sampling(f, x, y, h, scale, iter=0)             # warm-up
        np.random.seed(124)
        gh = []
        t0 = time.perf_counter()
        for i in range(iters):
            f, h = sds.surrogate_slice_sampling(f, x, y, h, scale, iter=i)
            gh.append(h.copy())
        t_gpu = (time.perf_counter() - t0) / iters
    finally:
        if literal:
            gp.ops.set_tuning(8, 0)
    rs = np.random.RandomState(124)
    f, h = np.zeros(n), np.array([0.35, 2.0, 0.2])
    oh, trips = [], []
    t0 = time.perf_counter()
    for i in range(cpu_iters):
        z, v, u0 = rs.standard_normal(n), rs.random_sample(3), rs.random_sample()
        st = rs.get_state()
        U = rs.random_sample((256, 3))
        tr = so.SweepTrace()
        f, h = so.surrogate_slice_sampling(f, x, y, h, scale, i, Tape(z, v, u0, U), trace=tr)
        rs.set_state(st)
        rs.random_sample((tr.n_trips, 3))
        oh.append(h.copy())
        trips.append(tr.n_trips)
    t_cpu = (time.perf_counter() - t0) / cpu_iters
    gh, oh = np.array(gh), np.array(oh)
    rel = np.abs(gh[:cpu_iters] - oh).max(axis=1) / np.abs(oh).max(axis=1)
    same = int(np.argmax(rel > 1e-9)) if np.any(rel > 1e-9) else cpu_iters
    return {'name': 'C1_chain' + ('_literalR' if literal else ''), 'kind': 'drop_in_chain',
            'workload': 'BASELINE config 1 (demoRegression.py): N=200, one chain, surrogate_slice_sampling called like '
                        'demoRegression.py:25, numpy arrays in and out, global numpy stream',
            'n': n, 'iterations': iters, 'ms_per_iteration': 1e3 * t_gpu, 'cpu_oracle_ms_per_iteration': 1e3 * t_cpu,
            'cpu_oracle_iterations': cpu_iters, 'mean_trips_cpu': float(np.mean(trips)),
            'iterations_with_identical_theta_to_1e-9': same, 'posterior_form': 'literal' if literal else 'reduced'}


def run_b200(args):
    import numpy as np
    import torch
    import gpmc_b200 as gp
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        # NCCL prints its version banner on STDOUT when NCCL_DEBUG=VERSION (the image default); keep stdout for the JSON line
        if os.environ.get('NCCL_DEBUG', 'VERSION').upper() == 'VERSION':
            os.environ['NCCL_DEBUG'] = 'WARN'
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    if args.gemm_cfg is not None:
        gp.ops.set_tuning(0, args.gemm_cfg)
    n, B = args.n, args.chains_per_gpu
    x_h = np.arange(n, dtype=np.float64).reshape(n, 1)
    # chains are keyed by GLOBAL id, so the job's inputs do not depend on how it is sharded
    G_h, H_h = gp.synthetic.loglik_batch(B, n, first_chain=rank * B)
    x = torch.tensor(x_h).cuda()
    G = torch.tensor(G_h).cuda()
    H = torch.tensor(H_h).cuda()
    gathered = torch.empty((world * B,), dtype=torch.float64, device='cuda') if world > 1 else None

    def step():
        ll, info = gp.ops.loglik_batched(x, G, H)
        if world > 1:
            dist.all_gather_into_tensor(gathered, ll)
        return ll, info

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    peaks = {}
    if not args.no_peaks:
        if rank == 0:
            peaks = measured_peaks(torch, gp)
        if world > 1:                                      # every rank needs the DGEMM figure for its sub-records
            t = torch.tensor([peaks.get('cublas_dgemm_8192_tflops', 0.0)], dtype=torch.float64, device='cuda')
            dist.broadcast(t, 0)
            if rank != 0:
                peaks = {'cublas_dgemm_8192_tflops': float(t.item())}

    for _ in range(max(1, args.warmup)):                  # at least one: first-touch allocations, lazy module load
        ll, info = step()
    barrier()
    assert int((info != 0).sum().item()) == 0, 'a factorisation failed on the synthetic workload'

    sampler = ClockSampler(local)
    sampler.start()
    gp.ops.profile(True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        ll, info = step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    prof = gp.ops.profile_read()
    gp.ops.profile(False)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = world * B * args.steps / (ms * 1e-3)
    if args.dump_outputs:
        out = {'loglik': ll, 'info': info}
        if world > 1:
            info_all = torch.empty((world * B,), dtype=torch.int32, device='cuda')
            dist.all_gather_into_tensor(info_all, info)
            out = {'loglik': gathered, 'info': info_all}
        if rank == 0:
            dump_outputs(args.dump_outputs, {k: v.cpu().numpy() for k, v in out.items()})

    # ---- end-to-end through the host-buffer C-ABI call (pinned H2D + D2H every step)
    e2e = None
    if not args.no_e2e:
        for _ in range(min(args.warmup, 2)):
            gp.ops.loglik_host(x_h, G_h, H_h)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            ll_h, info_h = gp.ops.loglik_host(x_h, G_h, H_h)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device='cuda')
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        e2e = {'value': world * B * args.steps / dt, 'unit': UNIT,
               'h2d_bytes_per_step': int(x_h.nbytes + G_h.nbytes + H_h.nbytes),
               'd2h_bytes_per_step': int(B * 8 + B * 4)}
        assert np.array_equal(ll_h, ll.cpu().numpy()), 'host-buffer path and device path disagree'
    ll_first = ll.cpu().numpy()[:max(1, args.cpu_sample)].copy()
    del G, H, gathered

    # ---- sub-records: the other BASELINE configs and the device-resident SDS sweeps (every rank takes part in the
    # SDS C5-shard record so that per-rank busy time and the 1->N curve of the real sampler are visible)
    peak_tf = peaks.get('cublas_dgemm_8192_tflops')
    configs = []
    if not args.no_configs:
        want = set(args.only_configs.split(',')) if args.only_configs else None

        def on(name):
            return want is None or name in want
        try:
            if world == 1:
                if on('C1_chain'):
                    configs.append(sub_c1(gp, np))
                if on('C1_chain_literalR'):
                    configs.append(sub_c1(gp, np, literal=True))
                if on('C2_loglik'):
                    configs.append(sub_loglik(gp, torch, np, 'C2_loglik', 2048, 64, 0, 10, peak_tf, 8,
                                              'BASELINE config 2: IH45-shaped series, N=2048, SE+noise, 64 chains, 1 B200'))
                if on('C3_loglik'):
                    configs.append(sub_loglik(gp, torch, np, 'C3_loglik', 512, 4096, 4, 5, peak_tf, 8,
                                              'BASELINE config 3: N=512, 4096 chains, ARD kernel D=4'))
                if on('C4_loglik'):
                    configs.append(sub_loglik(gp, torch, np, 'C4_loglik', 16384, 1, 0, 3, peak_tf, 1,
                                              'BASELINE config 4: single chain N=16384, blocked Cholesky per step'))
                if on('C2_sds'):
                    configs.append(sub_sds(gp, torch, np, 'C2_sds', 2048, 64, 0, 2, 0, peak_tf, 1,
                                           'BASELINE config 2 shape, whole SDS transitions on the device'))
                if on('C3_sds'):
                    configs.append(sub_sds(gp, torch, np, 'C3_sds', 512, 4096, 4, 2, 0, peak_tf, 2,
                                           'BASELINE config 3: fused on-device slice loop, N=512, 4096 chains, ARD D=4'))
                if on('F2_predict'):
                    configs.append(sub_predict(gp, torch, np))
                if on('F4_ess'):
                    configs.append(sub_ess(gp, torch, np))
            if on('C5_sds'):
                configs.append(sub_sds(gp, torch, np, 'C5_sds', n, 256, 0, 1, 0, peak_tf, 1 if world == 1 else 0,
                                       'BASELINE config 5 shard of the real sampler: N=%d, 256 chains per GPU, whole SDS '
                                       'transitions, chains sharded by GPU, one all-gather per sweep' % n,
                                       dist=dist, world=world, rank=rank))
            if on('C5_sds_run'):
                configs.append(sub_sds(gp, torch, np, 'C5_sds_run', n, 256, 0, 3, 0, peak_tf, 0,
                                       'same shard, 3 MCMC iterations per chain in ONE device call (gpmc_sds_run: the caller loop '
                                       'framework.py:68-75 on the device, no chain waits at an iteration boundary), one all-gather '
                                       'of the history at the end', dist=dist, world=world, rank=rank, run_mode=True))
        except Exception as e:                              # a sub-record must never cost the headline line
            configs.append({'name': 'error', 'error': repr(e)})

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel family: the blocked Cholesky (DMMA update + panel kernels)
    evals_timed = B * args.steps
    chol_flops = n ** 3 / 3.0                                    # SURVEY 8d: algorithmic flops per eval
    chol_ms = chol_kernel_ms(prof)
    gemm_ms, gemm_launches = prof['gemm_update']
    achieved = evals_timed * chol_flops / (chol_ms * 1e-3) / 1e12 if chol_ms > 0 else None
    # executed MACs of the update kernel: full 128-row tiles of every block column
    nb = gp._lib.load().gpmc_panel_width()                          # block-column width of this build (64 or 128)
    nt = (n + nb - 1) // nb
    # DMMA flops the update kernel really issues per factorisation: full 128-row tiles below the diagonal block, 8.5 of
    # the 16 32x32 sub-tiles of the diagonal block (6 skipped, 4 at 10/16), one 8-row fragment for the border row
    exec_flops = sum(2.0 * (j * nb) * nb * (((n - j * nb - nb + 127) // 128 * 128) + 0.53125 * nb + 8) for j in range(1, nt))
    peak = peaks.get('cublas_dgemm_8192_tflops')
    traffic, traffic_src = committed_traffic(n, nb)
    hbm_peak, hbm_src = hbm_peak_gbs()
    roofline = {
        'bound': 'tensor', 'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s',
        'frac': (achieved / peak) if (achieved and peak) else None,
        # DRAM bytes per eval of the dominant kernel (all update launches of one factorisation) from the committed ncu
        # capture of the current kernel (dram__bytes_read.sum + dram__bytes_write.sum), next to the algorithmic bytes
        # (every L row read once per block column + the block column read and written once)
        'traffic': traffic, 'traffic_unit': 'bytes per eval (update kernel)', 'traffic_source': traffic_src,
        'traffic_algorithmic': sum((n - j * nb) * (j * nb) * 8 + 2 * (n - j * nb) * nb * 8 for j in range(1, nt)),
        'peak_source': 'measured in this run: cuBLAS DGEMM 8192^3 FP64 (MEASURED_PEAKS.json has no FP64 figure); '
                       'nominal B200 FP64 tensor 40 TFLOP/s',
        'what': 'batched blocked Cholesky (TMA-staged DMMA update kernel + potf2 + panel solve launches), N^3/3 flop per eval '
                'over the summed CUDA-event durations of those launches on their stream',
        'frac_of_nominal_40tf': (achieved / 40.0) if achieved else None,
        'whole_step': {'tflops': world * evals_timed * chol_flops / (ms * 1e-3) / 1e12 / world,
                       'frac': (evals_timed * chol_flops / (ms * 1e-3) / 1e12 / peak) if peak else None,
                       'what': 'N^3/3 flop per eval over the wall time of the step (assembly and reductions included), per GPU'},
        'update_kernel': {'ms_total': gemm_ms, 'launches': gemm_launches,
                          'executed_tflops': evals_timed * exec_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else None},
        'kernel_ms': {k: v[0] for k, v in prof.items()},
        'assemble': {'bytes_per_eval': 8.0 * n * (n + 64) / 2, 'ms_total': prof['assemble'][0],
                     'achieved_gbs': evals_timed * 8.0 * n * (n + 64) / 2 / (prof['assemble'][0] * 1e-3) / 1e9 if prof['assemble'][0] > 0 else None,
                     'hbm_peak_gbs': hbm_peak, 'hbm_peak_source': hbm_src},
        'measured_fp64': peaks,
    }

    cpu = None
    if not args.no_cpu_baseline and world == 1:        # the CPU arm is reported at N=1 only
        threads = effective_blas_threads()
        v_inv, dt_inv, vals = cpu_unit_evals_per_s(n, args.cpu_sample, 'inv')
        v_chol, dt_chol, vals_c = cpu_unit_evals_per_s(n, args.cpu_sample, 'trsv')
        got = ll_first[:args.cpu_sample]
        relerr = float(np.max(np.abs(got - np.asarray(vals_c)) / np.abs(np.asarray(vals_c))))
        cpu = {'value': v_inv, 'unit': UNIT, 'cores': threads, 'host_cpus': os.cpu_count(), 'kind': 'port',
               'sample': '%d evals at N=%d of the same workload (rank 0 chains 0..%d): oracle port of sliceSample.py:136-147 '
                         'as written (dense inv), numpy/scipy OpenBLAS, %d threads in effect' % (args.cpu_sample, n, args.cpu_sample - 1, threads),
               'restated_unit_value': v_chol, 'restated_unit': 'cdist+exp, dpotrf, one solve_triangular, log-diag',
               'gpu_vs_oracle_max_rel_err': relerr}

    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f64', 'data': 'synthetic',
        'config': workload_config(n, B, world),
        'clocks': clocks, 'e2e': e2e, 'gpu_launches': int(sum(v[1] for v in prof.values())),
        'roofline': roofline, 'cpu_baseline': cpu, 'configs': configs,
    }
    sys.stdout.flush()
    emit(line)
    if world > 1:
        dist.destroy_process_group()


DUMP_LIMIT_BYTES = 60 * 10 ** 6          # data bytes: with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir, arrays):
    """Write ``arrays`` (name -> 1-D array over chains) as float64 ``out_dir/<name>.npy``.  Above DUMP_LIMIT_BYTES in all, every
    array keeps the same fixed, seeded sample of chains, whose indices are written beside them as ``sample_index.npy``."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    if 8 * n * len(arrays) > DUMP_LIMIT_BYTES:
        keep = DUMP_LIMIT_BYTES // (8 * (len(arrays) + 1))
        idx = np.sort(np.random.RandomState(0).choice(n, keep, replace=False))
        arrays = dict({k: a[idx] for k, a in arrays.items()}, sample_index=idx.astype(np.float64))
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), a)


_REAL_STDOUT = None


def protect_stdout():
    """The driver reads ONE JSON line from stdout.  Libraries write there too (NCCL prints its version banner on stdout
    at NCCL_DEBUG=VERSION/WARN), so file descriptor 1 is pointed at stderr for the whole run and the JSON line goes to
    a private duplicate of the original stdout."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), 'w')
    os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + '\n')
    out.flush()


def main():
    args = parse()
    set_blas_threads()                   # before numpy/scipy load their BLAS (both arms time a CPU sample)
    protect_stdout()
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if args.impl == 'reference':
        run_reference(args, rank, world)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
