"""Many independent SDS chains on one or more B200s.

The reference runs ONE chain (``framework.py:59-77``: ``for i in range(iters): propF, propHyp =
surrogate_slice_sampling(...)``).  Chains share nothing but the read-only data ``(x, y)``, so an ensemble of B
chains is the same loop with a batch dimension: the whole transition of every chain is one call into
``gpmc_sds_sweep``.  With ``torch.distributed`` initialised, chains are sharded contiguously over ranks (chain c on
rank ``c // (B / world)``), every rank sweeps only its shard, and the per-chain samples ``[theta, loglik, ntrips]``
are all-gathered once per sweep -- the only collective on the path (SURVEY 8e).  RNG streams are keyed by GLOBAL chain
id, so the samples do not depend on the number of ranks.
"""
import numpy as np

from . import ops


def shard_bounds(n_chains, world, rank):
    """Contiguous shard ``[lo, hi)`` of rank ``rank``; sizes differ by at most one."""
    base, rem = divmod(n_chains, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class ChainEnsemble(object):
    """B chains of the surrogate-data slice sampler over shared data ``(x, y)``.

    ``F0[B,N]``/``Hyp0[B,P]`` are the GLOBAL initial states (every rank passes the same arrays, or only its shard
    with ``sharded_input=True``); ``sweep(it)`` advances every local chain by one transition and returns the gathered
    ``(Hyp[B,P], loglik[B], ntrips[B])`` as numpy arrays on every rank.

    ``likelihood='gauss'``: the chains sample the hyper-parameters of GP regression with a Gaussian likelihood, the
    latent f integrated out (``ops.marginal_run``; ``F0`` may be None, loglik is ``log N(y - mean(y); 0, K + S)``, and
    ``burn_in`` is the iteration up to which the noise stays frozen).  ``'tg2'`` (default) is the surrogate-data slice
    sampler of the reference's truncated-Gaussian model."""

    def __init__(self, x, y, F0, Hyp0, scale, seed=0, max_trips=64, sweeper=None, gather_f=False, sharded_input=False,
                 distributed=True, strict=False, kind=None, likelihood='tg2', burn_in=500):
        self.x = np.asarray(x, dtype=np.float64)
        if self.x.ndim == 1:
            self.x = self.x.reshape(-1, 1)
        self.y = np.asarray(y, dtype=np.float64).reshape(-1)
        self.my = float(np.mean(self.y))                       # sliceSample.py:102
        self.scale = np.asarray(scale, dtype=np.float64).reshape(-1)
        self.seed, self.max_trips, self.gather_f = int(seed), int(max_trips), gather_f
        self.kind = kind                   # covariance kind (ops.KIND_*); None: SE iso / ARD from the width of Hyp0
        if likelihood not in ('tg2', 'gauss'):
            raise ValueError("likelihood must be 'tg2' or 'gauss'")
        self.likelihood, self.burn_in = likelihood, int(burn_in)
        # A chain whose slice does not close within ``max_trips`` proposals keeps its state and is reported with
        # status 1 (the reference's ``while True`` would loop on, or raise LinAlgError out of jitchol when the
        # factorisation at the current state is the reason).  ``strict`` turns that into an exception; otherwise the
        # ensemble counts such transitions (``exhausted_total``) and warns once per sweep.
        self.strict = bool(strict)
        self.exhausted_total = 0
        self.last_status = None            # gathered status[B] of the last sweep (0 accepted, 1 trip budget used up)
        self.last_busy_ms = None           # device time of this rank's local sweep (CUDA events), None for test doubles
        self.dist = None
        self.rank, self.world = 0, 1
        try:
            import torch.distributed as dist
            if distributed and dist.is_available() and dist.is_initialized():
                self.dist, self.rank, self.world = dist, dist.get_rank(), dist.get_world_size()
        except ImportError:
            pass
        F0 = None if F0 is None and likelihood == 'gauss' else np.asarray(F0, dtype=np.float64)
        Hyp0 = np.asarray(Hyp0, dtype=np.float64)
        if sharded_input:
            self.n_local = Hyp0.shape[0]
            counts = self._all_counts(self.n_local)
            self.n_chains = int(sum(counts))
            self.lo = int(sum(counts[:self.rank]))
            self.hi = self.lo + self.n_local
            self._counts = counts
        else:
            self.n_chains = Hyp0.shape[0]
            self.lo, self.hi = shard_bounds(self.n_chains, self.world, self.rank)
            self.n_local = self.hi - self.lo
            self._counts = [shard_bounds(self.n_chains, self.world, r)[1] - shard_bounds(self.n_chains, self.world, r)[0]
                            for r in range(self.world)]
            F0, Hyp0 = (None if F0 is None else F0[self.lo:self.hi]), Hyp0[self.lo:self.hi]
        self.P = Hyp0.shape[1]
        # the sweeper is the device path; tests of the host logic inject their own (gloo, no GPU)
        self._sweeper = sweeper or (_MarginalSweeper(self) if likelihood == 'gauss' else _DeviceSweeper(self))
        self._sweeper.load(F0, Hyp0)

    def _all_counts(self, n_local):
        if self.dist is None:
            return [n_local]
        import torch
        t = torch.zeros(self.world, dtype=torch.int64)
        t[self.rank] = n_local
        if self.dist.get_backend() == 'nccl':
            t = t.cuda()
        self.dist.all_reduce(t)
        return [int(v) for v in t.cpu().tolist()]

    def sweep(self, it):
        """One transition of every chain at MCMC iteration ``it``; returns gathered ``(Hyp, loglik, ntrips)``."""
        res = self._sweeper.sweep(it)                          # local shard, [n_local, ...] tensors/arrays
        hyp, ll, nt = res[0], res[1], res[2]
        status = res[3] if len(res) > 3 else None              # test doubles may not report a status
        self.last_busy_ms = getattr(self._sweeper, 'last_busy_ms', None)
        H, LL, NT, ST = self._gather(hyp, ll, nt, status)
        self.last_status = ST
        n_bad = int((ST != 0).sum())
        if n_bad:
            self.exhausted_total += n_bad
            msg = ('%d of %d chains did not close their slice within max_trips=%d proposals at iteration %d (state kept; '
                   'first: chain %d)' % (n_bad, self.n_chains, self.max_trips, it, int(np.flatnonzero(ST)[0])))
            if self.strict:
                raise RuntimeError(msg)
            import warnings
            warnings.warn(msg, RuntimeWarning)
        return H, LL, NT

    def local_state(self):
        return self._sweeper.state()

    # ---- checkpoint / resume (the reference only writes CSV files at the very end, framework.py:79-122: a crash loses the
    # chain).  Randomness is keyed by (seed, global chain id, iteration), so the state of a run is just (f, theta) of every
    # chain plus the next iteration: a resumed run continues bit for bit.
    def save(self, path, next_iter):
        """Write this rank's shard (``<path>.rank<r>.npz``): chain states, shard bounds, seed, next iteration."""
        F, H = self.local_state()
        np.savez(('%s.rank%d.npz' % (path, self.rank)), F=F, H=H, lo=self.lo, hi=self.hi, n_chains=self.n_chains,
                 seed=self.seed, next_iter=int(next_iter), scale=self.scale, max_trips=self.max_trips)

    @classmethod
    def resume(cls, path, x, y, **kw):
        """Rebuild the ensemble from files written by :meth:`save` (same number of ranks).  Returns ``(ensemble, next_iter)``."""
        rank = 0
        try:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized():
                rank = dist.get_rank()
        except ImportError:
            pass
        z = np.load('%s.rank%d.npz' % (path, rank))
        ens = cls(x, y, z['F'], z['H'], z['scale'], seed=int(z['seed']), max_trips=int(z['max_trips']), sharded_input=True, **kw)
        if (ens.lo, ens.hi, ens.n_chains) != (int(z['lo']), int(z['hi']), int(z['n_chains'])):
            raise ValueError('checkpoint was written with a different sharding: [%d, %d) of %d, now [%d, %d) of %d' % (
                int(z['lo']), int(z['hi']), int(z['n_chains']), ens.lo, ens.hi, ens.n_chains))
        return ens, int(z['next_iter'])

    def _gather(self, hyp, ll, nt, status=None):
        import torch
        P = self.P
        ll_t = torch.as_tensor(ll, dtype=torch.float64).reshape(self.n_local, 1)
        st_t = torch.zeros_like(ll_t) if status is None else torch.as_tensor(status).to(ll_t.device, torch.float64).reshape(self.n_local, 1)
        pack = torch.cat([torch.as_tensor(hyp, dtype=torch.float64).reshape(self.n_local, P), ll_t,
                          torch.as_tensor(nt).to(torch.float64).reshape(self.n_local, 1), st_t], dim=1)
        if self.dist is None:
            out = pack
        else:
            # ONE all-gather of [theta, loglik, ntrips, status] per sweep; shards may differ by one chain, so pad to the max
            mx = max(self._counts)
            buf = torch.zeros((mx, P + 3), dtype=torch.float64, device=pack.device)
            buf[:self.n_local] = pack
            full = torch.empty((self.world * mx, P + 3), dtype=torch.float64, device=pack.device)
            self.dist.all_gather_into_tensor(full, buf)
            out = torch.cat([full[r * mx: r * mx + c] for r, c in enumerate(self._counts)], dim=0)
        out = out.cpu().numpy()
        return out[:, :P].copy(), out[:, P].copy(), out[:, P + 1].astype(np.int64), out[:, P + 2].astype(np.int64)

    def run(self, iters, start_iter=0, thin_f=0, gather_every=None):
        """The caller loop of ``framework.py:68-75`` for the ensemble: returns ``histHyp[B, P, iters]``,
        ``histLL[B, iters]``, ``trips[B, iters]`` (and the local ``histF[n_local, N, kept]`` when ``thin_f > 0``).

        With the device sweeper the loop itself runs on the GPU (``gpmc_sds_run``): every chain of the shard goes through
        its iterations back to back, and the ranks exchange their history in ONE all-gather per ``gather_every`` iterations
        (default: once, at the end).  A sweeper without ``run`` (the CPU test double) is driven one sweep at a time."""
        B, P = self.n_chains, self.P
        histHyp = np.zeros((B, P, iters))
        histLL = np.zeros((B, iters))
        trips = np.zeros((B, iters), dtype=np.int64)
        keepF = []
        if hasattr(self._sweeper, 'run') and iters > 0:
            step = iters if not gather_every else max(1, int(gather_every))
            for i0 in range(0, iters, step):
                k = min(step, iters - i0)
                # thinning is relative to the start of the run: keep f after iterations 0, thin_f, 2 thin_f, ...
                hh, ll, nt, hf, n_exh = self._sweeper.run(start_iter + i0, k, thin_f, (-i0) % thin_f if thin_f else 0)
                self.last_busy_ms = getattr(self._sweeper, 'last_busy_ms', None)
                G = self._gather_block(hh, ll, nt)                         # [B, k, P + 2]
                histHyp[:, :, i0:i0 + k] = np.transpose(G[:, :, :P], (0, 2, 1))
                histLL[:, i0:i0 + k] = G[:, :, P]
                trips[:, i0:i0 + k] = G[:, :, P + 1].astype(np.int64)
                if hf is not None:
                    keepF.append(hf)
                if n_exh:
                    self.exhausted_total += n_exh
                    msg = '%d transitions of this rank\'s chains did not close their slice within max_trips=%d proposals (state kept)' % (n_exh, self.max_trips)
                    if self.strict:
                        raise RuntimeError(msg)
                    import warnings
                    warnings.warn(msg, RuntimeWarning)
            if thin_f:
                return histHyp, histLL, trips, np.concatenate(keepF, axis=-1)
            return histHyp, histLL, trips
        for i in range(iters):
            h, ll, nt = self.sweep(start_iter + i)
            histHyp[:, :, i], histLL[:, i], trips[:, i] = h, ll, nt
            if thin_f and (i % thin_f == 0):
                keepF.append(self.local_state()[0])
        if thin_f:
            return histHyp, histLL, trips, np.stack(keepF, axis=-1)
        return histHyp, histLL, trips

    def _gather_block(self, hh, ll, nt):
        """All-gather of a block of history ``[n_local, k, P + 2]`` -> ``[B, k, P + 2]`` (numpy) on every rank."""
        import torch
        P = self.P
        k = hh.shape[1]
        pack = torch.cat([hh, ll.reshape(self.n_local, k, 1), nt.to(torch.float64).reshape(self.n_local, k, 1)], dim=2).contiguous()
        if self.dist is None:
            return pack.cpu().numpy()
        mx = max(self._counts)
        buf = torch.zeros((mx, k, P + 2), dtype=torch.float64, device=pack.device)
        buf[:self.n_local] = pack
        full = torch.empty((self.world * mx, k, P + 2), dtype=torch.float64, device=pack.device)
        self.dist.all_gather_into_tensor(full, buf)
        out = torch.cat([full[r * mx: r * mx + c] for r, c in enumerate(self._counts)], dim=0)
        return out.cpu().numpy()


class _DeviceSweeper(object):
    """Holds the shard's chain state in HBM and advances it with ``gpmc_sds_sweep``."""

    def __init__(self, ens):
        self.ens = ens

    def load(self, F0, Hyp0):
        import torch
        self.torch = torch
        self.F = torch.tensor(np.ascontiguousarray(F0)).cuda()
        self.H = torch.tensor(np.ascontiguousarray(Hyp0)).cuda()
        self.x = torch.tensor(self.ens.x).cuda()
        self.y = torch.tensor(self.ens.y).cuda()
        self.scale = torch.tensor(self.ens.scale).cuda()

    def sweep(self, it):
        e = self.ens
        torch = self.torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        nt, ll, status = ops.sds_sweep(self.x, self.y, self.F, self.H, self.scale, it, my=e.my, seed=e.seed,
                                       chain0=e.lo, max_trips=e.max_trips, kind=e.kind)
        e1.record()
        e1.synchronize()
        self.last_busy_ms = e0.elapsed_time(e1)
        return self.H, ll, nt, status

    def run(self, it0, n_iters, thin_f=0, thin_phase=0):
        """``n_iters`` transitions of every local chain on the device; returns device history tensors and the local
        ``histF[n_local, N, kept]`` (numpy) when ``thin_f > 0`` (f after the iterations ``thin_phase, thin_phase + thin_f, ...``
        of this block)."""
        e = self.ens
        torch = self.torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if thin_f and thin_phase:
            # blocks that do not start on a kept iteration: run up to the next kept one first
            raise ValueError('gather_every must be a multiple of thin_f')
        hh, ll, nt, hf, n_exh = ops.sds_run(self.x, self.y, self.F, self.H, self.scale, it0, n_iters, my=e.my, seed=e.seed,
                                            chain0=e.lo, max_trips=e.max_trips, keep_f_every=thin_f, kind=e.kind)
        e1.record()
        e1.synchronize()
        self.last_busy_ms = e0.elapsed_time(e1)
        histF = None if hf is None else np.transpose(hf.cpu().numpy(), (0, 2, 1))
        return hh, ll, nt, histF, n_exh

    def state(self):
        return self.F.cpu().numpy(), self.H.cpu().numpy()


class _MarginalSweeper(_DeviceSweeper):
    """``likelihood='gauss'``: holds the shard's hyper-parameters in HBM and advances them with ``gpmc_marginal_run``."""

    def load(self, F0, Hyp0):
        super().load(np.zeros((Hyp0.shape[0], 0)) if F0 is None else F0, Hyp0)

    def _call(self, it0, n_iters):
        e = self.ens
        torch = self.torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = ops.marginal_run(self.x, self.y, self.H, self.scale, it0, n_iters, m=e.my, burn_in=e.burn_in, seed=e.seed,
                               chain0=e.lo, max_trips=e.max_trips, kind=e.kind)
        e1.record()
        e1.synchronize()
        self.last_busy_ms = e0.elapsed_time(e1)
        return out

    def sweep(self, it):
        hh, ll, nt, exh = self._call(it, 1)
        return self.H, ll[:, 0], nt[:, 0], (exh != 0).to(self.torch.int32)

    def run(self, it0, n_iters, thin_f=0, thin_phase=0):
        if thin_f:
            raise ValueError("likelihood='gauss' has no latent f to keep")
        hh, ll, nt, exh = self._call(it0, n_iters)
        # transitions that kept their state: budget used up, or every transition of a chain that cannot start
        n_exh = int(exh.clamp(min=0).sum().item()) + n_iters * int((exh < 0).sum().item())
        return hh, ll, nt, None, n_exh
