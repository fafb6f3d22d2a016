"""Worker of tests/test_marginal_oracle.py: world_size-2 run of ChainEnsemble(likelihood='gauss') on CPU (gloo).

The device sweeper is replaced by a test double that advances the hyper-parameters with the marginal oracle, with tapes
keyed by global chain id, so what is exercised is the multi-rank plumbing: sharding, F0 = None, and one all-gather per
block of iterations."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import gpmc_b200 as gp                                   # noqa: E402
from oracle import marginal_oracle as mo                 # noqa: E402
from oracle import sds_oracle as so                      # noqa: E402


def tape(seed, P, T=64):
    rng = np.random.default_rng(seed)
    return rng.uniform(size=P), rng.uniform(), rng.uniform(size=(T, P))


class OracleMarginalSweeper(object):
    """Test double for chains._MarginalSweeper: same interface, marginal oracle inside."""

    def __init__(self, x, y, scale, seed, lo, burn_in=0):
        self.x, self.y, self.scale, self.seed, self.lo, self.burn_in = x, y, scale, seed, lo, burn_in
        self.r = y - np.mean(y)

    def load(self, F0, Hyp0):
        assert F0 is None
        self.H = Hyp0.copy()
        k, th = so.prior_constants(self.H.shape[1] - 2)
        self.prior = (k, th)
        self.G = np.array([mo.loglik(self.x, self.r, h) for h in self.H])

    def sweep(self, it):
        nt = np.zeros(self.H.shape[0], dtype=np.int64)
        for c in range(self.H.shape[0]):
            v, u0, U = tape(self.seed + 100000 * (self.lo + c) + it, self.H.shape[1])
            self.H[c], self.G[c], nt[c], _ = mo.transition(self.x, self.r, self.H[c], self.G[c], self.scale, it, self.burn_in,
                                                           v, u0, U, *self.prior)
        return self.H.copy(), self.G.copy(), nt

    def run(self, it0, n_iters, thin_f=0, thin_phase=0):
        hh = np.zeros((self.H.shape[0], n_iters, self.H.shape[1]))
        ll = np.zeros((self.H.shape[0], n_iters))
        nt = np.zeros((self.H.shape[0], n_iters), dtype=np.int64)
        for k in range(n_iters):
            hh[:, k], ll[:, k], nt[:, k] = self.sweep(it0 + k)
        return torch.tensor(hh), torch.tensor(ll), torch.tensor(nt), None, 0

    def state(self):
        return None, self.H.copy()


def main():
    dist.init_process_group('gloo')
    rank, world = dist.get_rank(), dist.get_world_size()
    n, B, iters = 12, 5, 4
    x = np.linspace(0, 3, n).reshape(-1, 1)
    y = 2 * np.sin(2 * x[:, 0]) + 5 + 0.3 * np.random.default_rng(3).standard_normal(n)
    scale = np.array([2.0, 3.0, 2.0])
    H0 = np.tile([0.8, 1.5, 0.5], (B, 1)) * (1 + 0.1 * np.arange(B))[:, None]
    lo, hi = gp.chains.shard_bounds(B, world, rank)
    ens = gp.chains.ChainEnsemble(x, y, None, H0, scale, seed=7, likelihood='gauss', burn_in=0,
                                  sweeper=OracleMarginalSweeper(x, y, scale, 7, lo))
    assert (ens.lo, ens.hi) == (lo, hi) and ens.n_chains == B and ens.world == world
    hist, ll, trips = ens.run(iters, gather_every=3)
    solo = OracleMarginalSweeper(x, y, scale, 7, 0)
    solo.load(None, H0)
    for i in range(iters):
        H, l, t = solo.sweep(i)
        assert np.array_equal(hist[:, :, i], H), (rank, i)
        assert np.array_equal(ll[:, i], l) and np.array_equal(trips[:, i], t)
    dist.barrier()
    if rank == 0:
        print('GLOO_MARGINAL_OK')
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
