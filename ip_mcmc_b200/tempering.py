"""Replica exchange (parallel tempering) for Burgers chains.  Not in the reference.

    pt = ParallelTemperingSampler(proposer, accepter, rng, geometric_inv_temps(4, 0.05), swap_interval=10)
    samples = pt.run(np.zeros(3), n_samples, burn_in, sample_interval, n_ladders=256)   # [256, n_samples, d]

A ladder is K chains whose likelihoods are tempered by inverse temperatures 1 = t_0 > t_1 > ... > t_{K-1} >= 0:
rung k accepts with exp((t_k Phi(u) + reg_u) - (t_k Phi(v) + reg_v)).  After every `swap_interval` steps
adjacent rungs exchange states with a Metropolis test (even-odd pairing), so hot rungs carry states across
barriers to the t = 1 rung, the only one that samples the posterior.  The batch is n_ladders x K chains,
ladder-major (DESIGN.md section 4.4); swap rounds run between launches, on the device (ipmcmc_swap_replicas).
"""
import numpy as np
import torch

from . import _lib
from . import accepter as _acc
from . import diagnostics as _diag
from .engine import ChainBatch, F64, _ptr, _stream
from .sampler import MCMCSampler, run_recording


def geometric_inv_temps(K, t_min):
    """K inverse temperatures 1 = t_0 > ... > t_{K-1} = t_min in geometric progression (0 < t_min < 1)."""
    K = int(K)
    if K < 2 or not (0 < t_min < 1):
        raise ValueError("geometric_inv_temps needs K >= 2 and 0 < t_min < 1, got K=%d t_min=%r" % (K, t_min))
    t = np.float64(t_min) ** (np.arange(K, dtype=np.float64) / (K - 1))
    t[0], t[-1] = 1.0, t_min
    return t


class ParallelTemperingSampler:
    """MCMCSampler's interface over ladders of tempered chains (Burgers forward models only: the Lorenz operator
    carries its initial condition from solve to solve, so Phi(u) is not a function of u and a swap is not a valid
    Metropolis move for it)."""

    def __init__(self, proposal, acceptance, rng, inv_temps, swap_interval=10):
        t = np.asarray(inv_temps, dtype=np.float64).reshape(-1)
        if t.size < 2:
            raise ValueError("a ladder needs at least 2 inverse temperatures")
        if not np.all(np.isfinite(t)):
            raise ValueError("inv_temps must be finite")
        if t[0] != 1.0:
            raise ValueError("inv_temps must start at 1.0 (the rung that samples the posterior), got %r" % t[0])
        if not np.all(np.diff(t) < 0):
            raise ValueError("inv_temps must be strictly decreasing")
        if t[-1] < 0:
            raise ValueError("inv_temps must end >= 0")
        if int(swap_interval) < 1:
            raise ValueError("swap_interval must be >= 1")
        self.inv_temps = t
        self.K = t.size
        self.swap_interval = int(swap_interval)
        self._sampler = MCMCSampler(proposal, acceptance, rng)
        self.last_run = None

    @property
    def accepter(self):
        return self._sampler.accepter

    def run(self, u_0, n_samples, burn_in=1000, sample_interval=200, n_ladders=None, chain_offset=0,
            steps_per_launch=None, all_rungs=False, return_device=False, diagnostics=False):
        """Same step accounting as MCMCSampler.run.  u_0: (d,), (n_ladders, d) (every rung of a ladder starts there)
        or (n_ladders, K, d); n_ladders defaults to 1 or to u_0's leading dimension.  chain_offset: global id of
        local chain 0, a multiple of K (a shard holds whole ladders).  Swap round r runs after global step
        (r + 1) * swap_interval; launches end there and every `steps_per_launch` steps (results do not depend on it).

        Returns the t = 1 rung's samples [n_ladders, n_samples, d], or every rung's [n_ladders, K, n_samples, d]
        with `all_rungs` (the device records every rung either way).  `self.last_run` holds the t = 1 rung's pooled
        moments and counters, per-rung counters, swap acceptance per adjacent pair, round trips, the final replica
        ids and, with `diagnostics`, diagnostics.chain_diagnostics of the t = 1 rung."""
        K = self.K
        if sample_interval < 1:
            raise ValueError("sample_interval must be >= 1")
        if diagnostics and n_samples < 4:
            raise ValueError("diagnostics=True needs at least 4 samples per chain (split-R-hat), got %d" % n_samples)
        if chain_offset < 0 or chain_offset % K:
            raise ValueError("chain_offset=%d is not a multiple of the ladder size %d: a ladder would be split across "
                             "shards" % (chain_offset, K))
        u0 = u_0 if torch.is_tensor(u_0) else torch.as_tensor(np.asarray(u_0, dtype=np.float64))
        u0 = u0.to(F64)
        if n_ladders is None:
            n_ladders = 1 if u0.ndim == 1 else u0.shape[0]
        L = int(n_ladders)
        d = u0.shape[-1]
        if u0.ndim == 1:
            u0 = u0.reshape(1, 1, d).expand(L, K, d)
        elif u0.ndim == 2 and u0.shape[0] == L:
            u0 = u0.reshape(L, 1, d).expand(L, K, d)
        elif not (u0.ndim == 3 and tuple(u0.shape[:2]) == (L, K)):
            raise ValueError("u_0 has shape %s, expected (d,), (%d, d) or (%d, %d, d)" % (tuple(u0.shape), L, L, K))
        pre = max(0, burn_in - sample_interval)
        total = pre + n_samples * sample_interval
        spec, pot, a = self._sampler._compile(total, burn_in, sample_interval, None)
        if pot.G.stateful:
            raise ValueError("replica exchange needs a deterministic forward model (Phi(u) a function of u); "
                             "the Lorenz operator carries its initial condition")
        if isinstance(self.accepter, _acc.CountedAccepter):
            self.accepter.reset()
        problem = pot.problem()
        dev = problem.device
        B = L * K
        chains = ChainBatch(problem, u0.reshape(B, d), n_chains=B, chain_offset=chain_offset)
        chains.inv_temp = torch.as_tensor(np.tile(self.inv_temps, L)).to(dev)
        replica = torch.stack([torch.arange(K, dtype=torch.int32).repeat(L), torch.zeros(B, dtype=torch.int32)],
                              dim=1).to(dev).contiguous()
        swap_counts = torch.zeros((L, K - 1, 2), dtype=torch.int64, device=dev)
        round_trips = torch.zeros((L,), dtype=torch.int64, device=dev)
        trace = torch.empty((B, n_samples, d), dtype=F64, device=dev)

        def swap_round(step):
            chains.swap(K, spec.seed, step // self.swap_interval - 1, replica, swap_counts, round_trips)

        run_recording(chains, spec, total, pre, sample_interval, trace, steps_per_launch, self.swap_interval, swap_round)

        # the t = 1 rung: pooled moments and counters over its chains
        cold = [x[::K].contiguous() for x in (chains.mom_count, chains.mom_mean, chains.mom_m2, chains.counters)]
        pooled = torch.empty((2 * d + 1 + _lib.N_COUNTERS,), dtype=F64, device=dev)
        _lib.check(problem.lib.ipmcmc_pool_moments(L, d, *[_ptr(x) for x in cold], _ptr(pooled), None, 0, _stream()))
        chains.launches += 2
        pooled_h = pooled.cpu().numpy()
        sc = swap_counts.sum(dim=0).cpu().numpy()
        self.last_run = dict(
            n_ladders=L, ladder_size=K, inv_temps=self.inv_temps.copy(), swap_interval=self.swap_interval,
            total_steps=total, launches=chains.launches, seed=spec.seed,
            pooled_count=pooled_h[0], pooled_mean=pooled_h[1:1 + d],
            pooled_var=pooled_h[1 + d:1 + 2 * d] / max(pooled_h[0] - 1, 1),
            counters=dict(zip(ChainBatch.COUNTER_NAMES, pooled_h[1 + 2 * d:].astype(np.int64))),
            rung_counters=chains.counters.view(L, K, _lib.N_COUNTERS).sum(dim=0).cpu().numpy(),
            per_chain_counters=chains.counters, swap_counts=swap_counts,
            swap_acceptance=sc[:, 1] / np.maximum(sc[:, 0], 1),
            round_trips=int(round_trips.sum().item()), replica=replica[:, 0].reshape(L, K).cpu().numpy(),
            chains=chains, u=chains.u, phi=chains.phi)
        cn = self.last_run["counters"]
        _acc.credit_counters(a, cn["calls"], cn["accepts"], cn["constraint_rejects"])
        if diagnostics:
            self.last_run["diagnostics"] = _diag.chain_diagnostics(trace[::K])
        res = trace.view(L, K, n_samples, d) if all_rungs else trace[::K]
        if return_device:
            return res
        return res.cpu().numpy()
