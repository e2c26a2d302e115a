"""MCMCSampler with the reference's interface (ip_mcmc/ip_mcmc/sampler.py:6-54), driving the
fused CUDA Metropolis kernel instead of a Python loop.

    sampler = MCMCSampler(proposer, accepter, rng)
    samples = sampler.run(u_0, n_samples, burn_in=1000, sample_interval=200)      # [n_samples, d]
    samples = sampler.run(u_0, n_samples, 0, 1, n_chains=4096)                    # [4096, n_samples, d]

Differences that are inherent to batching (documented in DESIGN.md):
  * randomness comes from Philox4x32-10 streams keyed by (seed, global chain id); the seed is
    drawn from `rng` (one `rng.integers` call), so a run is reproducible from the rng's seed;
  * nothing is printed per sample (the reference prints a line per sample, sampler.py:24).
"""
import numpy as np
import torch

from . import _lib
from . import accepter as _acc
from . import diagnostics as _diag
from . import stats as _stats
from .engine import ChainBatch, SamplerSpec, F64
from .potential import EvolutionPotential
from .proposer import _GaussianStepProposer


def run_recording(chains, spec, total, pre, sample_interval, trace, steps_per_launch=None, every=None,
                  at_boundary=None):
    """Advance a fresh `chains` by `total` steps, recording sample i of every chain into trace[:, i] (the step
    accounting of MCMCSampler.run: `pre` unrecorded steps, then one sample every `sample_interval` steps).  One
    launch unless it is cut: launches end every `steps_per_launch` steps and, when `every` is given, at every
    multiple of `every` steps, after which at_boundary(step) runs.  A cut launch records into its own slice."""
    def recorded_before(x):          # samples recorded by global steps < x
        return max(0, x - pre) // sample_interval

    done = 0
    while True:
        n = total - done
        if steps_per_launch is not None:
            n = min(n, steps_per_launch)
        if every is not None:
            n = min(n, every - done % every)
        if n == total:
            chains.run(spec, total, trace=trace)
        else:
            r0, r1 = recorded_before(done), recorded_before(done + n)
            sub = None
            if r1 > r0:
                sub = torch.empty((chains.n, r1 - r0, chains.d), dtype=F64, device=trace.device)
            chains.run(spec, n, trace=sub)
            if sub is not None:
                trace[:, r0:r1] = sub
        done += n
        if every is not None and done > 0 and done % every == 0:
            at_boundary(done)
        if done >= total:
            return


class MCMCSampler:
    def __init__(self, proposal, acceptance, rng):
        self.proposer = proposal
        self.accepter = acceptance
        self.rng = rng
        self.last_run = None

    # ---- compilation of the object graph ------------------------------------------------------
    def _compile(self, total_steps, burn_in, sample_interval, recompute_phi_u):
        if not isinstance(self.proposer, _GaussianStepProposer):
            raise TypeError("proposer %r has no device implementation" % (self.proposer,))
        a = _acc.device_spec(self.accepter)
        pot = a["potential"]
        if not isinstance(pot, EvolutionPotential):
            raise TypeError("the accepter's potential must be an EvolutionPotential over a device forward "
                            "model (no CPU fallback)")
        p = self.proposer.device_spec(total_steps)
        prior_cov_dist = self.proposer.w
        d = prior_cov_dist.k
        chol = None
        if a["kind"] == _lib.ACCEPT_RW:
            chol = a["prior"].L
            if chol.shape != (d, d):
                raise ValueError("prior dimension mismatch between proposer and accepter")
        if recompute_phi_u is None:
            recompute_phi_u = pot.G.stateful       # reference order for the stateful Lorenz operator
        seed = int(self.rng.integers(0, 2 ** 63 - 1)) if hasattr(self.rng, "integers") else int(self.rng)
        spec = SamplerSpec(dim=d, proposer_kind=p["kind"], accepter_kind=a["kind"], coef_u=p["coef_u"],
                           coef_w=p["coef_w"], schedule=p["schedule"], factor=prior_cov_dist.sample_factor(),
                           prior_chol=chol, constraint=a["constraint"], recompute_phi_u=recompute_phi_u,
                           seed=seed, record_start=max(0, burn_in - sample_interval),
                           record_interval=sample_interval)
        return spec, pot, a

    def run(self, u_0, n_samples, burn_in=1000, sample_interval=200, n_chains=None, chain_offset=0,
            steps_per_launch=None, return_device=False, recompute_phi_u=None, out=None, phi_0=None, diagnostics=False):
        """Same step accounting as the reference (sampler.py:18-28): max(0, burn_in - interval)
        unrecorded steps, then n_samples * interval steps recording every interval-th state.

        Returns ndarray [n_samples, d] for a single chain (u_0 of shape (d,), n_chains None) or
        [n_chains, n_samples, d] for a batch.  Statistics of the run are left in `self.last_run`.
        `out`: optional preallocated host buffer for the samples (NumPy array or torch CPU tensor of
        n_chains * n_samples * d float64; a PINNED torch tensor makes the device->host copy a single DMA).
        `phi_0`: Phi(u_0) per chain when it is known -- `last_run["phi"]` of the run that ended in u_0 --
        so that a continued run does not pay one more forward solve per chain (deterministic models only).
        `diagnostics`: fill `last_run["diagnostics"]` with diagnostics.chain_diagnostics of the device trace (every
        chain; over all ranks of an initialised process group) before it is copied out; the samples are unchanged.
        """
        if sample_interval < 1:
            raise ValueError("sample_interval must be >= 1")
        if diagnostics and n_samples < 4:
            raise ValueError("diagnostics=True needs at least 4 samples per chain (split-R-hat), got %d" % n_samples)
        pre = max(0, burn_in - sample_interval)
        total = pre + n_samples * sample_interval
        spec, pot, a = self._compile(total, burn_in, sample_interval, recompute_phi_u)
        if isinstance(self.accepter, _acc.CountedAccepter):
            self.accepter.reset()                   # only when outermost (sampler.py:15-16)
        problem = pot.problem()
        single = n_chains is None and np.ndim(u_0) == 1
        if phi_0 is not None and pot.G.stateful:
            raise ValueError("phi_0 is meaningless for a stateful forward model (Phi(u) is re-evaluated every step)")
        chains = ChainBatch(problem, u_0, n_chains=n_chains, chain_offset=chain_offset, phi0=phi_0)
        trace = torch.empty((chains.n, n_samples, chains.d), dtype=F64, device=problem.device)
        run_recording(chains, spec, total, pre, sample_interval, trace, steps_per_launch)
        pooled = chains.pooled()
        counters = chains.counters
        if pot.G.stateful and single:
            pot.G.IC = chains.model_state[0].cpu().numpy()
        pooled_h = pooled.cpu().numpy()
        d = chains.d
        self.last_run = dict(n_chains=chains.n, total_steps=total, launches=chains.launches,
                             pooled_count=pooled_h[0], pooled_mean=pooled_h[1:1 + d],
                             pooled_var=pooled_h[1 + d:1 + 2 * d] / max(pooled_h[0] - 1, 1),
                             counters=dict(zip(ChainBatch.COUNTER_NAMES, pooled_h[1 + 2 * d:].astype(np.int64))),
                             per_chain_counters=counters, chains=chains, seed=spec.seed,
                             h2d_bytes=chains.h2d_bytes, u=chains.u, phi=chains.phi)
        cn = self.last_run["counters"]
        _acc.credit_counters(a, cn["calls"], cn["accepts"], cn["constraint_rejects"])
        if diagnostics:
            self.last_run["diagnostics"] = _diag.chain_diagnostics(trace)
        if return_device:
            return trace[0] if single else trace
        if out is not None:
            dst = out if torch.is_tensor(out) else torch.from_numpy(out)
            if dst.dtype != F64 or dst.numel() != trace.numel() or not dst.is_contiguous():
                raise ValueError("out must be a contiguous float64 buffer of %d elements" % trace.numel())
            dst.view(trace.shape).copy_(trace, non_blocking=True)
            torch.cuda.current_stream(problem.device).synchronize()
            res = dst.view(trace.shape).numpy()
        else:
            res = trace.cpu().numpy()
        self.last_run["d2h_bytes"] = res.nbytes + pooled_h.nbytes
        return res[0] if single else res

    def run_host(self, u_0, n_samples, burn_in=1000, sample_interval=200, n_chains=None, chain_offset=0,
                 recompute_phi_u=None, out=None, phi_0=None):
        """`run` through the C entry point `ipmcmc_sample_host` alone: NumPy (host) buffers in and out,
        every copy and the device arena inside the C call, no torch tensor anywhere on the path -- what a
        binding from another language would execute.  Same step accounting and results as `run` (tested
        bit-identical); returns [n_chains, n_samples, d] (squeezed for a single chain) and fills `last_run`
        with the pooled moments, counters, final states `u` and potentials `phi` as NumPy arrays."""
        import ctypes as C
        if sample_interval < 1:
            raise ValueError("sample_interval must be >= 1")
        pre = max(0, burn_in - sample_interval)
        total = pre + n_samples * sample_interval
        spec, pot, a = self._compile(total, burn_in, sample_interval, recompute_phi_u)
        if isinstance(self.accepter, _acc.CountedAccepter):
            self.accepter.reset()
        problem = pot.problem()
        d = spec.dim
        single = n_chains is None and np.ndim(u_0) == 1
        u0 = np.asarray(u_0, dtype=np.float64)
        if u0.ndim == 1:
            u0 = np.broadcast_to(u0, (n_chains or 1, d))
        if u0.shape != (n_chains or u0.shape[0], d):
            raise ValueError("u_0 has shape %s, expected (%d,) or (n_chains, %d)" % (u0.shape, d, d))
        u0 = np.ascontiguousarray(u0)
        B = u0.shape[0]

        class _Desc:      # what SamplerSpec.c_desc reads from a ChainBatch
            _keep, step = [], 0
        _Desc.chain_offset, _Desc.problem = int(chain_offset), problem
        desc = spec.c_desc(_Desc, total)
        io = _lib.HostIO()
        keep = [u0]
        io.u0_host = _lib.as_double_p(u0)
        if phi_0 is not None:
            ph = np.ascontiguousarray(phi_0, dtype=np.float64).reshape(B)
            io.phi0_host = _lib.as_double_p(ph)
            keep.append(ph)
        ms = None
        if pot.G.stateful:
            ms = np.ascontiguousarray(np.broadcast_to(np.asarray(pot.G.IC, dtype=np.float64), (B, problem.state_size))).copy()
            io.model_state_host = _lib.as_double_p(ms)
        if out is None:
            out = np.empty((B, n_samples, d))
        elif not (isinstance(out, np.ndarray) and out.dtype == np.float64 and out.size == B * n_samples * d and out.flags.c_contiguous):
            raise ValueError("out must be a C-contiguous float64 NumPy array of %d elements" % (B * n_samples * d))
        u_end, phi_end = np.empty((B, d)), np.empty(B)
        counters = np.zeros((B, _lib.N_COUNTERS), dtype=np.int64)
        pooled = np.empty(2 * d + 1 + _lib.N_COUNTERS)
        io.samples_host, io.n_record = _lib.as_double_p(out), n_samples
        io.u_host, io.phi_host = _lib.as_double_p(u_end), _lib.as_double_p(phi_end)
        io.counters_host, io.pooled_host = counters.ctypes.data_as(_lib.c_int64_p), _lib.as_double_p(pooled)
        _lib.check(problem.lib.ipmcmc_sample_host(problem.handle, C.byref(desc), B, total, C.byref(io), None))
        if ms is not None and single:
            pot.G.IC = ms[0]
        self.last_run = dict(n_chains=B, total_steps=total, launches=4, pooled_count=pooled[0], pooled_mean=pooled[1:1 + d],
                             pooled_var=pooled[1 + d:1 + 2 * d] / max(pooled[0] - 1, 1),
                             counters=dict(zip(ChainBatch.COUNTER_NAMES, pooled[1 + 2 * d:].astype(np.int64))),
                             per_chain_counters=counters, seed=spec.seed, u=u_end, phi=phi_end, model_state=ms,
                             h2d_bytes=u0.nbytes + (ms.nbytes if ms is not None else 0) + (8 * B if phi_0 is not None else 0),
                             d2h_bytes=out.nbytes + u_end.nbytes + phi_end.nbytes + counters.nbytes + pooled.nbytes
                             + (ms.nbytes if ms is not None else 0))
        cn = self.last_run["counters"]
        _acc.credit_counters(a, cn["calls"], cn["accepts"], cn["constraint_rejects"])
        res = out.reshape(B, n_samples, d)
        return res[0] if single else res

    @classmethod
    def autocorr(cls, x):
        return _stats.autocorr(x)
