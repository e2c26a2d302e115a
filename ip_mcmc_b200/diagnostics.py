"""Convergence diagnostics of every chain of a batch, computed on the device (include/ipmcmc.h, ipmcmc_diag_*):
per-chain integrated autocorrelation time and ESS (stats.integrated_autocorr_time / stats.ess_multichain),
split-R-hat (stats.split_rhat) and multi-chain ESS (stats.multichain_ess) over all chains, and, with an
initialised process group, over the chains of all ranks.

    d = chain_diagnostics(trace[:, burn_in:])      # trace: cuda float64 [n_chains, n, d] (or a NumPy array)
    d["rhat"], d["ess"], d["cutoff"], d["tau"], d["ess_per_chain_sum"]

The lag sums of the multi-chain ESS run in blocks of 64, 128, 256, ... lags.  Every block is enqueued without
waiting for the host: after each one a one-thread-per-parameter kernel advances the truncated sum and flags
the parameters whose cut-off is found, and the next blocks skip them.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib, parallel
from ._lib import check

F64 = torch.float64
LAG_BLOCK0 = 64


def lag_blocks(h):
    """[t0, t1) blocks covering the lags 1 .. h-1, of 64, 128, 256, ... lags."""
    blocks, t0, L = [], 1, LAG_BLOCK0
    while t0 < h:
        blocks.append((t0, min(t0 + L, h)))
        t0, L = t0 + L, 2 * L
    return blocks


def _as_trace(samples):
    if not torch.is_tensor(samples):
        samples = torch.from_numpy(np.ascontiguousarray(samples, dtype=np.float64)).cuda()
    x = samples
    if not x.is_cuda or x.dtype != F64 or x.dim() != 3:
        raise ValueError("samples must be a CUDA float64 tensor [n_chains, n, d] or a NumPy array")
    if x.shape[2] > 1 and x.stride(2) != 1 or x.shape[1] > 1 and x.stride(1) != x.shape[2]:
        raise ValueError("the rows of samples must be contiguous (any chain stride)")
    return x


def _chain_stride(x):
    n, d = x.shape[1], x.shape[2]
    return x.stride(0) if x.shape[0] > 1 else n * d


def _ptr(t, offset_elems=0):
    return C.c_void_p(t.data_ptr() + 8 * offset_elems)


def _diagnose(xs, gather):
    """Diagnostics of the chains of the traces `xs` (same n, d and device) together with those that `gather`
    brings in: gather(list of per-trace tensors) -> [world, ...] in a fixed order, the same on every rank."""
    lib = _lib.load()
    n, d = int(xs[0].shape[1]), int(xs[0].shape[2])
    if any(x.shape[1:] != xs[0].shape[1:] or x.device != xs[0].device for x in xs):
        raise ValueError("all traces must have the same draws, dimension and device")
    dev = xs[0].device
    h = n // 2
    with torch.cuda.device(dev):
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        blocks = lag_blocks(h) if n >= 4 else []
        if not blocks:
            raise ValueError("split-R-hat and multi-chain ESS need at least 4 draws per chain, got %d" % n)
        l_max = max(t1 - t0 for t0, t1 in blocks)
        taus, ess_sums, seqs, scratch = [], [], [], []
        for x in xs:
            M = int(x.shape[0])
            tau = torch.empty((M, d), dtype=F64, device=dev)
            check(lib.ipmcmc_diag_tau(M, n, d, _ptr(x), _chain_stride(x), _ptr(tau), st))
            taus.append(tau)
            ess_sums.append((n / tau).amin(dim=1).sum().reshape(1))
            sb = int(lib.ipmcmc_diag_scratch_bytes(M, d, l_max))
            scratch.append(torch.empty((sb,), dtype=torch.uint8, device=dev))
            ss = torch.empty((d, 4), dtype=F64, device=dev)
            check(lib.ipmcmc_diag_seqstats(M, n, d, _ptr(x), _chain_stride(x), _ptr(ss), _ptr(scratch[-1]), sb, st))
            seqs.append(ss)
        ess_sum = parallel.merge_sums(gather(ess_sums))
        seq = parallel.merge_seqstats(gather(seqs)).contiguous()
        vsum = torch.zeros((d, h), dtype=F64, device=dev)
        state = torch.zeros((2 * d,), dtype=F64, device=dev)
        done = torch.zeros((d,), dtype=torch.int32, device=dev)
        out = torch.full((3 * d,), float("nan"), dtype=F64, device=dev)
        for t0, t1 in blocks:
            parts = []
            for x, s in zip(xs, scratch):
                v = torch.zeros((d, t1 - t0), dtype=F64, device=dev)
                check(lib.ipmcmc_diag_variogram(int(x.shape[0]), n, d, _ptr(x), _chain_stride(x), t0, t1 - t0, _ptr(done),
                                                _ptr(v), t1 - t0, _ptr(s), s.numel(), st))
                parts.append(v)
            vsum[:, t0:t1] = parallel.merge_sums(gather(parts))
            check(lib.ipmcmc_diag_truncate(n, d, _ptr(seq), _ptr(vsum), h, t1, _ptr(state), _ptr(done), _ptr(out), st))
        res = torch.cat([out, ess_sum] + [t.reshape(-1) for t in taus]).cpu().numpy()   # the one synchronisation
    return dict(rhat=res[:d], ess=res[d:2 * d], cutoff=res[2 * d:3 * d].astype(np.int64),
                ess_per_chain_sum=float(res[3 * d]), tau=res[3 * d + 1:].reshape(-1, d))


def chain_diagnostics(samples, group=None):
    """Convergence diagnostics of samples [n_chains, n, d] (a CUDA float64 tensor whose rows are contiguous,
    any chain stride, e.g. trace[:, burn_in:]; or a NumPy array, uploaded once).  Returns a dict of NumPy
    results:
      rhat [d]              split-R-hat over all chains (stats.split_rhat)
      ess [d], cutoff [d]   multi-chain effective sample size and its truncation lag T (stats.multichain_ess)
      tau [n_chains, d]     per-chain integrated autocorrelation time (stats.integrated_autocorr_time)
      ess_per_chain_sum     sum over chains of min over parameters of n / tau (stats.ess_multichain's total)
    With an initialised process group of more than one rank, each rank passes its shard of the chains (same
    n and d) and every rank gets rhat, ess, cutoff and ess_per_chain_sum of all chains; tau stays per rank.
    Enqueued on the current stream, with one synchronisation at the end.
    Device memory besides small [d, h] buffers: the variogram partial sums, min(128, ceil(n_chains / 8)) x d x (the
    largest lag block, up to about h / 2 lags) doubles -- at most about half the size of the trace itself, e.g.
    1.07 GB for d = 256 and n = 20 000 (a 42 GB trace at 1024 chains)."""
    return _diagnose([_as_trace(samples)], lambda ts: parallel.allgather(ts[0], group))
