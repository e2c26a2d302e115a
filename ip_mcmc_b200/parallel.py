"""Multi-GPU plumbing: chains are independent, so ranks own contiguous blocks of GLOBAL chain ids
(Philox is keyed by the global id, results do not depend on the GPU count) and exchange nothing
while sampling.  The only collective of a run is the final reduction of pooled moments and counters
(SURVEY.md section 8(e)): ONE all-gather of 2d+7 doubles per rank followed by a local Chan merge
(latency-bound; NCCL over NVLink on the GPU box, gloo in the CPU tests).  Convergence diagnostics
(diagnostics.chain_diagnostics) merge their split-sequence statistics the same way and add one all-gather
of the variogram sums per block of lags."""
import torch
import torch.distributed as dist


def shard(n_chains, rank, world):
    """Contiguous block [start, stop) of global chain ids owned by `rank`."""
    base, rem = divmod(int(n_chains), int(world))
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def allreduce_pooled(pooled, d, group=None):
    """pooled: tensor [2d+7] = (n, mean[d], M2[d], 6 counters) of this rank (ChainBatch.pooled()).
    Returns the same layout merged over all ranks.  ONE collective: an all-gather of the 2d+7 doubles
    of every rank (latency-bound: 104 B per rank at d = 3), then Chan's merge locally on every rank:
      n = sum n_r;  mean = sum n_r mean_r / n;  M2 = sum (M2_r + n_r (mean_r - mean)^2);  counters add."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return pooled.clone()
    world = dist.get_world_size(group)
    allp = torch.empty((world * pooled.numel(),), dtype=pooled.dtype, device=pooled.device)
    dist.all_gather_into_tensor(allp, pooled.contiguous().reshape(-1), group=group)
    return merge_pooled(allp.reshape(world, pooled.numel()), d)


def merge_pooled(allp, d):
    """Chan merge of per-rank pooled rows [world, 2d+7] -> [2d+7]."""
    n = allp[:, 0:1]
    mean = allp[:, 1:1 + d]
    m2 = allp[:, 1 + d:1 + 2 * d]
    n_tot = n.sum(0)
    mean_tot = torch.where(n_tot > 0, (n * mean).sum(0) / torch.clamp(n_tot, min=1.0), torch.zeros_like(mean[0]))
    m2_tot = (m2 + n * (mean - mean_tot) ** 2).sum(0)
    return torch.cat([n_tot, mean_tot, m2_tot, allp[:, 1 + 2 * d:].sum(0)])


def distributed(group=None):
    """True when a process group with more than one rank is initialised."""
    return dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1


def allgather(x, group=None):
    """[world, *x.shape]: x of every rank in rank order (ONE all-gather); [1, *x.shape] without a group."""
    if not distributed(group):
        return x.unsqueeze(0).clone()
    world = dist.get_world_size(group)
    out = torch.empty((world * x.numel(),), dtype=x.dtype, device=x.device)
    dist.all_gather_into_tensor(out, x.contiguous().reshape(-1), group=group)
    return out.reshape((world,) + tuple(x.shape))


def merge_seqstats(alls):
    """Split-sequence statistics of several batches [world, d, 4] = (m, mean of the sequence means, M2 of the
    sequence means, sum of the sequence variances) (ipmcmc_diag_seqstats) -> [d, 4] of all their sequences:
    Chan's merge in rank order, the sums of variances added in rank order, so every rank gets the same bits."""
    r = alls[0].clone()
    for b in alls[1:]:
        n = r[:, 0] + b[:, 0]
        delta = b[:, 1] - r[:, 1]
        mean = r[:, 1] + delta * (b[:, 0] / n)
        m2 = (r[:, 2] + b[:, 2]) + delta * delta * (r[:, 0] * b[:, 0] / n)
        r = torch.stack([n, mean, m2, r[:, 3] + b[:, 3]], dim=1)
    return r


def merge_sums(alls):
    """Sums of several batches [world, ...] (variogram sums of one lag block, ESS totals) -> their sum,
    added in rank order."""
    r = alls[0].clone()
    for b in alls[1:]:
        r = r + b
    return r


def max_over_ranks(x, device, group=None):
    """Device-timed milliseconds -> max over ranks (the number a multi-GPU run reports)."""
    t = torch.tensor([float(x)], dtype=torch.float64, device=device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return float(t.item())
