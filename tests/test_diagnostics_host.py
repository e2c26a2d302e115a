"""Host reference of the convergence diagnostics (stats.split_rhat, stats.multichain_ess) against a naive
restatement of BDA3 sections 11.4-11.5, its statistical behaviour, its IEEE special values, and the merge
functions that combine per-rank partials (parallel.merge_seqstats / merge_sums) under gloo."""
import ctypes as C
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from ip_mcmc_b200 import parallel, stats
from ip_mcmc_b200.diagnostics import lag_blocks


def ar1(M, n, d, phi, seed):
    """AR(1) chains started from their stationary law N(0, 1 / (1 - phi^2))."""
    rng = np.random.default_rng(seed)
    x = np.empty((M, n, d))
    x[:, 0] = rng.standard_normal((M, d)) / math.sqrt(1 - phi * phi)
    for i in range(1, n):
        x[:, i] = phi * x[:, i - 1] + rng.standard_normal((M, d))
    return x


def naive(traces):
    """Double loops over sequences and draws, one parameter at a time -> (rhat, n_eff, T)."""
    M, n, d = traces.shape
    h = n // 2
    seqs = []
    for c in range(M):
        seqs.append([list(traces[c, i]) for i in range(h)])
        seqs.append([list(traces[c, n - h + i]) for i in range(h)])
    m = len(seqs)
    rhat, neff, cut = [], [], []
    for j in range(d):
        psi = [[s[i][j] for i in range(h)] for s in seqs]
        means = [sum(p) / h for p in psi]
        var = [sum((v - mu) ** 2 for v in p) / (h - 1) for p, mu in zip(psi, means)]
        grand = sum(means) / m
        B = h / (m - 1) * sum((mu - grand) ** 2 for mu in means)
        W = sum(var) / m
        vp = (h - 1) / h * W + B / h
        rhat.append(math.sqrt(vp / W))

        def rho(t):
            V = sum((p[i] - p[i - t]) ** 2 for p in psi for i in range(t, h)) / (m * (h - t))
            return 1 - V / (2 * vp)
        S, t = 0.0, 1
        while True:
            S += rho(t)
            if t + 2 > h - 1 or rho(t + 1) + rho(t + 2) < 0:
                break
            S += rho(t + 1)
            t += 2
        neff.append(m * h / (1 + 2 * S))
        cut.append(t)
    return np.array(rhat), np.array(neff), np.array(cut)


@pytest.mark.parametrize("M,n,d,phi", [(3, 4, 1, 0.0), (2, 5, 2, 0.5), (4, 17, 2, 0.3), (5, 40, 3, 0.8), (3, 41, 1, 0.95)])
def test_split_estimators_match_naive_restatement(M, n, d, phi):
    x = ar1(M, n, d, phi, seed=M * 100 + n) + np.arange(d)
    rhat, neff, cut = naive(x)
    np.testing.assert_allclose(stats.split_rhat(x), rhat, rtol=1e-12)
    ne, T = stats.multichain_ess(x)
    np.testing.assert_allclose(ne, neff, rtol=1e-12)
    assert np.array_equal(T, cut)


def test_split_sequences_drop_the_middle_draw():
    x = np.arange(2 * 7 * 1, dtype=float).reshape(2, 7, 1)
    s = stats.split_sequences(x)
    assert s.shape == (4, 3, 1)
    assert s[:, :, 0].tolist() == [[0, 1, 2], [4, 5, 6], [7, 8, 9], [11, 12, 13]]
    with pytest.raises(ValueError):
        stats.split_sequences(np.zeros((2, 3, 1)))


def test_ar1_multichain_ess_matches_theory():
    phi = 0.9
    x = ar1(2048, 2000, 1, phi, seed=1)
    ne, _ = stats.multichain_ess(x)
    m, h = 2 * 2048, 1000
    assert abs(ne[0] / (m * h) / ((1 - phi) / (1 + phi)) - 1) < 0.05


def test_rhat_separates_disagreeing_chains():
    rng = np.random.default_rng(2)
    x = rng.standard_normal((64, 500, 2))
    assert np.all(stats.split_rhat(x) < 1.01)
    x[32:] += 3.0
    assert np.all(stats.split_rhat(x) > 1.5)


def test_special_values():
    same = np.full((3, 10, 1), 0.25)
    assert np.isnan(stats.split_rhat(same)[0])
    ne, T = stats.multichain_ess(same)
    assert np.isnan(ne[0]) and T[0] == 3            # NaN never stops the sum: runs to t + 2 > h - 1 = 4
    apart = np.full((3, 10, 1), 0.25) * np.arange(3)[:, None, None]
    assert np.isinf(stats.split_rhat(apart)[0])
    ne, T = stats.multichain_ess(apart)
    assert T[0] == 3 and ne[0] == 6 * 5 / (1 + 2 * 3.0)   # V_t = 0: rho_t = 1, S = rho_1 + rho_2 + rho_3


def test_lag_blocks_cover_every_lag_once():
    for h in (2, 3, 64, 65, 66, 500, 2500):
        b = lag_blocks(h)
        assert b[0][0] == 1 and b[-1][1] == h
        assert all(b[k][1] == b[k + 1][0] for k in range(len(b) - 1))
        assert [t1 - t0 for t0, t1 in b[:-1]] == [64 << k for k in range(len(b) - 1)]


def host_partials(x, lags):
    """What ipmcmc_diag_seqstats / ipmcmc_diag_variogram compute, from the host reference's sequences."""
    psi = stats.split_sequences(x)
    means = psi.mean(axis=1)
    ss = np.stack([np.full(x.shape[2], float(psi.shape[0])), means.mean(0), ((means - means.mean(0)) ** 2).sum(0),
                   psi.var(axis=1, ddof=1).sum(0)], axis=1)
    v = np.stack([((psi[:, t:] - psi[:, :psi.shape[1] - t]) ** 2).sum(axis=(0, 1)) for t in lags], axis=1)
    return ss, v


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, data, lags, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    lo, hi = parallel.shard(data.shape[0], rank, world)
    ss, v = host_partials(data[lo:hi], lags)
    s = parallel.merge_seqstats(parallel.allgather(torch.tensor(ss)))
    vv = parallel.merge_sums(parallel.allgather(torch.tensor(v)))
    ret.put((rank, s.numpy(), vv.numpy()))
    dist.destroy_process_group()


def test_merge_functions_two_ranks():
    data = ar1(7, 30, 3, 0.7, seed=3) * [1, 2, 3] + [100, -5, 0.1]     # 7 chains: uneven shards
    lags = list(range(1, 15))
    ctx = mp.get_context("spawn")
    ret = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, data, lags, ret)) for r in range(2)]
    for p in procs:
        p.start()
    got = [ret.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    (_, s0, v0), (_, s1, v1) = got
    assert np.array_equal(s0, s1) and np.array_equal(v0, v1)      # every rank takes the same decision
    ss, v = host_partials(data, lags)
    assert np.array_equal(s0[:, 0], ss[:, 0])
    np.testing.assert_allclose(s0[:, 1:], ss[:, 1:], rtol=1e-12)
    np.testing.assert_allclose(v0, v, rtol=1e-12)


def test_merge_without_process_group_is_identity():
    x = torch.arange(12, dtype=torch.float64).reshape(3, 4)
    assert torch.equal(parallel.merge_seqstats(parallel.allgather(x)), x)
    assert torch.equal(parallel.merge_sums(parallel.allgather(x)), x)


def test_device_entry_points_check_arguments_without_gpu():
    from ip_mcmc_b200 import _lib
    lib = _lib.load()
    p = C.c_void_p(8)          # never dereferenced: every call below fails its argument check first
    assert lib.ipmcmc_diag_seqstats(4, 3, 1, p, 3, p, None, 0, None) == -1 and b"n_draws" in lib.ipmcmc_last_error()
    assert lib.ipmcmc_diag_seqstats(4, 10, 257, p, 2570, p, None, 0, None) == -1 and b"dim" in lib.ipmcmc_last_error()
    assert lib.ipmcmc_diag_tau(4, 10, 3, p, 29, p, None) == -1 and b"chain_stride" in lib.ipmcmc_last_error()
    assert lib.ipmcmc_diag_tau(0, 10, 3, p, 30, p, None) == -1
    assert lib.ipmcmc_diag_variogram(4, 10, 1, p, 10, 3, 3, None, p, 3, None, 0, None) == -1   # lag 5 >= h
    assert lib.ipmcmc_diag_variogram(4, 10, 1, p, 10, 1, 4, None, p, 4, p, 8, None) == -1      # scratch too small
    assert b"scratch" in lib.ipmcmc_last_error()
    assert lib.ipmcmc_diag_truncate(10, 1, p, p, 5, 6, p, p, p, None) == -1                     # lag_end > h
    assert lib.ipmcmc_diag_scratch_bytes(128, 3, 64) == 16 * 3 * 64 * 8
    with pytest.raises(ValueError):
        _lib.check(-1)


def test_run_with_diagnostics_rejects_short_runs_before_sampling():
    from ip_mcmc_b200 import MCMCSampler
    with pytest.raises(ValueError, match="at least 4 samples"):
        MCMCSampler(None, None, None).run(np.zeros(3), 3, 0, 1, diagnostics=True)   # raises before touching the GPU
