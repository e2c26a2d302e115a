"""Times diagnostics.chain_diagnostics (all-chain tau, split-R-hat and multi-chain ESS on the device) against the host
path bench.py and sweep.py use today (stats.ess_multichain on a subset of the chains).

    python tools/diag_bench.py [--reps 5]

Traces:
  * bench: the cold-start leg of bench.py's burgers_pcn_256 workload: 1024 chains x 5000 steps x 3 parameters from
    u_0 = 0 (Burgers, 256 cells, pCN beta = 0.25, FUSED numerics), sampled in one launch; its sampling time is timed too;
  * ar1_65536: 65 536 seeded AR(1) chains (phi = 0.9) x 1000 draws x 3, generated on the device;
  * wide: 1024 seeded AR(1) chains (phi = 0.9) x 1000 draws x 64 parameters, generated on the device.
Each call is timed with CUDA events around the whole call (its launches, its one synchronisation and the copy of
the results to the host), after one untimed warm-up call of the same shape, with L2 overwritten (256 MiB memset,
untimed) before every timed call.
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import ip_mcmc_b200 as M  # noqa: E402

TRUTH = np.array([0.025, -0.025, -0.02])
PRIOR_MEAN = np.array([1.5, 0.25, -0.5])


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return q.stdout.strip() or name
    except (OSError, subprocess.SubprocessError):
        return name + " (power limit not readable)"


def ar1_device(n_chains, n, d, phi, seed):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    x = torch.empty((n_chains, n, d), dtype=torch.float64, device="cuda")
    x[:, 0] = torch.randn((n_chains, d), generator=g, dtype=torch.float64, device="cuda") / np.sqrt(1 - phi * phi)
    for i in range(1, n):
        x[:, i] = phi * x[:, i - 1] + torch.randn((n_chains, d), generator=g, dtype=torch.float64, device="cuda")
    return x


def bench_trace():
    f = M.BurgersFVM(N=256, numerics="fused")
    prior = M.GaussianDistribution(PRIOR_MEAN, 0.25 ** 2 * np.identity(3))
    pot = M.EvolutionPotential(f, f.at_parameters(TRUTH), M.GaussianDistribution(np.zeros(5), 0.05 ** 2 * np.identity(5)))
    s = M.MCMCSampler(M.ConstSteppCNProposer(0.25, prior), M.pCNAccepter(pot), np.random.default_rng(100))
    s.run(np.zeros(3), 200, 0, 1, n_chains=1024, return_device=True)          # warm-up
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    tr = s.run(np.zeros(3), 5000, 0, 1, n_chains=1024, return_device=True)
    e1.record()
    e1.synchronize()
    return tr, e0.elapsed_time(e1)


def time_diag(x, reps):
    flush = torch.empty((256 << 20,), dtype=torch.uint8, device="cuda")
    res = M.chain_diagnostics(x)                                                # warm-up
    ms = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = M.chain_diagnostics(x)
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return ms, res


def report(name, x, ms, res, extra=""):
    M_, n, d = x.shape
    print("%-10s %6d x %5d x %3d  %8.2f ms (median of %d; min %.2f, max %.2f)  rhat max %.4f  ess min %.0f  T max %d  "
          "sum ESS %.0f%s" % (name, M_, n, d, float(np.median(ms)), len(ms), min(ms), max(ms), np.nanmax(res["rhat"]),
                              np.nanmin(res["ess"]), res["cutoff"].max(), res["ess_per_chain_sum"], extra))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("diag_bench needs a CUDA device")
    print("device: %s" % card())
    print("torch %s, CUDA %s" % (torch.__version__, torch.version.cuda))

    tr, sample_ms = bench_trace()
    ms, res = time_diag(tr, args.reps)
    report("bench", tr, ms, res, "  | sampling it took %.1f ms: diagnostics = %.2f %%"
           % (sample_ms, 100 * float(np.median(ms)) / sample_ms))
    host = tr[:32].cpu().numpy()
    t0 = time.perf_counter()
    M.stats.ess_multichain(host)
    t_host = time.perf_counter() - t0
    print("host       stats.ess_multichain on 32 of those chains (5000 draws, d = 3, one CPU core): %.1f ms "
          "(%.2f ms per chain)" % (1e3 * t_host, 1e3 * t_host / 32))
    del tr

    x = ar1_device(65536, 1000, 3, 0.9, seed=1)
    ms, res = time_diag(x, args.reps)
    report("ar1_65536", x, ms, res, "  | ess/(m h) = %.4f (theory %.4f)"
           % (float(np.mean(res["ess"])) / (2 * 65536 * 500), 0.1 / 1.9))
    host = x[:32].cpu().numpy()
    t0 = time.perf_counter()
    M.stats.ess_multichain(host)
    t_host = time.perf_counter() - t0
    print("host       stats.ess_multichain on 32 of those chains (1000 draws, d = 3, one CPU core): %.1f ms "
          "(%.2f ms per chain; x 65536 chains = %.0f s)" % (1e3 * t_host, 1e3 * t_host / 32, t_host / 32 * 65536))
    del x

    x = ar1_device(1024, 1000, 64, 0.9, seed=2)
    ms, res = time_diag(x, args.reps)
    report("wide", x, ms, res)


if __name__ == "__main__":
    main()
