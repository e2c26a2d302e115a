#!/usr/bin/env python
"""Replica exchange on the bench problem (Burgers pCN beta = 0.25, 256 cells, FUSED), two measurements:

  overhead  chain-steps/s over all rungs of ParallelTemperingSampler (K = 4 geometric rungs x 256 ladders) for
            swap_interval in {1, 10, 100, 1000}, against MCMCSampler.run with the same 1024 chains; the swap
            kernel's event time per round; FV time steps per Metropolis step on each rung
  benefit   from the cold start u_0 = 0 over 5000 steps: t = 1 split-R-hat, multi-chain ESS per second, round trips
            and the fraction of t = 1 chains still near sigma_0 = -1 (end state sigma_0 = -0.5 + u_2 < -0.75), against
            1024 untempered chains
python tools/pt_bench.py [--steps 1000] [--t-min 0.05] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ip_mcmc_b200 as M  # noqa: E402
import bench  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def problem():
    wl = dict(bench.WORKLOADS["burgers_pcn_256"])
    pot, proposer, accepter, u0 = bench.build_problem(M, wl, "fused")
    return proposer, accepter.accepter if isinstance(accepter, M.CountedAccepter) else accepter


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return r, time.perf_counter() - t0


def overhead(steps, temps, n_chains, seed=3):
    K = len(temps)
    L = n_chains // K
    prop, acc = problem()
    out = {}
    base = M.MCMCSampler(prop, acc, np.random.default_rng(seed))
    base.run(np.zeros(3), 1, 0, 50, n_chains=n_chains, return_device=True)            # warm-up
    _, dt = timed(lambda: base.run(np.zeros(3), 1, 0, steps, n_chains=n_chains, return_device=True))
    c = base.last_run["per_chain_counters"]
    out["untempered"] = dict(chain_steps_per_s=n_chains * steps / dt, seconds=dt,
                             fv_steps_per_step=float(c[:, 2].sum().item() / c[:, 0].sum().item()))
    for si in (1, 10, 100, 1000):
        pt = M.ParallelTemperingSampler(prop, acc, np.random.default_rng(seed), temps, swap_interval=si)
        _, dt = timed(lambda: pt.run(np.zeros(3), 1, 0, steps, n_ladders=L, return_device=True))
        rc = pt.last_run["rung_counters"]
        out["swap_interval_%d" % si] = dict(
            chain_steps_per_s=n_chains * steps / dt, seconds=dt, launches=pt.last_run["launches"],
            fv_steps_per_step_by_rung=(rc[:, 2] / rc[:, 0]).tolist(),
            nonfinite_by_rung=rc[:, 4].tolist(), swap_acceptance=pt.last_run["swap_acceptance"].tolist(),
            round_trips=pt.last_run["round_trips"])
    # the swap kernel alone on the final state of the last run: event time per round
    ch = pt.last_run["chains"]
    rep = torch.zeros((ch.n, 2), dtype=torch.int32, device="cuda")
    sc = torch.zeros((L, K - 1, 2), dtype=torch.int64, device="cuda")
    rt = torch.zeros((L,), dtype=torch.int64, device="cuda")
    for r in range(10):
        ch.swap(K, 1, r, rep, sc, rt)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_rounds = 1000
    e0.record()
    for r in range(n_rounds):
        ch.swap(K, 1, r, rep, sc, rt)
    e1.record()
    torch.cuda.synchronize()
    out["swap_round_us"] = 1e3 * e0.elapsed_time(e1) / n_rounds
    return out


def benefit(steps, temps, n_chains, swap_interval=10, seed=4):
    K = len(temps)
    L = n_chains // K
    prop, acc = problem()
    n_samples, interval = steps // 10, 10

    def near_minus_one(u_end):
        return float(np.mean(-0.5 + u_end[:, 2] < -0.75))

    base = M.MCMCSampler(prop, acc, np.random.default_rng(seed))
    _, dt = timed(lambda: base.run(np.zeros(3), n_samples, 0, interval, n_chains=n_chains, return_device=True,
                                   diagnostics=True))
    dg = base.last_run["diagnostics"]
    res = dict(untempered=dict(chains=n_chains, seconds=dt, rhat=dg["rhat"].tolist(), ess=dg["ess"].tolist(),
                               ess_per_s=(dg["ess"] / dt).tolist(),
                               frac_near_sigma_minus_one=near_minus_one(base.last_run["u"].cpu().numpy())))
    pt = M.ParallelTemperingSampler(prop, acc, np.random.default_rng(seed), temps, swap_interval=swap_interval)
    _, dt = timed(lambda: pt.run(np.zeros(3), n_samples, 0, interval, n_ladders=L, return_device=True,
                                 diagnostics=True))
    dg = pt.last_run["diagnostics"]
    u_cold = pt.last_run["u"].view(L, K, 3)[:, 0].cpu().numpy()
    res["tempered"] = dict(ladders=L, rungs=K, inv_temps=list(map(float, temps)), swap_interval=swap_interval,
                           seconds=dt, rhat=dg["rhat"].tolist(), ess=dg["ess"].tolist(),
                           ess_per_s=(dg["ess"] / dt).tolist(), round_trips=pt.last_run["round_trips"],
                           swap_acceptance=pt.last_run["swap_acceptance"].tolist(),
                           frac_near_sigma_minus_one=near_minus_one(u_cold))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=1000, help="Metropolis steps of the overhead runs")
    ap.add_argument("--benefit-steps", type=int, default=5000)
    ap.add_argument("--t-min", type=float, default=0.05, help="inverse temperature of the hottest of the 4 rungs")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pt_bench.py measures on the GPU; no CUDA device found")
    temps = M.geometric_inv_temps(4, a.t_min)
    r = dict(card=card(), overhead=overhead(a.steps, temps, 1024), benefit=benefit(a.benefit_steps, temps, 1024))
    s = json.dumps(r, indent=1)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
