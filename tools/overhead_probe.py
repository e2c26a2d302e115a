#!/usr/bin/env python
"""Per-Metropolis-step overhead outside the FV time loop (run on the GPU box):
flat-work chain launches (every chain repeats the same proposal: identical solves) for several
final times T; time per chain-step is fitted as a + b * n_fv.  `a` is what one Metropolis step costs
besides the time loop (initial condition, first peeled step, measurement, Phi, Philox, exp, queue)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import ip_mcmc_b200 as M
from ip_mcmc_b200 import _lib
import bench

N = int(sys.argv[1]) if len(sys.argv) > 1 else 256
S = 20
for nch in (1024, 16384):
    rows = []
    for T in (0.125, 0.25, 0.5, 1.0, 2.0):
        f = M.BurgersFVM(N=N, T=T, numerics="fused")
        y = f.at_parameters(bench.TRUTH)
        pot = M.EvolutionPotential(f, y, M.GaussianDistribution(np.zeros(5), 0.05 ** 2 * np.identity(5)))
        spec = M.SamplerSpec(3, _lib.PROPOSE_PCN, _lib.ACCEPT_PCN, coef_u=1.0, coef_w=0.0)
        ch = M.ChainBatch(pot.problem(), bench.TRUTH - bench.PRIOR_MEAN, n_chains=nch)
        w = torch.zeros((nch, S, 3), dtype=torch.float64, device="cuda")
        U = torch.ones((nch, S), dtype=torch.float64, device="cuda")
        ts = []
        for _ in range(4):
            c0 = ch.counters[:, 2].sum().item()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); ch.run(spec, S, inject_w=w, inject_u=U); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
            nfv = (ch.counters[:, 2].sum().item() - c0) / nch / S
        rows.append((nfv, min(ts) * 1e-3 / S))
    x = np.array([r[0] for r in rows]); t = np.array([r[1] for r in rows])
    b, a = np.polyfit(x, t, 1)
    print("N=%d chains=%d: n_fv %s  t/step(us) %s" % (N, nch, x.round(1).tolist(), (t * 1e6).round(2).tolist()))
    print("   fit: a = %.2f us per launch-step (= %.1f FV-step equivalents), b = %.4f us per FV step; overhead at T=1: %.1f %%"
          % (a * 1e6, a / b, b * 1e6, 100 * a / (a + b * x[3])))

# section cycles (library built with -DIPMCMC_PROF=1 only)
import ctypes
lib = ctypes.CDLL(os.environ.get("IPMCMC_LIB", ""), mode=ctypes.RTLD_GLOBAL) if os.environ.get("IPMCMC_LIB") else None
if lib is not None and hasattr(lib, "ipmcmc_prof_read"):
    buf = (ctypes.c_ulonglong * 16)()
    for nch in (1024, 16384):
        f = M.BurgersFVM(N=N, T=1.0, numerics="fused")
        y = f.at_parameters(bench.TRUTH)
        pot = M.EvolutionPotential(f, y, M.GaussianDistribution(np.zeros(5), 0.05 ** 2 * np.identity(5)))
        wl = dict(bench.WORKLOADS["burgers_pcn_256"]); wl["N"] = N
        pot2, proposer, accepter, u0 = bench.build_problem(M, wl, "fused")
        sampler = M.MCMCSampler(proposer, accepter, np.random.default_rng(2))
        spec, pot2, a = sampler._compile(10 ** 9, 0, 1, None)
        ch = M.ChainBatch(pot2.problem(), bench.TRUTH - bench.PRIOR_MEAN, n_chains=nch)
        ch.run(spec, 200)
        lib.ipmcmc_prof_read(buf, 1)
        c0 = ch.counters[:, 2].sum().item()
        ch.run(spec, 50)
        lib.ipmcmc_prof_read(buf, 1)
        v = np.array(list(buf), dtype=np.float64)
        items = v[8]
        nfv = (ch.counters[:, 2].sum().item() - c0) / items
        names = ["item total", "pop (ticket, ring, progress)", "proposal noise", "integrate (IC + time loop)",
                 "store + measure + Phi", "accept (exp, U, update)", "state load + steps + write-back", "push"]
        print("chains=%d: %d items, %.1f FV steps per item" % (nch, items, nfv))
        for k, nm in enumerate(names):
            print("   %-34s %9.0f cycles per item  (%5.1f %%)" % (nm, v[k] / items, 100 * v[k] / v[0]))
        print("   integrate per FV step: %.1f cycles" % (v[3] / items / nfv))
