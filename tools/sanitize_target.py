#!/usr/bin/env python
"""Tiny end-to-end exercise of every kernel family for compute-sanitizer --tool memcheck (small sizes)."""
import os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ip_mcmc_b200 as M
from ip_mcmc_b200 import studies
TRUTH, PM = np.array([0.025, -0.025, -0.02]), np.array([1.5, 0.25, -0.5])
noise = M.GaussianDistribution(np.zeros(5), 0.05 ** 2 * np.identity(5))
prior = M.GaussianDistribution(PM, 0.25 ** 2 * np.identity(3))
for N, num in ((64, "fused"), (100, "exact"), (256, "fused")):
    f = M.BurgersFVM(N=N, numerics=num)
    pot = M.EvolutionPotential(f, f.at_parameters(TRUTH), noise)
    s = M.MCMCSampler(M.ConstSteppCNProposer(0.25, prior), M.CountedAccepter(M.pCNAccepter(pot)), np.random.default_rng(1))
    out = s.run(np.zeros(3), 6, 0, 1, n_chains=37)
    h = M.MCMCSampler(M.ConstStepStandardRWProposer(0.01, prior), M.CountedAccepter(M.StandardRWAccepter(pot, prior)), np.random.default_rng(1))
    h.run_host(np.zeros(3), 5, 0, 1, n_chains=11)
print("burgers ok")
f = M.BurgersFVM(N=2048, numerics="fused")
pot = M.EvolutionPotential(f, f.at_parameters(TRUTH), noise)
M.MCMCSampler(M.ConstSteppCNProposer(0.25, prior), M.pCNAccepter(pot), np.random.default_rng(1)).run(TRUTH - PM, 2, 0, 1, n_chains=3)
print("team ok")
m = 40
fw = M.BurgersFVM(N=128, kl_modes=m, numerics="fused")
lam = np.concatenate([np.full(3, 0.25 ** 2), M.BurgersFVM.kl_prior_variances(m, scale=0.05)])
pw = M.GaussianDistribution(fw.prior_means, np.diag(lam))
potw = M.EvolutionPotential(fw, fw.at_parameters(np.concatenate([TRUTH, np.zeros(m)])), noise)
box = M.BoxConstraint(np.r_[-np.inf, -np.inf, -1.0, np.full(m, -np.inf)], np.r_[np.inf, np.inf, 1.0, np.full(m, np.inf)], shift=np.r_[0, 0, -0.5, np.zeros(m)])
M.MCMCSampler(M.ConstStepStandardRWProposer(0.01, pw), M.ConstrainAccepter(M.CountedAccepter(M.StandardRWAccepter(potw, pw)), box),
              np.random.default_rng(1)).run(np.zeros(3 + m), 5, 0, 1, n_chains=9)
print("wide ok")
g = np.load(os.path.join(ROOT, "tests", "golden", "lorenz_problem_K6_J4.npz"))
for num in ("fused", "exact"):
    fl = M.Lorenz96Moments(6, 4, 0.25, 1.0, g["prior_means"], g["IC"], numerics=num)
    pl = M.EvolutionPotential(fl, g["y"], M.GaussianDistribution(np.zeros(30), 0.25 * np.diag(g["var"])))
    pr = M.GaussianDistribution(np.zeros(3), np.diag([10., 1, 10]))
    M.MCMCSampler(M.ConstStepStandardRWProposer(0.125, pr), M.CountedAccepter(M.StandardRWAccepter(pl, pr)),
                  np.random.default_rng(1)).run(g["u0"], 3, 0, 1, n_chains=13)
print("lorenz ok")
r = studies.chain_length_study(chain_length=200, n_chains=3, N=32, sample_interval=5, steps_per_launch=70)
print("study ok", r["counts"].sum())
torch.cuda.synchronize()
