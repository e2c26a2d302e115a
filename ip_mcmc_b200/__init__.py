"""ip_mcmc_b200 -- B200-native batched MCMC engine behind ip_mcmc's Python interfaces.

The export list follows the reference's (ip_mcmc/ip_mcmc/__init__.py:1-5) for the hot path, plus
the device forward models and the pieces batching adds.  Out of scope (SURVEY.md section 8):
AnalyticAccepter, AnalyticPotential, LogNormalDistribution, IndependentDistributions.
"""
from .sampler import MCMCSampler
from .proposer import (ConstStepStandardRWProposer, VarStepStandardRWProposer, ConstSteppCNProposer,
                       VarSteppCNProposer)
from .accepter import (StandardRWAccepter, pCNAccepter, CountedAccepter, ConstrainAccepter, BoxConstraint)
from .potential import EvolutionPotential
from .distribution import GaussianDistribution
from .forward import BurgersFVM, Lorenz96Moments
from .engine import Problem, ChainBatch, SamplerSpec, fp64_peak_tflops
from . import stats, parallel, studies, diagnostics
from .diagnostics import chain_diagnostics
from . import tempering
from .tempering import ParallelTemperingSampler, geometric_inv_temps

# the stale name the reference's scripts import (lorenz_mcmc.py:6-10, burgers_mcmc.py:4-8)
pCNProposer = ConstSteppCNProposer

__all__ = ["MCMCSampler", "ConstStepStandardRWProposer", "VarStepStandardRWProposer", "ConstSteppCNProposer",
           "VarSteppCNProposer", "pCNProposer", "StandardRWAccepter", "pCNAccepter", "CountedAccepter",
           "ConstrainAccepter", "BoxConstraint", "EvolutionPotential", "GaussianDistribution", "BurgersFVM",
           "Lorenz96Moments", "Problem", "ChainBatch", "SamplerSpec", "fp64_peak_tflops", "stats", "parallel", "studies", "diagnostics",
           "chain_diagnostics", "tempering", "ParallelTemperingSampler", "geometric_inv_temps"]
