"""TEST INFRASTRUCTURE ONLY -- CPU statement of replica exchange (ip_mcmc_b200/csrc/tempering.cuh and the
tempered accept line of metropolis_step, burgers_kernels.cuh).  The reference has no tempering.

  tempered accept   a = exp((t*Phi(u) + reg_u) - (t*Phi(v) + reg_v)),  accepted = a > U
                    reg = .5||L w||^2 (RW) or 0 (pCN), not tempered; t = 1 multiplies exactly, so t = 1 is
                    mcmc_np.run_chain bit for bit; t = 0 still rejects a non-finite Phi (0*NaN, 0*inf are NaN)
  swap round r      pairs (k, k+1), k = r (mod 2), of every ladder; swap iff
                    exp((t_k - t_{k+1}) * (Phi_k - Phi_{k+1})) > U
  swap uniform      Philox4x32-10 key (seed lo, global id of slot k), counter (r lo, r hi, SLOT_SWAP, seed hi),
                    mapped as philox_np.uniform maps the accept uniform
  replica records   (replica id, direction) move with the state; after the swaps slot 0 takes direction +1 (a
                    round trip when it was -1) and slot K-1 direction -1, in the rounds that propose (0, 1),
                    resp. (K-2, K-1)
"""
import numpy as np

from . import mcmc_np
from . import philox_np

SLOT_SWAP = 0xFFFFFFFE


class _TemperedPotential:
    """t * Phi(u): handed to mcmc_np.run_chain, whose accept line then evaluates the tempered rule above in the
    engine's operation order (the pCN line exp(phi_u - phi_v) equals exp((phi_u + 0) - (phi_v + 0)))."""

    def __init__(self, potential, inv_temp):
        self.potential = potential
        self.t = np.float64(inv_temp)

    def __call__(self, u):
        return self.t * self.potential(u)


def run_chain(potential, u0, normals, uniforms, inv_temp=1.0, **kw):
    """mcmc_np.run_chain of a chain whose likelihood is tempered by inv_temp.  Same outputs; phi_u and phi_v
    hold the TEMPERED values t * Phi."""
    return mcmc_np.run_chain(_TemperedPotential(potential, inv_temp), u0, normals, uniforms, **kw)


def pairs(K, r):
    """Rungs k of the pairs (k, k+1) round r proposes."""
    return list(range(r % 2, K - 1, 2))


def swap_uniform(seed, chain, r):
    x0, x1, _, _ = philox_np.draw_words(seed, chain, r, SLOT_SWAP)
    return np.float64(((x1 << 32 | x0) >> 11)) * np.float64(2.0 ** -53)


def swap_uniforms(seed, chain_offset, n_ladders, K, r):
    """[n_ladders, K-1] swap uniforms of round r (NaN for the pairs the round does not propose)."""
    U = np.full((n_ladders, K - 1), np.nan)
    for l in range(n_ladders):
        for k in pairs(K, r):
            U[l, k] = swap_uniform(seed, chain_offset + l * K + k, r)
    return U


def swap_round(u, phi, inv_temp, K, r, U, replica, swap_counts, round_trips):
    """Round r over the ladder-major arrays, in place: u [B, d], phi [B], inv_temp [B], U [n_ladders, K-1],
    replica [B, 2] int, swap_counts [n_ladders, K-1, 2] int, round_trips [n_ladders] int."""
    n_ladders = u.shape[0] // K
    for l in range(n_ladders):
        for k in pairs(K, r):
            a, b = l * K + k, l * K + k + 1
            with np.errstate(over="ignore", invalid="ignore"):
                acc = np.exp((inv_temp[a] - inv_temp[b]) * (phi[a] - phi[b]))
            swap = bool(acc > U[l, k])
            swap_counts[l, k, 0] += 1
            swap_counts[l, k, 1] += swap
            if swap:
                u[[a, b]] = u[[b, a]]
                phi[[a, b]] = phi[[b, a]]
                replica[[a, b]] = replica[[b, a]]
            if k == 0:
                if replica[l * K, 1] == -1:
                    round_trips[l] += 1
                replica[l * K, 1] = 1
            if k + 1 == K - 1:
                replica[l * K + K - 1, 1] = -1
