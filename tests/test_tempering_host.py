"""Replica exchange without a GPU: the CPU statement (oracle/tempering_np.py) against the golden chains and
hand-built rounds, the Philox swap slot, and the argument checks of the C entry points and of
ParallelTemperingSampler."""
import ctypes as C

import numpy as np
import pytest

from conftest import golden
from oracle import burgers_np as B
from oracle import mcmc_np as O
from oracle import philox_np as P
from oracle import tempering_np as T

NOISE_COV = 0.05 ** 2 * np.identity(5)
PRIOR_COV = 0.25 ** 2 * np.identity(3)


def _pot(N):
    Pb = B.BurgersProblem(N)
    return O.Potential(Pb, Pb.G_params(np.array([0.025, -0.025, -0.02])), NOISE_COV)


@pytest.mark.parametrize("name,kind", [("chain_burgers_pcn_N64.npz", O.PCN), ("chain_burgers_pcn_N128.npz", O.PCN),
                                       ("chain_burgers_rw_N64.npz", O.RW)])
def test_untempered_rung_reproduces_golden_chains(name, kind):
    g = golden(name)
    step = float(g["beta"] if kind == O.PCN else g["delta"])
    out = T.run_chain(_pot(int(g["N"])), g["u0"], g["normals"], g["uniforms"], inv_temp=1.0, proposer=kind,
                      accepter=kind, step=step, prior_cov=PRIOR_COV)
    assert np.array_equal(out["u"], g["samples"]) and np.array_equal(out["v"], g["v"])
    assert np.array_equal(out["phi_v"], g["phi_v"])
    assert out["accepts"] == int(g["accepts"]) and out["calls"] == int(g["calls"])


def test_tempered_accept_line():
    """t scales Phi, not the RW regulariser; t = 0 still rejects a non-finite Phi."""
    pot = _pot(64)
    g = golden("chain_burgers_pcn_N64.npz")
    n = 40
    for t in (0.5, 0.0):
        out = T.run_chain(pot, g["u0"], g["normals"][:n], g["uniforms"][:n], inv_temp=t, step=float(g["beta"]))
        ok = ~np.isnan(out["a"])
        phi_v = np.array([pot(v) for v in out["v"]])
        with np.errstate(invalid="ignore"):
            assert np.array_equal(out["phi_v"][ok], t * phi_v[ok])
        if t == 0.0:   # the prior alone: every finite proposal is accepted
            assert np.array_equal(out["accepted"], np.isfinite(phi_v))
    with np.errstate(invalid="ignore"):
        assert not (np.exp(0.0 * 1.0 - 0.0 * np.nan) > 0.0) and not (np.exp(0.0 * 1.0 - 0.0 * np.inf) > 0.0)


def _round(K, r, phi, t, U, d=2, n_ladders=1, replica=None):
    B_ = n_ladders * K
    u = np.arange(B_ * d, dtype=float).reshape(B_, d)
    replica = np.stack([np.tile(np.arange(K), n_ladders), np.zeros(B_, int)], 1) if replica is None else replica
    sc, rt = np.zeros((n_ladders, K - 1, 2), int), np.zeros(n_ladders, int)
    phi = np.array(phi, dtype=float)
    u0 = u.copy()
    T.swap_round(u, phi, np.array(t, dtype=float), K, r, np.array(U, dtype=float).reshape(n_ladders, K - 1),
                 replica, sc, rt)
    return u0, u, phi, replica, sc, rt


def test_even_odd_pairing():
    assert T.pairs(8, 0) == [0, 2, 4, 6] and T.pairs(8, 1) == [1, 3, 5]
    assert T.pairs(3, 0) == [0] and T.pairs(3, 1) == [1] and T.pairs(2, 0) == [0] and T.pairs(2, 1) == []
    # equal temperatures everywhere: every proposed pair swaps, the others stay
    K = 5
    u0, u, phi, rep, sc, _ = _round(K, 1, np.arange(K) * 3.0, np.ones(K), np.full(K - 1, 0.999999))
    assert np.array_equal(u, u0[[0, 2, 1, 4, 3]]) and np.array_equal(rep[:, 0], [0, 2, 1, 4, 3])
    assert np.array_equal(phi, [0, 6, 3, 12, 9])
    assert np.array_equal(sc[0, :, 0], [0, 1, 0, 1]) and np.array_equal(sc[0, :, 1], [0, 1, 0, 1])


def test_equal_temperature_always_swaps_and_nan_never():
    for phi in ([1e300, -1e300], [0.0, 5.0], [-3.0, 7.5]):
        _, _, _, _, sc, _ = _round(2, 0, phi, [0.7, 0.7], [np.nextafter(1.0, 0.0)])
        assert sc[0, 0, 1] == 1
    for phi in ([np.nan, 1.0], [1.0, np.nan], [np.nan, np.nan]):
        u0, u, ph, _, sc, _ = _round(2, 0, phi, [1.0, 0.0], [0.0])
        assert sc[0, 0].tolist() == [1, 0] and np.array_equal(u, u0)
    # the swap rule: (t_k - t_k1) * (Phi_k - Phi_k1): the colder rung sitting at the higher Phi always swaps
    assert _round(2, 0, [10.0, 1.0], [1.0, 0.5], [0.999])[4][0, 0, 1] == 1
    assert _round(2, 0, [1.0, 10.0], [1.0, 0.5], [np.exp(-4.5) + 1e-12])[4][0, 0, 1] == 0
    assert _round(2, 0, [1.0, 10.0], [1.0, 0.5], [np.exp(-4.5) - 1e-12])[4][0, 0, 1] == 1


def test_round_trips_on_hand_built_rounds():
    """K = 3, every pair swaps: replica 0 goes 0 -> 1 -> 2 (direction -1) -> 1 -> 0 (a round trip)."""
    K = 3
    rep = np.stack([np.arange(K), np.zeros(K, int)], 1)
    u = np.zeros((K, 1))
    phi = np.zeros(K)
    t = np.ones(K)
    sc, rt = np.zeros((1, K - 1, 2), int), np.zeros(1, int)
    pos, trips = [], []
    for r in range(8):
        T.swap_round(u, phi, t, K, r, np.full((1, K - 1), 0.5), rep, sc, rt)
        pos.append(int(np.where(rep[:, 0] == 0)[0][0]))
        trips.append(int(rt[0]))
    assert pos == [1, 2, 2, 1, 0, 0, 1, 2]
    # round 0: slot 0 gets replica 1 (direction 0 -> +1, no trip); round 4: replica 0 comes back down to slot 0
    # after reaching slot 2 in round 1; round 6: replica 1, at the top in round 3, comes back down
    assert trips == [0, 0, 0, 0, 1, 1, 2, 2]
    assert np.array_equal(sc[0], [[4, 4], [4, 4]])


def test_swap_uniform_uses_its_own_philox_slot():
    seed = 0x1234_5678_9ABC_DEF0
    for chain in (0, 7, 2 ** 32 - 1):
        for step in (0, 5, 2 ** 33 + 1):
            us = T.swap_uniform(seed, chain, step)
            assert 0.0 <= us < 1.0
            assert us != P.uniform(seed, chain, step)
            w = P.draw_words(seed, chain, step, T.SLOT_SWAP)
            for slot in (0, 1, 31, 255, P.SLOT_UNIFORM):
                assert w != P.draw_words(seed, chain, step, slot)
                assert us != P.normal(seed, chain, step, slot)
    U = T.swap_uniforms(seed, 8, 2, 4, 1)
    assert np.isnan(U[:, [0, 2]]).all() and U[1, 1] == T.swap_uniform(seed, 8 + 4 + 1, 1)


def test_entry_points_check_arguments_without_gpu():
    from ip_mcmc_b200 import _lib
    lib = _lib.load()
    p = C.c_void_p(8)          # never dereferenced: every call below fails its argument check first
    sw = lib.ipmcmc_swap_replicas

    def err():
        return lib.ipmcmc_last_error()

    assert sw(4, 1, 3, p, p, p, 0, 0, 0, None, p, p, p, None) == -1 and b"ladder_size" in err()
    assert sw(0, 4, 3, p, p, p, 0, 0, 0, None, p, p, p, None) == -1 and b"n_ladders" in err()
    assert sw(4, 4, 0, p, p, p, 0, 0, 0, None, p, p, p, None) == -1 and b"dim" in err()
    assert sw(4, 4, 257, p, p, p, 0, 0, 0, None, p, p, p, None) == -1 and b"dim" in err()
    assert sw(4, 4, 3, p, p, p, 0, 0, -1, None, p, p, p, None) == -1 and b"round" in err()
    assert sw(4, 4, 3, p, p, p, 0, 6, 0, None, p, p, p, None) == -1 and b"split" in err()
    assert sw(2 ** 30, 4, 3, p, p, p, 0, 4, 0, None, p, p, p, None) == -3 and b"2^32" in err()
    for i in (3, 4, 5, 10, 11, 12):
        args = [4, 4, 3, p, p, p, 0, 0, 0, None, p, p, p, None]
        args[i] = None
        assert sw(*args) == -1 and b"NULL" in err()
    desc, bufs = _lib.SamplerDesc(), _lib.ChainBuffers()
    assert lib.ipmcmc_run_tempered(p, C.byref(desc), C.byref(bufs), None, 4, 1, None) == -1 and b"inv_temp" in err()
    assert lib.ipmcmc_run_tempered(None, C.byref(desc), C.byref(bufs), p, 4, 1, None) == -1 and b"NULL" in err()


def test_sampler_rejects_bad_ladders_before_sampling():
    from ip_mcmc_b200 import ParallelTemperingSampler, geometric_inv_temps
    for bad in ([1.0], [1.0, np.nan], [0.9, 0.5], [1.0, 0.5, 0.5], [1.0, 0.2, 0.4], [1.0, -0.1], [1.0, np.inf]):
        with pytest.raises(ValueError):
            ParallelTemperingSampler(None, None, None, bad)
    with pytest.raises(ValueError):
        ParallelTemperingSampler(None, None, None, [1.0, 0.0], swap_interval=0)
    pt = ParallelTemperingSampler(None, None, None, [1.0, 0.5, 0.0])
    with pytest.raises(ValueError, match="ladder"):
        pt.run(np.zeros(3), 10, 0, 1, n_ladders=4, chain_offset=4)       # raises before touching the GPU
    with pytest.raises(ValueError, match="at least 4 samples"):
        pt.run(np.zeros(3), 3, 0, 1, diagnostics=True)
    t = geometric_inv_temps(4, 0.05)
    assert t[0] == 1.0 and t[-1] == 0.05 and np.all(np.diff(t) < 0)
    with pytest.raises(ValueError):
        geometric_inv_temps(1, 0.5)
