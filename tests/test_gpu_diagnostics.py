"""Device convergence diagnostics (diagnostics.chain_diagnostics, ipmcmc_diag_*) against the host reference in
stats.py: per-chain tau, split-R-hat, multi-chain ESS and its cut-off T, for every chain of a batch."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import ip_mcmc_b200 as M
from ip_mcmc_b200 import _lib, diagnostics, stats
from gpu_common import burgers_setup

pytestmark = pytest.mark.gpu


def ar1(Mc, n, d, phi, seed):
    """AR(1) chains started from their stationary law N(0, 1 / (1 - phi^2))."""
    rng = np.random.default_rng(seed)
    x = np.empty((Mc, n, d))
    x[:, 0] = rng.standard_normal((Mc, d)) / math.sqrt(1 - phi * phi)
    for i in range(1, n):
        x[:, i] = phi * x[:, i - 1] + rng.standard_normal((Mc, d))
    return x


def deciding_margin(x):
    """Smallest |rho_{t+1} + rho_{t+2}| over the pairs the host's truncation loop tests, over all parameters:
    a fixture whose margin is not clear of zero could flip T under rounding and is not a fair comparison."""
    psi = stats.split_sequences(x)
    m, h, d = psi.shape
    _, vp = stats._split_var_plus(psi)
    _, T = stats.multichain_ess(x)
    margin = np.inf
    for j in range(d):
        def rho(t):
            return 1.0 - ((psi[:, t:, j] - psi[:, :h - t, j]) ** 2).sum() / (m * (h - t)) / (2.0 * vp[j])
        for t in range(1, T[j] + 1, 2):
            if t + 2 <= h - 1:
                margin = min(margin, abs(rho(t + 1) + rho(t + 2)))
    return margin


def check_against_host(x, res, split=True):
    tau = np.array([[stats.integrated_autocorr_time(x[c, :, j]) for j in range(x.shape[2])] for c in range(x.shape[0])])
    np.testing.assert_allclose(res["tau"], tau, rtol=1e-10)
    np.testing.assert_allclose(res["ess_per_chain_sum"], stats.ess_multichain(x)[0], rtol=1e-10)
    if split:
        np.testing.assert_allclose(res["rhat"], stats.split_rhat(x), rtol=1e-10)
        ne, T = stats.multichain_ess(x)
        assert np.array_equal(res["cutoff"], T)
        np.testing.assert_allclose(res["ess"], ne, rtol=1e-10)


def stuck_chains(x, first, count, seed):
    """Chains first .. first+count-1 stuck at random doubles (a chain that accepts nothing).  Returns how many
    of these series NumPy's mean reproduces exactly (y = 0: all-ones autocorrelation) and how many it does not
    (y = a constant rounding residue)."""
    vals = np.random.default_rng(seed).standard_normal((count, x.shape[2])) * 10.0 ** np.arange(-2, x.shape[2] - 2)[None, :]
    x[first:first + count] = vals[:, None, :]
    exact = sum(np.mean(x[c, :, j]) == x[c, 0, j] for c in range(first, first + count) for j in range(x.shape[2]))
    return exact, count * x.shape[2] - exact


@pytest.mark.parametrize("d", [1, 3, 33])
@pytest.mark.parametrize("n", [7, 1000, 2500, 5000])
@pytest.mark.parametrize("phi", [0.0, 0.5, 0.95])
def test_tau_matches_host_for_every_series(phi, n, d):
    Mc = 12 if d == 33 else 24
    x = ar1(Mc, n, d, phi, seed=int(100 * phi) + n + d)
    x[1] = 0.75                                # a constant chain: all-ones autocorrelation
    x[2, :, 0] = -3.0
    exact, residue = stuck_chains(x, 3, 8, seed=n + d)
    assert exact > 0 and residue > 0
    res = M.chain_diagnostics(torch.from_numpy(x).cuda())
    assert res["tau"][1].tolist() == [1 + 4 * ((n - 1) // 2)] * d
    check_against_host(x, res, split=False)


SPLIT_CASES = {
    "ar1_d3": dict(Mc=64, n=1000, d=3, phi=0.5),
    "odd_n": dict(Mc=40, n=999, d=2, phi=0.7),
    "single_chain": dict(Mc=1, n=400, d=2, phi=0.3),
    "many_chains": dict(Mc=300, n=200, d=2, phi=0.6),
    "cutoff_beyond_first_block": dict(Mc=32, n=2000, d=2, phi=0.98),
    "wide": dict(Mc=8, n=300, d=33, phi=0.5),
    "unstaged_long": dict(Mc=4, n=26000, d=1, phi=0.9),
}


@pytest.mark.parametrize("case", sorted(SPLIT_CASES))
def test_split_rhat_and_ess_match_host(case):
    c = SPLIT_CASES[case]
    x = ar1(c["Mc"], c["n"], c["d"], c["phi"], seed=len(case))
    assert deciding_margin(x) > 1e-8
    res = M.chain_diagnostics(x)                         # NumPy input: uploaded once
    check_against_host(x, res)
    if case == "cutoff_beyond_first_block":
        assert np.all(res["cutoff"] > diagnostics.LAG_BLOCK0)


def test_two_modes():
    x = ar1(64, 600, 3, 0.8, seed=5)
    x[32:] += 3.0 * np.sqrt(1 / (1 - 0.64))
    assert deciding_margin(x) > 1e-8
    res = M.chain_diagnostics(x)
    check_against_host(x, res)
    assert np.all(res["rhat"] > 1.5)


def test_constant_chains_special_values():
    same = np.full((8, 20, 2), 0.75)
    res = M.chain_diagnostics(same)
    ne, T = stats.multichain_ess(same)
    assert np.all(np.isnan(res["rhat"])) and np.all(np.isnan(res["ess"])) and np.all(np.isnan(ne))
    assert np.array_equal(res["cutoff"], T)
    apart = same * np.arange(1, 9)[:, None, None]
    res = M.chain_diagnostics(apart)
    ne, T = stats.multichain_ess(apart)
    assert np.all(np.isinf(res["rhat"])) and np.all(np.isinf(stats.split_rhat(apart)))
    assert np.array_equal(res["cutoff"], T) and np.array_equal(res["ess"], ne)


def test_sliced_trace_is_read_in_place():
    full = torch.from_numpy(ar1(50, 537, 3, 0.6, seed=6)).cuda()
    a = M.chain_diagnostics(full[:, 37:])
    b = M.chain_diagnostics(full[:, 37:].contiguous())
    for k in ("rhat", "ess", "cutoff", "tau"):
        assert np.array_equal(a[k], b[k]), k
    assert a["ess_per_chain_sum"] == b["ess_per_chain_sum"]


def test_two_shards_merged_equal_one_call():
    x = torch.from_numpy(ar1(101, 800, 3, 0.7, seed=7)).cuda()
    one = M.chain_diagnostics(x)
    two = diagnostics._diagnose([x[:50], x[50:]], torch.stack)
    np.testing.assert_allclose(two["rhat"], one["rhat"], rtol=1e-12)
    np.testing.assert_allclose(two["ess"], one["ess"], rtol=1e-12)
    assert np.array_equal(two["cutoff"], one["cutoff"])
    np.testing.assert_allclose(two["ess_per_chain_sum"], one["ess_per_chain_sum"], rtol=1e-12)
    assert np.array_equal(two["tau"], one["tau"])


def test_caller_scratch_or_not_gives_the_same_bits():
    lib = _lib.load()
    x = torch.from_numpy(ar1(200, 300, 2, 0.5, seed=8)).cuda()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    n, d, L = 300, 2, 100
    nbytes = lib.ipmcmc_diag_scratch_bytes(200, d, L)
    scratch = torch.empty((nbytes,), dtype=torch.uint8, device="cuda")
    outs = []
    for s in (C.c_void_p(scratch.data_ptr()), None):
        ss = torch.empty((d, 4), dtype=torch.float64, device="cuda")
        v = torch.empty((d, L), dtype=torch.float64, device="cuda")
        _lib.check(lib.ipmcmc_diag_seqstats(200, n, d, C.c_void_p(x.data_ptr()), n * d, C.c_void_p(ss.data_ptr()), s, nbytes, st))
        _lib.check(lib.ipmcmc_diag_variogram(200, n, d, C.c_void_p(x.data_ptr()), n * d, 1, L, None, C.c_void_p(v.data_ptr()), L,
                                             s, nbytes, st))
        outs.append((ss.cpu(), v.cpu()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


def test_burgers_end_to_end():
    f, pot, prior, _ = burgers_setup(64, numerics="fused")

    def sampler():
        return M.MCMCSampler(M.ConstSteppCNProposer(0.25, prior), M.pCNAccepter(pot), np.random.default_rng(11))

    s = sampler()
    tr = s.run(np.zeros(3), 1000, 0, 1, n_chains=256, return_device=True)
    res = M.chain_diagnostics(tr)
    host = tr[:32].cpu().numpy()
    tau = np.array([[stats.integrated_autocorr_time(host[c, :, j]) for j in range(3)] for c in range(32)])
    np.testing.assert_allclose(res["tau"][:32], tau, rtol=1e-10)
    assert res["tau"].shape == (256, 3) and np.all(np.isfinite(res["rhat"])) and np.all(res["ess"] > 0)
    plain = sampler().run(np.zeros(3), 1000, 0, 1, n_chains=256)
    s2 = sampler()
    with_diag = s2.run(np.zeros(3), 1000, 0, 1, n_chains=256, diagnostics=True)
    assert np.array_equal(plain, with_diag)
    dd = s2.last_run["diagnostics"]
    for k in ("rhat", "ess", "cutoff", "tau"):
        assert np.array_equal(dd[k], res[k]), k
