"""Replica exchange on the device: the tempered Metropolis step against ipmcmc_run and against the CPU
statement (oracle/tempering_np.py), the swap kernel against the oracle's rounds, ParallelTemperingSampler's
reproducibility across launches and shards, and the stationary laws of a (1, 0) ladder."""
import numpy as np
import pytest
import torch

from conftest import golden
from oracle import burgers_np as B
from oracle import mcmc_np as O
from oracle import tempering_np as T

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def G():
    import gpu_common
    return gpu_common


def _pcn_spec(d, beta=0.25, factor=None, **kw):
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import _lib
    return M.SamplerSpec(d, _lib.PROPOSE_PCN, _lib.ACCEPT_PCN, coef_u=np.sqrt(1 - beta ** 2), coef_w=beta,
                         factor=np.full(d, 0.25) if factor is None else factor, **kw)


def _rw_spec(d, delta=0.001, box=False, **kw):
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import _lib
    c = None
    if box:
        lo = np.full(d, -np.inf)
        hi = np.full(d, np.inf)
        lo[2], hi[2] = -0.58, -0.42
        sh = np.zeros(d)
        sh[2] = -0.5
        c = M.BoxConstraint(lo, hi, shift=sh)
    return M.SamplerSpec(d, _lib.PROPOSE_RW, _lib.ACCEPT_RW, coef_u=1.0, coef_w=np.sqrt(2 * delta),
                         factor=np.full(d, 0.25), prior_chol=0.25 * np.identity(d), constraint=c, **kw)


def _problem(G, N, numerics, d):
    import ip_mcmc_b200 as M
    if d == 3:
        return G.burgers_setup(N, numerics)[1]
    m = d - 3
    f = M.BurgersFVM(N=N, kl_modes=m, numerics=numerics)
    truth = np.concatenate([G.TRUTH, 0.01 * np.ones(m)])
    return M.EvolutionPotential(f, f.at_parameters(truth), M.GaussianDistribution(np.zeros(5), G.NOISE_COV))


def _run_batch(pot, spec, n_chains, n_steps, inv_temp, u0, scheduler=None):
    import ip_mcmc_b200 as M
    ch = M.ChainBatch(pot.problem(), u0, n_chains=n_chains, scheduler=scheduler)
    if inv_temp is not None:
        ch.inv_temp = torch.as_tensor(inv_temp, dtype=torch.float64).cuda().contiguous()
    trace = torch.empty((n_chains, n_steps, ch.d), dtype=torch.float64, device="cuda")
    ch.run(spec, n_steps, trace=trace)
    return trace, ch


@pytest.mark.parametrize("N,numerics,d,kind,scheduler", [
    (256, "fused", 3, "pcn", "dynamic"),     # the bench shape
    (64, "exact", 3, "pcn", "dynamic"),
    (64, "exact", 3, "rw", "static"),
    (64, "fused", 3, "boxrw", "dynamic"),
    (2048, "fused", 3, "pcn", None),          # team solver
    (64, "fused", 33, "pcn", None),           # wide path
    (64, "exact", 33, "boxrw", None),
])
def test_unit_inverse_temperature_is_ipmcmc_run(G, N, numerics, d, kind, scheduler):
    """ipmcmc_run_tempered with t = 1 everywhere: the same bits as ipmcmc_run in samples, u, Phi, counters, moments."""
    pot = _problem(G, N, numerics, d)
    spec = {"pcn": _pcn_spec, "rw": _rw_spec, "boxrw": lambda d: _rw_spec(d, box=True)}[kind](d)
    spec.seed = 1234
    n, steps = (16 if N > 1024 else 96), (6 if N > 1024 else 30)
    u0 = np.zeros(d)
    t0, c0 = _run_batch(pot, spec, n, steps, None, u0, scheduler)
    t1, c1 = _run_batch(pot, spec, n, steps, np.ones(n), u0, scheduler)
    assert torch.equal(t0, t1)
    for name in ("u", "mom_count", "mom_mean", "mom_m2", "counters"):
        assert torch.equal(getattr(c0, name), getattr(c1, name)), name
    assert torch.equal(torch.nan_to_num(c0.phi, nan=7.0), torch.nan_to_num(c1.phi, nan=7.0))
    assert c1.counters[:, 1].sum().item() > 0


@pytest.mark.parametrize("numerics", ["exact", "fused"])
@pytest.mark.parametrize("name,kind", [("chain_burgers_pcn_N64.npz", "pcn"), ("chain_burgers_rw_N64.npz", "rw"),
                                       ("chain_burgers_pcn_N256.npz", "pcn")])
def test_tempered_replay_against_oracle(G, numerics, name, kind):
    """Injected noise at t in {0.5, 0.1, 0}: EXACT reproduces the CPU statement's states and decisions bit for bit,
    FUSED every decision (none of them borderline at the FUSED tolerance)."""
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import _lib
    g = golden(name)
    Nn = int(g["N"])
    f, pot, prior, _ = G.burgers_setup(Nn, numerics)
    if kind == "pcn":
        beta = float(g["beta"])
        spec = M.SamplerSpec(3, _lib.PROPOSE_PCN, _lib.ACCEPT_PCN, coef_u=np.sqrt(1 - beta ** 2), coef_w=beta)
        okw = dict(proposer=O.PCN, accepter=O.PCN, step=beta)
    else:
        delta = float(g["delta"])
        spec = M.SamplerSpec(3, _lib.PROPOSE_RW, _lib.ACCEPT_RW, coef_u=1.0, coef_w=np.sqrt(2 * delta),
                             prior_chol=prior.L)
        okw = dict(proposer=O.RW, accepter=O.RW, step=delta, prior_cov=G.PRIOR_COV)
    P = B.BurgersProblem(Nn)
    opot = O.Potential(P, P.G_params(G.TRUTH), G.NOISE_COV)
    temps = [0.5, 0.1, 0.0]
    nst = len(g["normals"])
    ch = M.ChainBatch(pot.problem(), g["u0"], n_chains=len(temps))
    ch.inv_temp = torch.tensor(temps, dtype=torch.float64, device="cuda")
    w = G.cuda(np.stack([g["normals"]] * len(temps)))
    U = G.cuda(np.stack([g["uniforms"]] * len(temps)))
    trace = torch.empty((len(temps), nst, 3), dtype=torch.float64, device="cuda")
    slog = torch.empty((len(temps), nst, 4), dtype=torch.float64, device="cuda")
    ch.run(spec, nst, trace=trace, steplog=slog, inject_w=w, inject_u=U)
    states, slog = trace.cpu().numpy(), slog.cpu().numpy()
    cnt = ch.counters.cpu().numpy()
    for c, t in enumerate(temps):
        ref = T.run_chain(opot, g["u0"], g["normals"], g["uniforms"], inv_temp=t, uniforms_by_step=True, **okw)
        assert np.array_equal(slog[c, :, 2].astype(bool), ref["accepted"]), t
        assert cnt[c, 1] == ref["accepts"]
        if numerics == "exact":
            assert np.array_equal(states[c], ref["u"])
            with np.errstate(invalid="ignore"):
                assert np.array_equal(t * slog[c, :, 0], ref["phi_v"], equal_nan=True)
        else:
            np.testing.assert_allclose(states[c], ref["u"], rtol=1e-9, atol=1e-12)
            a_ref, ok = ref["a"], np.isfinite(ref["a"])
            margin = np.abs(a_ref[ok] - g["uniforms"][ok]) / np.maximum(a_ref[ok], 1e-300)
            assert margin.size == 0 or np.min(margin) > 1e-6
        if t == 0.0 and kind == "pcn":
            assert cnt[c, 1] == cnt[c, 0] - cnt[c, 4]


def _swap_case(K, d, L, rng):
    B_ = L * K
    u = rng.standard_normal((B_, d))
    phi = rng.standard_normal(B_) * 3.0
    phi[rng.random(B_) < 0.1] = np.nan
    t = np.tile(np.sort(rng.random(K))[::-1], L)
    t[::K] = 1.0
    if K >= 3:
        t[1::K] = t[2::K]        # an equal-temperature pair in every ladder
    return u, phi, t


@pytest.mark.parametrize("K", [2, 3, 8])
@pytest.mark.parametrize("d", [3, 33])
@pytest.mark.parametrize("inject", [False, True])
def test_swap_rounds_against_oracle(K, d, inject):
    from ip_mcmc_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(K * 100 + d + inject)
    L, seed, off = 37, 0xDEADBEEF12345, 8 * K
    u, phi, t = _swap_case(K, d, L, rng)
    rep = np.stack([np.tile(np.arange(K), L), np.zeros(L * K, int)], 1).astype(np.int32)
    sc, rt = np.zeros((L, K - 1, 2), np.int64), np.zeros(L, np.int64)
    dev = [torch.as_tensor(x).cuda().contiguous() for x in (u, phi, t, rep, sc, rt)]
    ptr = lambda x: x.data_ptr()
    for r in range(7):
        U = rng.random((L, K - 1)) if inject else T.swap_uniforms(seed, off, L, K, r)
        Ud = torch.as_tensor(U).cuda() if inject else None
        _lib.check(lib.ipmcmc_swap_replicas(L, K, d, ptr(dev[0]), ptr(dev[1]), ptr(dev[2]), seed, off, r,
                                            ptr(Ud) if inject else None, ptr(dev[3]), ptr(dev[4]), ptr(dev[5]), None))
        T.swap_round(u, phi, t, K, r, U, rep, sc, rt)
        if r == 2:   # change Phi between rounds as Metropolis steps would
            phi[:] = rng.standard_normal(L * K)
            phi[rng.random(L * K) < 0.1] = np.nan
            dev[1].copy_(torch.as_tensor(phi))
    torch.cuda.synchronize()
    assert np.array_equal(dev[0].cpu().numpy(), u)
    assert np.array_equal(dev[1].cpu().numpy(), phi, equal_nan=True)
    assert np.array_equal(dev[3].cpu().numpy(), rep)
    assert np.array_equal(dev[4].cpu().numpy(), sc)
    assert np.array_equal(dev[5].cpu().numpy(), rt)
    assert sc[..., 1].sum() > 0 and sc[..., 1].sum() < sc[..., 0].sum()


def _pt(G, N=64, temps=(1.0, 0.3, 0.05), swap_interval=5, seed=11):
    import ip_mcmc_b200 as M
    f, pot, prior, _ = G.burgers_setup(N, "fused")
    return M.ParallelTemperingSampler(M.ConstSteppCNProposer(0.25, prior), M.pCNAccepter(pot),
                                      np.random.default_rng(seed), list(temps), swap_interval=swap_interval)


def test_sampler_is_reproducible_across_launches_and_shards(G):
    L, K = 24, 3
    args = (np.zeros(3), 12, 30, 5)
    whole = _pt(G)
    s0 = whole.run(*args, n_ladders=L, all_rungs=True)
    r0 = whole.last_run
    a = _pt(G)
    s1 = a.run(*args, n_ladders=L, all_rungs=True, steps_per_launch=3)
    assert np.array_equal(s0, s1)
    assert torch.equal(r0["u"], a.last_run["u"]) and np.array_equal(r0["replica"], a.last_run["replica"])
    assert torch.equal(r0["swap_counts"], a.last_run["swap_counts"]) and r0["round_trips"] == a.last_run["round_trips"]
    assert a.last_run["launches"] > r0["launches"]
    parts = []
    for off in (0, 10 * K):
        sh = _pt(G)
        n = 10 if off == 0 else L - 10
        parts.append((sh.run(*args, n_ladders=n, chain_offset=off, all_rungs=True), sh.last_run))
    assert np.array_equal(np.concatenate([p[0] for p in parts]), s0)
    assert np.array_equal(np.concatenate([p[1]["replica"] for p in parts]), r0["replica"])
    assert sum(p[1]["round_trips"] for p in parts) == r0["round_trips"]
    # the t = 1 rung alone, its pooled moments and its diagnostics
    again = _pt(G)
    cold = again.run(*args, n_ladders=L, diagnostics=True)
    assert np.array_equal(cold, s0[:, 0])
    lr = again.last_run
    np.testing.assert_allclose(lr["pooled_mean"], s0[:, 0].reshape(-1, 3).mean(0), rtol=1e-10, atol=1e-14)
    assert lr["counters"]["calls"] == L * 85 and lr["rung_counters"].shape == (K, 6)
    assert lr["diagnostics"]["rhat"].shape == (3,)
    assert 0 < lr["swap_acceptance"].min() and lr["swap_acceptance"].max() <= 1


def _zscore(a, b):
    return (a.mean(0) - b.mean(0)) / np.sqrt(a.var(0, ddof=1) / len(a) + b.var(0, ddof=1) / len(b))


def test_two_rung_ladder_stationary_laws(G):
    """(1, 0) ladder, pCN, N = 64, 4096 ladders: the t = 0 rung samples the prior, the t = 1 rung the posterior
    that untempered chains sample."""
    import ip_mcmc_b200 as M
    L = 4096
    pt = _pt(G, temps=(1.0, 0.0), swap_interval=10, seed=5)
    u0 = np.tile(G.TRUTH, (L, 1))
    s = pt.run(u0, 40, 300, 10, all_rungs=True)
    hot = pt.last_run["u"].view(L, 2, 3)[:, 1].cpu().numpy()
    se_mean, se_var = 0.25 / np.sqrt(L), 0.25 ** 2 * np.sqrt(2.0 / (L - 1))
    assert np.all(np.abs(hot.mean(0)) < 4 * se_mean), hot.mean(0)
    assert np.all(np.abs(hot.var(0, ddof=1) - 0.25 ** 2) < 4 * se_var), hot.var(0, ddof=1)
    assert pt.last_run["round_trips"] > 0
    f, pot, prior, _ = G.burgers_setup(64, "fused")
    ref = M.MCMCSampler(M.ConstSteppCNProposer(0.25, prior), M.pCNAccepter(pot), np.random.default_rng(6))
    r = ref.run(u0, 40, 300, 10, n_chains=L)
    cold = s[:, 0]
    z_mean = _zscore(cold.mean(1), r.mean(1))
    z_var = _zscore(cold.var(1, ddof=1), r.var(1, ddof=1))
    assert np.all(np.abs(z_mean) < 4) and np.all(np.abs(z_var) < 4), (z_mean, z_var)


def test_lorenz_chains_cannot_be_tempered(G):
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import _lib
    K, J = 6, 4
    f = M.Lorenz96Moments(K, J, 0.25, 1.0, np.array([12., 8, 9]), np.random.default_rng(1).random(K * (J + 1)))
    pot = M.EvolutionPotential(f, np.zeros(5 * K), M.GaussianDistribution(np.zeros(5 * K), np.identity(5 * K)))
    ch = M.ChainBatch(pot.problem(), np.zeros(3), n_chains=2)
    ch.inv_temp = torch.ones(2, dtype=torch.float64, device="cuda")
    spec = M.SamplerSpec(3, _lib.PROPOSE_PCN, _lib.ACCEPT_PCN, coef_u=0.9, coef_w=0.1, recompute_phi_u=True)
    with pytest.raises(_lib.EngineError, match="cannot be tempered"):
        ch.run(spec, 1)
