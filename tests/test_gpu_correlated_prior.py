"""GPU parity off the reference problem: correlated (dense) Gaussian priors, and Burgers with up to 64 observations.

A dense prior covariance C makes the proposal noise w = A z a dense product on the lanes (sampler.cuh, proposal_noise,
factor_kind 2) and the RW regulariser 1/2 |L w|^2 a full lower-triangular product (prior_regulariser).  More than 32
observations send the window loop of burgers_measure and the residual loop of potential_from_G round a second time.
The oracle (oracle/*_np.py) states both in plain NumPy; the device's own Philox normals are replayed through it."""
import numpy as np
import pytest
import torch

from oracle import burgers_np as B
from oracle import lorenz_np as L
from oracle import mcmc_np as O
from oracle import philox_np as P

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def G():
    import gpu_common
    return gpu_common


def correlated_cov(sd, seed):
    """diag(sd) R diag(sd) with R a seeded correlation matrix of strong off-diagonal entries (rank 2 + 0.3 I)."""
    rng = np.random.default_rng(seed)
    sd = np.asarray(sd, dtype=np.float64)
    F = rng.standard_normal((len(sd), 2))
    S = F @ F.T + 0.3 * np.identity(len(sd))
    C = S / np.sqrt(np.outer(np.diag(S), np.diag(S))) * np.outer(sd, sd)
    return 0.5 * (C + C.T)


def _check_margin(a, U):
    """No decision of the replay is borderline: a pass does not rest on the last bits of a."""
    ok = np.isfinite(a)
    assert ok.any()
    assert np.min(np.abs(a[ok] - U[ok]) / np.maximum(a[ok], 1e-300)) > 1e-6


# ------------------------------------------------------------------------------------------------------------------
# correlated priors
# ------------------------------------------------------------------------------------------------------------------
def _burgers_case(G, name, numerics):
    """(pot, prior, u0, oracle potential factory, n_chains, n_steps) of a Burgers chain with a dense prior."""
    import ip_mcmc_b200 as M
    if name == "kl32":           # d = 32: the parameter vector fills every lane of the warp
        m = 29
        f = M.BurgersFVM(N=64, kl_modes=m, numerics=numerics)
        BP = B.BurgersProblem(64, kl_basis=f.kl_basis)
        truth = np.concatenate([G.TRUTH, np.zeros(m)])
        sd = np.concatenate([np.full(3, 0.25), np.sqrt(M.BurgersFVM.kl_prior_variances(m))])
        n_chains, n_steps = 3, 12
    else:
        N = 2048 if name == "team" else 64
        f = M.BurgersFVM(N=N, numerics=numerics)
        BP = B.BurgersProblem(N)
        truth, sd = G.TRUTH, np.full(3, 0.25)
        n_chains, n_steps = (2, 3) if name == "team" else (3, 12)
    y = BP.G_params(truth)
    pot = M.EvolutionPotential(f, y, M.GaussianDistribution(np.zeros(5), G.NOISE_COV))
    prior = M.GaussianDistribution(f.prior_means, correlated_cov(sd, len(sd)))
    return pot, prior, truth - f.prior_means, lambda: O.Potential(BP, y, G.NOISE_COV), n_chains, n_steps


def _lorenz_case(K, J, numerics):
    from test_gpu_lorenz import _lorenz_setup
    import ip_mcmc_b200 as M
    T = 0.05                   # 2 carried solves per step: rounding differences stay ~1e-8 over the replay
    f, pot, _, p = _lorenz_setup(T, numerics=numerics, K=K, J=J)
    prior = M.GaussianDistribution(np.zeros(3), correlated_cov(np.sqrt([10.0, 1.0, 10.0]), 3))
    opot = lambda: O.Potential(L.LorenzProblem(K, J, T, 1, p["prior_means"], p["IC"]), p["y"], 0.25 * np.diag(p["var"]))
    return pot, prior, np.asarray(p["u0"], dtype=np.float64), opot, 32 // K + 1, 8


def _sampler(kind, pot, prior, step, seed):
    import ip_mcmc_b200 as M
    if kind == "pcn":
        return M.MCMCSampler(M.ConstSteppCNProposer(step, prior), M.CountedAccepter(M.pCNAccepter(pot)),
                             np.random.default_rng(seed))
    return M.MCMCSampler(M.ConstStepStandardRWProposer(step, prior), M.CountedAccepter(M.StandardRWAccepter(pot, prior)),
                         np.random.default_rng(seed))


def device_noise_replay(G, pot, prior, kind, step, u0, make_opot, n_chains, n_steps, seed=3):
    """Free-running chains (Philox noise, dense factor) through MCMCSampler.run and ChainBatch.run, and their replay
    on the oracle: the device's normals z from ipmcmc_rng_probe (same seed, global chain ids 0.., steps 0..), the
    accept uniforms from oracle.philox_np (bit-exact), and w = A z formed as the kernel forms it (j ascending, a
    separate multiply and add: -fmad=false), so that w is the device's bit for bit.  Asserts the proposals, every
    decision, the states and the counters; returns (steplog, oracle chains)."""
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import _lib
    s = _sampler(kind, pot, prior, step, seed)
    states = s.run(u0, n_steps, 0, 1, n_chains=n_chains)
    spec, _, _ = _sampler(kind, pot, prior, step, seed)._compile(n_steps, 0, 1, None)
    assert spec.seed == s.last_run["seed"] and spec.factor_kind == 2
    d = spec.dim
    ch = M.ChainBatch(pot.problem(), u0, n_chains=n_chains)
    trace = torch.empty((n_chains, n_steps, d), dtype=torch.float64, device="cuda")
    slog = torch.empty((n_chains, n_steps, 4), dtype=torch.float64, device="cuda")
    vlog = torch.empty((n_chains, n_steps, d), dtype=torch.float64, device="cuda")
    ch.run(spec, n_steps, trace=trace, steplog=slog, vlog=vlog)
    trace, slog, vlog = trace.cpu().numpy(), slog.cpu().numpy(), vlog.cpu().numpy()
    assert np.array_equal(trace, states)
    assert torch.equal(ch.counters, s.last_run["per_chain_counters"])

    probe = torch.empty((n_chains, n_steps, d + 1), dtype=torch.float64, device="cuda")
    _lib.check(_lib.load().ipmcmc_rng_probe(spec.seed, 0, 0, n_chains, n_steps, d, probe.data_ptr(), None))
    z = probe.cpu().numpy()[..., :d]
    A = spec.factor.reshape(d, d)
    w = np.zeros((n_chains, n_steps, d))
    for j in range(d):
        w = w + A[:, j] * z[..., j:j + 1]
    U = np.array([[P.uniform(spec.seed, c, t) for t in range(n_steps)] for c in range(n_chains)])
    k = O.PCN if kind == "pcn" else O.RW
    cnt = ch.counters.cpu().numpy()
    refs = []
    for c in range(n_chains):
        opot = make_opot()
        ref = O.run_chain(opot, u0, w[c], U[c], k, k, step, prior_cov=prior.covariance,
                          recompute_phi_u=pot.G.stateful)
        assert np.array_equal(vlog[c], ref["v"]), c                 # the probe's normals are the chain kernel's
        assert np.array_equal(slog[c, :, 2].astype(bool), ref["accepted"]), c
        assert np.array_equal(states[c], ref["u"]), c
        assert cnt[c, 0] == n_steps and cnt[c, 1] == ref["accepts"] and cnt[c, 4] == 0, c
        if pot.G.stateful:
            assert cnt[c, 2] + cnt[c, 3] == opot.G.n_accepted + opot.G.n_rejected, c
        refs.append(ref)
    acc = np.array([r["accepted"] for r in refs])
    assert acc.any() and not acc.all()                   # both kinds of decision are exercised
    _check_margin(np.array([r["a"] for r in refs]), U)
    return slog, refs


REPLAYS = [("d3", "exact"), ("d3", "fused"), ("kl32", "exact"), ("kl32", "fused"), ("team", "exact"),
           ("lorenz_K6J4", "exact"), ("lorenz_K6J4", "fused"), ("lorenz_K7J4", "exact"), ("lorenz_K7J4", "fused")]


@pytest.mark.parametrize("kind", ["pcn", "rw"])
@pytest.mark.parametrize("case,numerics", REPLAYS)
def test_correlated_prior_chain_replays_device_noise(G, case, numerics, kind):
    """Chains under a dense prior covariance C on the one-warp (d = 3 and d = 32), team (N = 2048) and Lorenz
    (K = 6 and a run-time K) kernels, free-running on Philox noise, replayed on the oracle with the device's own
    draws.  EXACT Burgers: Phi(v) bit-identical and the accept probability within 1e-12 (NumPy's norm(L @ w)
    sums in another order); FUSED Burgers: 1e-10 / 1e-6 as in test_replay_reference_chain; Lorenz at T = 0.05:
    1e-6 as in test_lorenz_box_constraint_matches_oracle."""
    if case.startswith("lorenz"):
        K, J = int(case[8:case.index("J")]), int(case[case.index("J") + 1:])
        pot, prior, u0, make_opot, n_chains, n_steps = _lorenz_case(K, J, numerics)
        step = 0.3 if kind == "pcn" else 0.05
    else:
        pot, prior, u0, make_opot, n_chains, n_steps = _burgers_case(G, case, numerics)
        step = 0.1 if kind == "pcn" else 0.001
    slog, refs = device_noise_replay(G, pot, prior, kind, step, u0, make_opot, n_chains, n_steps)
    for c, ref in enumerate(refs):
        if case.startswith("lorenz"):
            np.testing.assert_allclose(slog[c, :, 0], ref["phi_v"], rtol=1e-6)
        elif numerics == "exact":
            assert np.array_equal(slog[c, :, 0], ref["phi_v"]), c
            np.testing.assert_allclose(slog[c, :, 1], ref["a"], rtol=1e-12, atol=1e-300)
        else:
            np.testing.assert_allclose(slog[c, :, 0], ref["phi_v"], rtol=1e-10)
            np.testing.assert_allclose(slog[c, :, 1], ref["a"], rtol=1e-6, atol=1e-300)


def test_correlated_prior_stationary_law(G):
    """The law of the dense sampling factor, independent of any host restatement of it: with a flat likelihood
    (noise covariance 1e12, as in test_flat_likelihood_exact_stationary_law) every pCN proposal is accepted and the
    chain is the AR(1) process v = sqrt(1 - beta^2) u + beta A z with stationary law N(0, A A^T) = N(0, C).
    4096 chains, beta = 0.5, 60 steps from 0 (the start is forgotten to 0.75^60 = 3e-8): the end-state mean and
    every covariance entry within 4 standard errors of 0 and of C.  A transposed factor has covariance
    A^T A = diag(singular values) and fails."""
    import ip_mcmc_b200 as M
    d, n_chains, n_steps, beta = 8, 4096, 60, 0.5
    f = M.BurgersFVM(N=32, kl_modes=d - 3, numerics="fused", max_fv_steps=10 ** 7)
    C = correlated_cov(np.full(d, 0.25), 8)
    prior = M.GaussianDistribution(f.prior_means, C)
    pot = M.EvolutionPotential(f, f.at_parameters(np.concatenate([G.TRUTH, np.zeros(d - 3)])),
                               M.GaussianDistribution(np.zeros(5), 1e12 * np.identity(5)))
    s = M.MCMCSampler(M.ConstSteppCNProposer(beta, prior), M.CountedAccepter(M.pCNAccepter(pot)), np.random.default_rng(12))
    end = s.run(np.zeros(d), 1, n_steps, 1, n_chains=n_chains)[:, 0]        # max(0, 60 - 1) + 1 steps
    c = s.last_run["counters"]
    assert c["calls"] == n_chains * n_steps and c["nonfinite"] == 0
    assert c["accepts"] >= 0.999 * c["calls"]
    se_mean = np.sqrt(np.diag(C) / n_chains)
    assert np.all(np.abs(end.mean(0)) < 4 * se_mean), end.mean(0) / se_mean
    emp = end.T @ end / n_chains                      # the mean is known: 0
    se_cov = np.sqrt((np.outer(np.diag(C), np.diag(C)) + C ** 2) / n_chains)
    z = (emp - C) / se_cov
    assert np.all(np.abs(z) < 4), np.round(z, 1)
    assert np.abs(C / np.sqrt(np.outer(np.diag(C), np.diag(C))) - np.identity(d)).max() > 0.7    # strongly correlated


def test_wide_path_refuses_correlated_priors(G):
    """d = 33 runs on the wide kernel, which samples with a diagonal factor and regularises with a diagonal prior
    Cholesky factor only: a dense factor (pCN under a correlated prior) and a non-diagonal prior_chol (RW accepter
    under a correlated prior) each raise the library's refusal instead of running."""
    import ip_mcmc_b200 as M
    from ip_mcmc_b200._lib import EngineError
    m = 30
    f = M.BurgersFVM(N=64, kl_modes=m)
    pot = M.EvolutionPotential(f, f.at_parameters(np.concatenate([G.TRUTH, np.zeros(m)])),
                               M.GaussianDistribution(np.zeros(5), G.NOISE_COV))
    sd = np.concatenate([np.full(3, 0.25), np.sqrt(M.BurgersFVM.kl_prior_variances(m))])
    dense = M.GaussianDistribution(f.prior_means, correlated_cov(sd, 33))
    diag = M.GaussianDistribution(f.prior_means, np.diag(sd ** 2))
    u0 = np.zeros(3 + m)
    s = M.MCMCSampler(M.ConstSteppCNProposer(0.1, dense), M.pCNAccepter(pot), np.random.default_rng(0))
    with pytest.raises(EngineError, match=r"dim=33 > 32: the wide path samples with a diagonal factor only"):
        s.run(u0, 2, 0, 1, n_chains=3)
    s = M.MCMCSampler(M.ConstStepStandardRWProposer(0.001, diag), M.StandardRWAccepter(pot, dense), np.random.default_rng(0))
    with pytest.raises(EngineError, match=r"dim=33 > 32: the wide path needs a diagonal prior_chol"):
        s.run(u0, 2, 0, 1, n_chains=3)
    # the same samplers with the diagonal prior run
    s = M.MCMCSampler(M.ConstStepStandardRWProposer(0.001, diag), M.StandardRWAccepter(pot, diag), np.random.default_rng(0))
    assert s.run(u0, 2, 0, 1, n_chains=3).shape == (3, 2, 3 + m)


def test_host_entry_point_matches_device_path_with_dense_prior(G):
    """MCMCSampler.run_host (ipmcmc_sample_host) == MCMCSampler.run under a correlated prior (dense factor and dense
    prior Cholesky factor, RW): samples, counters, final states and potentials."""
    import ip_mcmc_b200 as M
    f, pot, _, _ = G.burgers_setup(32, "fused")
    prior = M.GaussianDistribution(G.PRIOR_MEAN, correlated_cov(np.full(3, 0.25), 5))
    mk = lambda: _sampler("rw", pot, prior, 0.001, 4)
    s, h = mk(), mk()
    ref = s.run(G.TRUTH - G.PRIOR_MEAN, 25, 0, 1, n_chains=9)
    got = h.run_host(G.TRUTH - G.PRIOR_MEAN, 25, 0, 1, n_chains=9)
    assert h.last_run["seed"] == s.last_run["seed"]
    assert np.array_equal(got, ref)
    assert np.array_equal(h.last_run["per_chain_counters"], s.last_run["per_chain_counters"].cpu().numpy())
    assert 0 < h.accepter.accepts == s.accepter.accepts < 9 * 25
    assert np.array_equal(h.last_run["u"], s.last_run["u"].cpu().numpy())
    assert np.array_equal(h.last_run["phi"], s.last_run["phi"].cpu().numpy())


# ------------------------------------------------------------------------------------------------------------------
# more than 32 observations
# ------------------------------------------------------------------------------------------------------------------
N_OBS = [1, 8, 31, 33, 64]


def _points(N, q, seed):
    """q measurement points; from q = 8 on the last two windows are the edge cases: one reaches past x = 1 (its
    right limit is clipped to N), the other holds a single cell centre (no trapezoid: G = 0)."""
    if q == 1:
        return np.array([0.25])
    dx = 2.0 / N
    rng = np.random.default_rng(seed)
    return np.concatenate([np.sort(rng.uniform(-0.9, 0.9, q - 2)), [0.99, 1.0 - 0.75 * dx + 0.05]])


def _noise(q, dense, seed):
    sd = 0.05 * (1.0 + np.random.default_rng(seed).random(q))
    return correlated_cov(sd, seed) if dense else np.diag(sd ** 2)


@pytest.mark.parametrize("numerics", ["exact", "fused"])
@pytest.mark.parametrize("path", ["one_warp", "wide", "team"])
def test_many_observations_forward_vs_oracle(G, path, numerics):
    """G, FV steps and Phi for q = 1 ... 64 measurement windows (lane i measures windows i, i + 32: two rounds of
    the window loop from q = 33; Phi sums q residuals^2 with NumPy's 8-accumulator pairwise order from q = 8) on the
    one-warp (N = 256), wide (d = 33) and team (N = 2048) solvers, against oracle.burgers_np and mcmc_np.Potential.
    Noise diagonal, and dense at q = 33 and 64.  EXACT: G and the FV steps bit-identical, Phi bit-identical with
    diagonal noise and within 1e-12 with dense noise (the oracle's dev @ LP is a BLAS product of unspecified
    summation order, as in test_dense_noise_covariance); FUSED: 1e-10."""
    import ip_mcmc_b200 as M
    N, m = {"one_warp": (256, 0), "wide": (128, 30), "team": (2048, 0)}[path]
    rng = np.random.default_rng(N + m)
    base = M.BurgersFVM(N=N, kl_modes=m)
    BP = B.BurgersProblem(N, kl_basis=base.kl_basis if m else None)
    truth = np.concatenate([G.TRUTH, np.zeros(m)])
    u = np.vstack([truth - base.prior_means, np.concatenate([0.25 * rng.standard_normal((3, 3)),
                                                             0.05 * rng.standard_normal((3, m))], axis=1)])
    ends, n_fv = [], []
    for x in np.vstack([truth, base.prior_means + u]):
        ends.append(BP.end_state(x))
        n_fv.append(BP.last_n_fv)
    for q in N_OBS:
        pts = _points(N, q, q)
        left, right, dx_meas = B.measurer_windows(pts, 0.1, BP.x[1:-1])
        if q >= 8:
            assert right[-2] == N and right[-2] - left[-2] > 2 and right[-1] - left[-1] == 1
        G_ref = np.array([B.measure(e, left, right, dx_meas) for e in ends])
        y = G_ref[0] + 0.05 * rng.standard_normal(q)
        for dense in ([False, True] if q > 32 else [False]):
            cov = _noise(q, dense, q)
            f = M.BurgersFVM(N=N, kl_modes=m, points=pts, numerics=numerics)
            assert np.array_equal(f.left_limits, left) and np.array_equal(f.right_limits, right)
            r = M.EvolutionPotential(f, y, M.GaussianDistribution(np.zeros(q), cov)).problem().forward(u)
            Gd, phi, work = r["G"].cpu().numpy(), r["phi"].cpu().numpy(), r["work"].cpu().numpy()
            opot = O.Potential(None, y, cov)
            phi_ref = np.array([-O.gaussian_logpdf(y - g, opot.LP, opot.log_pdet, opot.rank) for g in G_ref[1:]])
            msg = str((path, q, dense))
            if q >= 8:
                assert np.all(Gd[:, -1] == 0), msg
            if numerics == "exact":
                assert np.array_equal(Gd, G_ref[1:]), msg
                assert np.array_equal(work[:, 0], n_fv[1:]), msg
                if dense:
                    np.testing.assert_allclose(phi, phi_ref, rtol=1e-12, err_msg=msg)
                else:
                    assert np.array_equal(phi, phi_ref), msg
            else:
                np.testing.assert_allclose(Gd, G_ref[1:], rtol=1e-10, atol=1e-13, err_msg=msg)
                np.testing.assert_allclose(phi, phi_ref, rtol=1e-10, err_msg=msg)


@pytest.mark.parametrize("numerics", ["exact", "fused"])
def test_many_observations_chain_replay(G, numerics):
    """pCN chain with q = 64 observations and dense noise, injected noise, against the oracle: every decision and
    every state equal, Phi(v) within 1e-12 (EXACT) / 1e-10 (FUSED), no borderline decision."""
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import _lib
    N, q, beta, n_steps = 64, 64, 0.05, 16
    pts = _points(N, q, q)
    BP = B.BurgersProblem(N, points=pts)
    rng = np.random.default_rng(64)
    y = BP.G_params(G.TRUTH) + 0.05 * rng.standard_normal(q)
    cov = _noise(q, True, q)
    f = M.BurgersFVM(N=N, points=pts, numerics=numerics)
    pot = M.EvolutionPotential(f, y, M.GaussianDistribution(np.zeros(q), cov))
    u0 = G.TRUTH - G.PRIOR_MEAN
    z = 0.25 * rng.standard_normal((n_steps, 3))
    U = rng.random(n_steps)
    ref = O.run_chain(O.Potential(BP, y, cov), u0, z, U, O.PCN, O.PCN, beta)
    spec = M.SamplerSpec(3, _lib.PROPOSE_PCN, _lib.ACCEPT_PCN, coef_u=np.sqrt(1 - beta ** 2), coef_w=beta)
    states, slog, vlog, ch = G.run_injected(pot, spec, u0, z, U, n_copies=2)
    assert ref["accepted"].any() and not ref["accepted"].all()
    _check_margin(ref["a"], U)
    for c in range(2):
        assert np.array_equal(vlog[c], ref["v"]) and np.array_equal(states[c], ref["u"])
        assert np.array_equal(slog[c, :, 2].astype(bool), ref["accepted"])
        np.testing.assert_allclose(slog[c, :, 0], ref["phi_v"], rtol=1e-12 if numerics == "exact" else 1e-10)
    assert ch.counters[:, 1].tolist() == [ref["accepts"]] * 2


def test_more_than_64_observations_are_refused(G):
    """ipmcmc_burgers_create refuses q = 65 (IPMCMC_EINVAL), raised as the ValueError of every argument check."""
    import ip_mcmc_b200 as M
    q = 65
    f = M.BurgersFVM(N=64, points=np.linspace(-0.9, 0.9, q))
    pot = M.EvolutionPotential(f, np.zeros(q), M.GaussianDistribution(np.zeros(q), np.identity(q)))
    with pytest.raises(ValueError, match=r"n_obs=65 outside \[1,64\]"):
        pot.problem()
